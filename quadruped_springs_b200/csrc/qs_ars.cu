// qs_ars.cu -- qs_obs_stats and qs_ars_act (include/qs_b200.h): the per-step kernels of batched ARS training
// (quadruped_springs_b200/ars.py).  Its own translation unit: the step's kernels and their compile are not touched.
//
// qs_ars_act: one thread per env, one block per tile of envs of ONE candidate.  The block forms that candidate's weights
// theta +- delta_std * delta once into shared memory, zero-padded to fixed shapes (inputs to QS_MAX_OBS, hidden layers
// to QS_ARS_MAX_HIDDEN, outputs to QS_ARS_MAX_ACT), so every thread runs the same fully unrolled network with its
// activations in registers; the padded terms add exact zeros.  Every env's arithmetic is a fixed sequence of operations on
// its own row, so its action does not depend on the batch.
//
// qs_obs_stats: one cluster of kStatsBlocks blocks.  Warp w of the cluster owns rows w, w + 256, ...; lane c owns column
// c.  Each lane sums its alive rows shifted by its first one (no cancellation against a far-away origin), the 32 warps of
// a block are merged in order (Chan et al.), and block 0 merges the block partials in order through distributed shared
// memory and then into the running statistics.  A warp updates the bookkeeping of exactly the rows it read, after
// reading them, so no block ever sees another block's update of `alive`.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/qs_b200.h"

namespace qs {
int abi_fail(int code, const std::string& msg);  // qs_kernels.cu: error text of qs_last_error
void abi_count_launch();                          // qs_kernels.cu: qs_launch_count
}  // namespace qs

namespace cg = cooperative_groups;

namespace {

// ------------------------------------------------------------------------------------------------ qs_ars_act
constexpr int kIn = QS_MAX_OBS;          // padded input width
constexpr int kH = QS_ARS_MAX_HIDDEN;    // padded hidden width
constexpr int kA = QS_ARS_MAX_ACT;       // padded output width
constexpr int kActThreads = 128;

// padded shared layout of a network with kLayers hidden layers: from offset 0, for every hidden layer W [kH][in] then b [kH]; the
// output layer transposed, WT [in][kA], then b [kA] (a thread reads one input's kA weights as three float4)
template <int kLayers>
struct Layout {
  static constexpr int kHid1 = kH * kIn + kH;                            // second hidden layer (kLayers == 2)
  static constexpr int kOut = kLayers == 0 ? 0 : (kLayers == 1 ? kHid1 : kHid1 + kH * kH + kH);
  static constexpr int kOutIn = kLayers == 0 ? kIn : kH;
  static constexpr int kSize = kOut + kOutIn * kA + kA;
};
static_assert(Layout<2>::kSize % 4 == 0 && Layout<2>::kHid1 % 4 == 0 && Layout<2>::kOut % 4 == 0, "float4 layout");

struct Candidate {
  const float* theta;
  const float* delta;   // NULL: theta itself
  float std;
  bool minus;
  __device__ __forceinline__ float operator()(int k) const {
    // torch: theta + (delta * delta_std) and theta - (delta * delta_std), each op rounded on its own
    if (!delta) return theta[k];
    const float d = __fmul_rn(delta[k], std);
    return minus ? __fsub_rn(theta[k], d) : __fadd_rn(theta[k], d);
  }
};

__host__ __device__ inline int arch_params(const qs_ars_arch& a) {
  int P = 0, in = a.obs_dim;
  for (int l = 0; l < a.n_hidden; l++) {
    P += a.hidden[l] * in + (a.bias ? a.hidden[l] : 0);
    in = a.hidden[l];
  }
  return P + a.act_dim * in + (a.bias ? a.act_dim : 0);
}

// one Linear layer of `in` x `out` real weights at theta offset `off` into a padded shared block; returns the next offset
__device__ int load_layer(float* W, float* b, int in_pad, int out_pad, bool transposed, int in, int out, bool bias,
                          const Candidate& cand, int off) {
  for (int q = threadIdx.x; q < in_pad * out_pad; q += blockDim.x) {
    const int row = transposed ? q % out_pad : q / in_pad;   // output index
    const int col = transposed ? q / out_pad : q % in_pad;   // input index
    W[q] = (row < out && col < in) ? cand(off + row * in + col) : 0.f;
  }
  for (int q = threadIdx.x; q < out_pad; q += blockDim.x) b[q] = (bias && q < out) ? cand(off + out * in + q) : 0.f;
  return off + out * in + (bias ? out : 0);
}

__device__ __forceinline__ float activate(float v, int act) { return act == QS_ARS_TANH ? tanhf(v) : fmaxf(v, 0.f); }

// acc[kA] += WT[kA] * h for one input, the weights read as three float4
__device__ __forceinline__ void out_fma(const float* WT, float h, float* out) {
  const float4* w4 = reinterpret_cast<const float4*>(WT);
#pragma unroll
  for (int q = 0; q < kA / 4; q++) {
    const float4 w = w4[q];
    out[4 * q] = fmaf(w.x, h, out[4 * q]);
    out[4 * q + 1] = fmaf(w.y, h, out[4 * q + 1]);
    out[4 * q + 2] = fmaf(w.z, h, out[4 * q + 2]);
    out[4 * q + 3] = fmaf(w.w, h, out[4 * q + 3]);
  }
}

// b + W row . v over kN inputs (W row kN floats, 16-byte aligned)
template <int kN>
__device__ __forceinline__ float row_dot(const float* Wrow, float b, const float* v) {
  const float4* w4 = reinterpret_cast<const float4*>(Wrow);
  float acc = b;
#pragma unroll
  for (int q = 0; q < kN / 4; q++) {
    const float4 w = w4[q];
    acc = fmaf(w.x, v[4 * q], acc);
    acc = fmaf(w.y, v[4 * q + 1], acc);
    acc = fmaf(w.z, v[4 * q + 2], acc);
    acc = fmaf(w.w, v[4 * q + 3], acc);
  }
  return acc;
}

template <int kLayers>
__global__ void __launch_bounds__(kActThreads) k_ars_act(const float* __restrict__ obs, const double* __restrict__ mean,
                                                         const double* __restrict__ var, double clip_obs, double eps,
                                                         const float* __restrict__ theta, const float* __restrict__ deltas,
                                                         float delta_std, int n_delta, int first_candidate, int epc,
                                                         int tiles, qs_ars_arch arch, float* __restrict__ actions, int n) {
  using L = Layout<kLayers>;
  __shared__ __align__(16) float sw[L::kSize];
  __shared__ double s_mean[kIn], s_std[kIn];
  const int cand_local = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int c = first_candidate + cand_local;
  const Candidate cand{theta, deltas ? deltas + size_t(c < n_delta ? c : c - n_delta) * size_t(arch_params(arch)) : nullptr,
                       delta_std, c >= n_delta};
  int off = 0, in = arch.obs_dim;
  if constexpr (kLayers >= 1) {
    off = load_layer(sw, sw + kH * kIn, kIn, kH, false, in, arch.hidden[0], arch.bias, cand, off);
    in = arch.hidden[0];
  }
  if constexpr (kLayers >= 2) {
    off = load_layer(sw + L::kHid1, sw + L::kHid1 + kH * kH, kH, kH, false, in, arch.hidden[1], arch.bias, cand, off);
    in = arch.hidden[1];
  }
  load_layer(sw + L::kOut, sw + L::kOut + L::kOutIn * kA, L::kOutIn, kA, true, in, arch.act_dim, arch.bias, cand, off);
  if (mean && threadIdx.x < arch.obs_dim) {
    s_mean[threadIdx.x] = mean[threadIdx.x];
    s_std[threadIdx.x] = sqrt(var[threadIdx.x] + eps);
  }
  __syncthreads();

  const int j = tile * kActThreads + threadIdx.x;   // index of the env among its candidate's envs
  const int e = cand_local * epc + j;
  if (j >= epc || e >= n) return;
  const int o = arch.obs_dim;
  float x[kIn];
#pragma unroll
  for (int i = 0; i < kIn; i++) {
    float v = 0.f;
    if (i < o) {
      v = obs[size_t(e) * o + i];
      if (mean) {   // VecNormalize.normalize_obs in float64, then rounded to fp32
        double d = (double(v) - s_mean[i]) / s_std[i];
        d = d < -clip_obs ? -clip_obs : (d > clip_obs ? clip_obs : d);
        v = float(d);
      }
    }
    x[i] = v;
  }
  const float* Wo = sw + L::kOut;
  float out[kA];
#pragma unroll
  for (int a = 0; a < kA; a++) out[a] = Wo[L::kOutIn * kA + a];
  if constexpr (kLayers == 0) {
#pragma unroll
    for (int i = 0; i < kIn; i++) out_fma(Wo + i * kA, x[i], out);
  } else if constexpr (kLayers == 1) {
    const float* W0 = sw;
#pragma unroll 2
    for (int h = 0; h < kH; h++) {
      const float y = activate(row_dot<kIn>(W0 + h * kIn, W0[kH * kIn + h], x), arch.activation);
      out_fma(Wo + h * kA, y, out);
    }
  } else {
    const float* W0 = sw;
    const float* W1 = sw + L::kHid1;
    float h1[kH];
#pragma unroll
    for (int h = 0; h < kH; h++) h1[h] = activate(row_dot<kIn>(W0 + h * kIn, W0[kH * kIn + h], x), arch.activation);
#pragma unroll 1
    for (int h = 0; h < kH; h++) {
      const float y = activate(row_dot<kH>(W1 + h * kH, W1[kH * kH + h], h1), arch.activation);
      out_fma(Wo + h * kA, y, out);
    }
  }
  float* dst = actions + size_t(e) * arch.act_dim;
#pragma unroll
  for (int a = 0; a < kA; a++) {
    if (a < arch.act_dim) {
      float v = arch.squash ? tanhf(out[a]) : out[a];
      v = v < -1.f ? -1.f : (v > 1.f ? 1.f : v);   // torch clamp: NaN stays NaN
      dst[a] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------ qs_obs_stats
constexpr int kStatsBlocks = 8;        // one portable cluster
constexpr int kStatsThreads = 1024;
constexpr int kWarpsPerBlock = kStatsThreads / 32;
constexpr int kWarps = kStatsBlocks * kWarpsPerBlock;
constexpr int kBatch = 8;             // rows a warp loads before it uses them

struct Moments {   // count, mean, sum of squared deviations
  double n, m, M2;
};

__device__ __forceinline__ void chan_merge(Moments& a, const Moments& b) {
  if (b.n == 0.0) return;
  if (a.n == 0.0) {
    a = b;
    return;
  }
  const double n = a.n + b.n, d = b.m - a.m;
  a.m = a.m + d * b.n / n;
  a.M2 = a.M2 + b.M2 + d * d * a.n * b.n / n;
  a.n = n;
}

__global__ void __cluster_dims__(kStatsBlocks, 1, 1) __launch_bounds__(kStatsThreads)
    k_obs_stats(const float* __restrict__ obs, uint8_t* __restrict__ alive, int n, int o, double* __restrict__ mean,
                double* __restrict__ var, double* __restrict__ count, const float* __restrict__ reward,
                const uint8_t* __restrict__ done, double* __restrict__ ret, int32_t* __restrict__ len) {
  __shared__ double s_m[kWarpsPerBlock][32], s_M2[kWarpsPerBlock][32];
  __shared__ double s_n[kWarpsPerBlock];
  __shared__ Moments s_block[32];   // this block's partial, per column
  cg::cluster_group cluster = cg::this_cluster();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gw = blockIdx.x * kWarpsPerBlock + warp;

  if (mean) {
    double K = 0.0, s1 = 0.0, s2 = 0.0;
    int cnt = 0;
    // rows gw, gw + kWarps, ... in order; the loads of kBatch rows are issued before any is used (latency, not
    // bandwidth, bounds a warp that walks its rows one by one)
    for (int r0 = gw; r0 < n; r0 += kWarps * kBatch) {
      bool av[kBatch];
      float xv[kBatch];
#pragma unroll
      for (int b = 0; b < kBatch; b++) {
        const int r = r0 + b * kWarps;
        av[b] = r < n && (!alive || alive[r]);
        xv[b] = (av[b] && lane < o) ? obs[size_t(r) * o + lane] : 0.f;
      }
#pragma unroll
      for (int b = 0; b < kBatch; b++) {
        if (!av[b]) continue;
        if (lane < o) {
          const double x = xv[b];
          if (cnt == 0) K = x;
          const double d = x - K;
          s1 += d;
          s2 += d * d;
        }
        cnt++;
      }
    }
    double m = 0.0, M2 = 0.0;
    if (cnt > 0) {
      m = K + s1 / cnt;
      M2 = fmax(s2 - s1 * s1 / cnt, 0.0);
    }
    s_m[warp][lane] = m;
    s_M2[warp][lane] = M2;
    if (lane == 0) s_n[warp] = cnt;
  }
  if (ret) {   // bookkeeping of this warp's rows, after the statistics read their alive flags
    __syncwarp();
    for (int r = gw + kWarps * lane; r < n; r += kWarps * 32) {
      const uint8_t a = alive[r];
      if (a) {
        ret[r] += double(reward[r]);
        len[r] += 1;
      }
      alive[r] = a && !done[r];
    }
  }
  if (!mean) return;
  __syncthreads();
  if (warp == 0) {
    Moments acc{0.0, 0.0, 0.0};
    for (int w = 0; w < kWarpsPerBlock; w++) chan_merge(acc, Moments{s_n[w], s_m[w][lane], s_M2[w][lane]});
    s_block[lane] = acc;
  }
  cluster.sync();
  if (blockIdx.x == 0 && warp == 0) {
    Moments acc{0.0, 0.0, 0.0};
    for (int b = 0; b < kStatsBlocks; b++) chan_merge(acc, *cluster.map_shared_rank(&s_block[lane], b));
    const double c0 = *count;
    __syncwarp();
    if (acc.n > 0.0) {
      if (lane < o) {
        // RunningMeanStd.update_from_moments, operation for operation
        const double bc = acc.n, bm = acc.m, bv = acc.M2 / bc;
        const double mu = mean[lane], s2 = var[lane];
        const double delta = __dsub_rn(bm, mu), tot = __dadd_rn(c0, bc);
        const double m_a = __dmul_rn(s2, c0), m_b = __dmul_rn(bv, bc);
        mean[lane] = __dadd_rn(mu, __ddiv_rn(__dmul_rn(delta, bc), tot));
        const double corr = __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), c0), bc), tot);
        var[lane] = __ddiv_rn(__dadd_rn(__dadd_rn(m_a, m_b), corr), tot);
      }
      if (lane == 0) *count = __dadd_rn(c0, acc.n);
    }
  }
  cluster.sync();   // block 0 has read every block's partial before any block exits
}

}  // namespace

extern "C" int qs_obs_stats(const float* obs, uint8_t* alive, int n, int o, double* mean, double* var, double* count,
                            const float* reward, const uint8_t* done, double* ret, int32_t* len, void* stream) {
  using qs::abi_fail;
  if (n < 1) return abi_fail(QS_ERR_ARG, "qs_obs_stats: n must be at least 1");
  const bool stats = mean || var || count;
  const bool book = reward || done || ret || len;
  if (!stats && !book) return abi_fail(QS_ERR_ARG, "qs_obs_stats: neither statistics nor bookkeeping requested");
  if (stats && (!mean || !var || !count || !obs))
    return abi_fail(QS_ERR_ARG, "qs_obs_stats: obs, mean, var and count must all be given for the statistics");
  if (stats && (o < 1 || o > QS_MAX_OBS)) return abi_fail(QS_ERR_ARG, "qs_obs_stats: o must lie in [1, QS_MAX_OBS]");
  if (book && (!reward || !done || !ret || !len || !alive))
    return abi_fail(QS_ERR_ARG, "qs_obs_stats: bookkeeping needs reward, done, ret, len and alive");
  k_obs_stats<<<kStatsBlocks, kStatsThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      obs, alive, n, o, stats ? mean : nullptr, var, count, reward, done, book ? ret : nullptr, len);
  qs::abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_obs_stats: ") + cudaGetErrorString(e));
  return QS_OK;
}

extern "C" int qs_ars_act(const float* obs, const double* mean, const double* var, double clip_obs, double eps,
                          const float* theta, const float* deltas, float delta_std, int n_delta, int first_candidate,
                          int envs_per_candidate, const qs_ars_arch* arch, float* actions, int n, void* stream) {
  using qs::abi_fail;
  if (!arch) return abi_fail(QS_ERR_ARG, "qs_ars_act: arch is NULL");
  const qs_ars_arch a = *arch;
  if (a.obs_dim < 1 || a.obs_dim > QS_MAX_OBS || a.act_dim < 1 || a.act_dim > QS_ARS_MAX_ACT || a.n_hidden < 0 ||
      a.n_hidden > 2 || (a.activation != QS_ARS_RELU && a.activation != QS_ARS_TANH) || (a.bias != 0 && a.bias != 1) ||
      (a.squash != 0 && a.squash != 1))
    return abi_fail(QS_ERR_ARG, "qs_ars_act: unsupported policy architecture");
  for (int l = 0; l < a.n_hidden; l++)
    if (a.hidden[l] < 1 || a.hidden[l] > QS_ARS_MAX_HIDDEN)
      return abi_fail(QS_ERR_ARG, "qs_ars_act: hidden sizes must lie in [1, QS_ARS_MAX_HIDDEN]");
  if (n < 1 || envs_per_candidate < 1 || n_delta < 1)
    return abi_fail(QS_ERR_ARG, "qs_ars_act: n, envs_per_candidate and n_delta must be at least 1");
  if (!obs || !theta || !actions || (mean && !var))
    return abi_fail(QS_ERR_ARG, "qs_ars_act: obs, theta, actions (and var with mean) must be given");
  const int64_t n_cand = (int64_t(n) + envs_per_candidate - 1) / envs_per_candidate;
  if (first_candidate < 0 || first_candidate + n_cand > 2 * int64_t(n_delta))
    return abi_fail(QS_ERR_ARG, "qs_ars_act: a candidate index lies outside [0, 2 n_delta)");
  const int tiles = (envs_per_candidate + kActThreads - 1) / kActThreads;
  if (n_cand * tiles > INT32_MAX) return abi_fail(QS_ERR_ARG, "qs_ars_act: too many blocks");
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned grid = unsigned(n_cand * tiles);
#define QS_ARS_LAUNCH(L)                                                                                            \
  k_ars_act<L><<<grid, kActThreads, 0, s>>>(obs, mean, var, clip_obs, eps, theta, deltas, delta_std, n_delta,        \
                                            first_candidate, envs_per_candidate, tiles, a, actions, n)
  if (a.n_hidden == 0) QS_ARS_LAUNCH(0);
  else if (a.n_hidden == 1) QS_ARS_LAUNCH(1);
  else QS_ARS_LAUNCH(2);
#undef QS_ARS_LAUNCH
  qs::abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_ars_act: ") + cudaGetErrorString(e));
  return QS_OK;
}
