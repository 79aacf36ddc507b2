// qs_ppo.cu -- qs_ppo_act, qs_ppo_reward and qs_ppo_gae (include/qs_b200.h): the per-step kernels of batched PPO
// training (quadruped_springs_b200/ppo.py).  Its own translation unit: the step's kernels and their compile are not touched.
//
// qs_ppo_act: one thread per env.  A block loads the shared parameters once into shared memory, zero-padded to fixed
// shapes (inputs to QS_MAX_OBS, hidden layers to QS_ARS_MAX_HIDDEN, actions to QS_ARS_MAX_ACT), so every thread runs the
// same unrolled actor and critic with its activations in registers; the padded terms add exact zeros.  An env's noise is
// Philox keyed by (seed, global env id, iteration, step), so its action has the same bits alone, in any batch or shard.
//
// qs_ppo_reward: one cluster of kBlocks blocks (like k_obs_stats in qs_ars.cu).  Thread g owns rows g, g + kThreads, ...
// in order; the per-thread moments of the discounted returns are merged by a fixed shuffle tree in each warp, the warps
// of a block in order, and the blocks in order through distributed shared memory.  The result depends on the rows and
// their order only.  The Chan merge is a copy of qs_ars.cu's so that the ARS kernels' SASS stays as it is.
//
// qs_ppo_gae: one thread per env, a reverse scan over step-major [n_steps, n] arrays (loads coalesced across envs).
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/qs_b200.h"
#include "qs_env.cuh"   // Philox4x32-10 (qs::normal4)

namespace qs {
int abi_fail(int code, const std::string& msg);  // qs_kernels.cu: error text of qs_last_error
void abi_count_launch();                          // qs_kernels.cu: qs_launch_count
}  // namespace qs

namespace cg = cooperative_groups;

namespace {

// ------------------------------------------------------------------------------------------------ qs_ppo_act
constexpr int kIn = QS_MAX_OBS;
constexpr int kH = QS_ARS_MAX_HIDDEN;
constexpr int kA = QS_ARS_MAX_ACT;
constexpr int kActThreads = 128;
// salt of the policy-noise key: the env's own observation noise uses the seed unchanged
constexpr uint64_t kNoiseSalt = 0x50504F5F4E4F4953ull;   // "PPO_NOIS"

// padded shared layout, in floats: the actor extractor, the critic extractor (each: per hidden layer W [kH][in] then
// b [kH]), the action head transposed WT [in][kA] then b [kA], the value head w [in] then b (padded to 4), log_std [kA]
template <int kLayers>
struct Layout {
  static constexpr int kHid1 = kH * kIn + kH;                                 // second hidden layer of an extractor
  static constexpr int kExt = kLayers == 0 ? 0 : (kLayers == 1 ? kHid1 : kHid1 + kH * kH + kH);
  static constexpr int kOutIn = kLayers == 0 ? kIn : kH;
  static constexpr int kPi = 0, kVf = kExt;
  static constexpr int kAct = 2 * kExt;
  static constexpr int kVal = kAct + kOutIn * kA + kA;
  static constexpr int kLogStd = kVal + kOutIn + 4;
  static constexpr int kSize = kLogStd + kA;
};
static_assert(Layout<2>::kVf % 4 == 0 && Layout<2>::kAct % 4 == 0 && Layout<2>::kVal % 4 == 0 &&
              Layout<1>::kAct % 4 == 0 && Layout<0>::kVal % 4 == 0, "float4 layout");

// one Linear layer of `in` x `out` real weights at theta offset `off` into a padded shared block; returns the next offset
__device__ int load_layer(float* W, float* b, int in_pad, int out_pad, bool transposed, int in, int out,
                          const float* __restrict__ theta, int off) {
  for (int q = threadIdx.x; q < in_pad * out_pad; q += blockDim.x) {
    const int row = transposed ? q % out_pad : q / in_pad;   // output index
    const int col = transposed ? q / out_pad : q % in_pad;   // input index
    W[q] = (row < out && col < in) ? theta[off + row * in + col] : 0.f;
  }
  for (int q = threadIdx.x; q < out_pad; q += blockDim.x) b[q] = q < out ? theta[off + out * in + q] : 0.f;
  return off + out * in + out;
}

template <int kLayers>
__device__ int load_extractor(float* base, const qs_ppo_arch& a, const float* __restrict__ theta, int off) {
  using L = Layout<kLayers>;
  if constexpr (kLayers >= 1) off = load_layer(base, base + kH * kIn, kIn, kH, false, a.obs_dim, a.hidden[0], theta, off);
  if constexpr (kLayers >= 2)
    off = load_layer(base + L::kHid1, base + L::kHid1 + kH * kH, kH, kH, false, a.hidden[0], a.hidden[1], theta, off);
  return off;
}

__device__ __forceinline__ float activate(float v, int act) { return act == QS_ARS_TANH ? tanhf(v) : fmaxf(v, 0.f); }

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

// Head(extractor(x)) where the head is either the action net (kOut = kA outputs, transposed weights) or the value net
// (one output); `head(y, i)` consumes the extractor's output i.
template <int kLayers, typename Head>
__device__ __forceinline__ void run_extractor(const float* ext, const float* x, int act, Head head) {
  using L = Layout<kLayers>;
  if constexpr (kLayers == 0) {
#pragma unroll
    for (int i = 0; i < kIn; i++) head(x[i], i);
  } else if constexpr (kLayers == 1) {
#pragma unroll 2
    for (int h = 0; h < kH; h++) head(activate(row_dot<kIn>(ext + h * kIn, ext[kH * kIn + h], x), act), h);
  } else {
    const float* W1 = ext + L::kHid1;
    float h1[kH];
#pragma unroll
    for (int h = 0; h < kH; h++) h1[h] = activate(row_dot<kIn>(ext + h * kIn, ext[kH * kIn + h], x), act);
#pragma unroll 1
    for (int h = 0; h < kH; h++) head(activate(row_dot<kH>(W1 + h * kH, W1[kH * kH + h], h1), act), h);
  }
}

template <int kLayers>
__device__ __forceinline__ float critic(const float* sw, const float* x, int act) {
  using L = Layout<kLayers>;
  const float* wv = sw + L::kVal;
  float v = wv[L::kOutIn];
  run_extractor<kLayers>(sw + L::kVf, x, act, [&](float y, int i) { v = fmaf(wv[i], y, v); });
  return v;
}

// VecNormalize.normalize_obs in float64, rounded to fp32 (VecNormalizeTorch's operations, so the same bits)
__device__ __forceinline__ void normalise(const float* __restrict__ row, int o, const double* s_mean, const double* s_std,
                                          bool norm, double clip_obs, float* x) {
#pragma unroll
  for (int i = 0; i < kIn; i++) {
    float v = 0.f;
    if (i < o) {
      v = row[i];
      if (norm) {
        double d = (double(v) - s_mean[i]) / s_std[i];
        d = d < -clip_obs ? -clip_obs : (d > clip_obs ? clip_obs : d);
        v = float(d);
      }
    }
    x[i] = v;
  }
}

template <int kLayers>
__global__ void __launch_bounds__(kActThreads) k_ppo_act(const qs_ppo_args p, const qs_ppo_arch a) {
  using L = Layout<kLayers>;
  extern __shared__ __align__(16) float sw[];
  __shared__ double s_mean[kIn], s_std[kIn];
  // theta (module parameters before its children's): log_std, policy_net layers, value_net layers, action_net (W, b),
  // value_net (W, b)
  for (int q = threadIdx.x; q < kA; q += blockDim.x) sw[L::kLogStd + q] = q < a.act_dim ? p.theta[q] : 0.f;
  int off = load_extractor<kLayers>(sw + L::kPi, a, p.theta, a.act_dim);
  off = load_extractor<kLayers>(sw + L::kVf, a, p.theta, off);
  const int last = kLayers == 0 ? a.obs_dim : a.hidden[kLayers - 1];
  off = load_layer(sw + L::kAct, sw + L::kAct + L::kOutIn * kA, L::kOutIn, kA, true, last, a.act_dim, p.theta, off);
  load_layer(sw + L::kVal, sw + L::kVal + L::kOutIn, L::kOutIn, 1, false, last, 1, p.theta, off);
  const bool norm = p.obs_mean != nullptr;
  if (norm && threadIdx.x < a.obs_dim) {
    s_mean[threadIdx.x] = p.obs_mean[threadIdx.x];
    s_std[threadIdx.x] = sqrt(p.obs_var[threadIdx.x] + p.epsilon);
  }
  __syncthreads();

  const int e = blockIdx.x * kActThreads + threadIdx.x;
  if (e >= p.n) return;
  const int o = a.obs_dim, A = a.act_dim;
  const size_t n = size_t(p.n), t = size_t(p.step);
  float x[kIn];

  // the previous step ended this env's episode by its time limit: rewards[t - 1] += gamma V(terminal obs), the terminal
  // observation normalised with the statistics that already include that step (VecNormalize.step_wait)
  if (p.step > 0 && p.prev_truncated && p.episode_start[e] && p.prev_truncated[e]) {
    normalise(p.terminal_obs + size_t(e) * o, o, s_mean, s_std, norm, p.clip_obs, x);
    const float vt = critic<kLayers>(sw, x, a.activation);
    float* r = p.buf_rewards + (t - 1) * n + e;
    *r = __fadd_rn(*r, __fmul_rn(p.gamma, vt));
  }

  normalise(p.obs + size_t(e) * o, o, s_mean, s_std, norm, p.clip_obs, x);
  const float value = critic<kLayers>(sw, x, a.activation);
  if (p.values_only) {
    p.last_values[e] = value;
    return;
  }
  float mean[kA];
  const float* Wa = sw + L::kAct;
#pragma unroll
  for (int i = 0; i < kA; i++) mean[i] = Wa[L::kOutIn * kA + i];
  run_extractor<kLayers>(sw + L::kPi, x, a.activation, [&](float y, int i) { out_fma(Wa + i * kA, y, mean); });

  if (p.mean_out) {
#pragma unroll
    for (int i = 0; i < kA; i++)
      if (i < A) p.mean_out[size_t(e) * A + i] = mean[i];
  }
  if (p.deterministic) {
#pragma unroll
    for (int i = 0; i < kA; i++)
      if (i < A) p.actions[size_t(e) * A + i] = fminf(fmaxf(mean[i], -1.f), 1.f);
    return;
  }

  // a = mean + std * eps (torch's Normal.rsample: two roundings); log_prob = sum_i Normal(mean_i, std_i).log_prob(a_i)
  float eps[kA];
  const uint64_t gid = uint64_t(p.env_id_offset + e);
#pragma unroll
  for (int b = 0; b < kA / 4; b++)
    if (4 * b < A) qs::normal4(p.seed ^ kNoiseSalt, gid, uint32_t(p.iteration), uint32_t(p.step), uint32_t(b), eps + 4 * b);
  const float* log_std = sw + L::kLogStd;
  float lp = 0.f;
  float* act_row = p.buf_actions + (t * n + e) * A;
  float* env_row = p.actions + size_t(e) * A;
#pragma unroll
  for (int i = 0; i < kA; i++) {
    if (i < A) {
      const float s = expf(log_std[i]);
      const float ai = __fadd_rn(mean[i], __fmul_rn(eps[i], s));
      const float d = __fsub_rn(ai, mean[i]);
      const float q = __fdiv_rn(-__fmul_rn(d, d), __fmul_rn(2.f, __fmul_rn(s, s)));
      lp = __fadd_rn(lp, __fsub_rn(__fsub_rn(q, logf(s)), 0.91893853320467274178f));
      act_row[i] = ai;
      env_row[i] = fminf(fmaxf(ai, -1.f), 1.f);
    }
  }
  float* obs_row = p.buf_obs + (t * n + e) * o;
#pragma unroll
  for (int i = 0; i < kIn; i++)
    if (i < o) obs_row[i] = x[i];
  p.buf_values[t * n + e] = value;
  p.buf_log_probs[t * n + e] = lp;
  p.buf_episode_starts[t * n + e] = p.episode_start[e] ? 1.f : 0.f;
}

// ------------------------------------------------------------------------------------------------ qs_ppo_reward
constexpr int kBlocks = 8;   // one portable cluster
constexpr int kThreads = 1024;
constexpr int kWarpsPerBlock = kThreads / 32;
constexpr int kAll = kBlocks * kThreads;

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

struct Part {   // one reduction unit: return moments, finished episodes (count, sum of returns, sum of lengths), and
                // the sum of every row's raw reward
  Moments mo;
  double cnt, ret, len, rew;
};

__device__ __forceinline__ void merge(Part& a, const Part& b) {
  chan_merge(a.mo, b.mo);
  a.cnt += b.cnt;
  a.ret += b.ret;
  a.len += b.len;
  a.rew += b.rew;
}

__device__ __forceinline__ Part shfl_down(const Part& p, int d) {
  Part q;
  q.mo.n = __shfl_down_sync(0xffffffffu, p.mo.n, d);
  q.mo.m = __shfl_down_sync(0xffffffffu, p.mo.m, d);
  q.mo.M2 = __shfl_down_sync(0xffffffffu, p.mo.M2, d);
  q.cnt = __shfl_down_sync(0xffffffffu, p.cnt, d);
  q.ret = __shfl_down_sync(0xffffffffu, p.ret, d);
  q.len = __shfl_down_sync(0xffffffffu, p.len, d);
  q.rew = __shfl_down_sync(0xffffffffu, p.rew, d);
  return q;
}

__global__ void __cluster_dims__(kBlocks, 1, 1) __launch_bounds__(kThreads)
    k_ppo_reward(const float* __restrict__ reward, const uint8_t* __restrict__ done, int n, double* __restrict__ ret,
                 double* __restrict__ ret_mean, double* __restrict__ ret_var, double* __restrict__ ret_count,
                 double gamma, double eps, double clip_reward, float* __restrict__ reward_out,
                 double* __restrict__ ep_return, int32_t* __restrict__ ep_length, double* __restrict__ totals) {
  __shared__ Part s_warp[kWarpsPerBlock];
  __shared__ Part s_block;
  __shared__ double s_scale;   // block 0: sqrt(var_ret + eps) after the update
  cg::cluster_group cluster = cg::this_cluster();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = blockIdx.x * kThreads + threadIdx.x;
  const bool norm = ret_mean != nullptr;

  Part acc{{0.0, 0.0, 0.0}, 0.0, 0.0, 0.0, 0.0};
  double K = 0.0, s1 = 0.0, s2 = 0.0;
  int cnt = 0;
  for (int r = g; r < n; r += kAll) {
    const float rw = reward[r];
    const bool d = done[r] != 0;
    if (norm) {   // VecNormalize._update_reward: ret = ret * gamma + r, merged into ret_rms, then zeroed on done
      const double x = __dadd_rn(__dmul_rn(ret[r], gamma), double(rw));
      if (cnt == 0) K = x;
      const double dx = x - K;
      s1 += dx;
      s2 += dx * dx;
      cnt++;
      ret[r] = d ? 0.0 : x;
    }
    // Monitor's episode return and length (raw rewards), folded into the rollout totals on done
    const double er = ep_return[r] + double(rw);
    const int32_t el = ep_length[r] + 1;
    acc.rew += double(rw);
    if (d) {
      acc.cnt += 1.0;
      acc.ret += er;
      acc.len += double(el);
    }
    ep_return[r] = d ? 0.0 : er;
    ep_length[r] = d ? 0 : el;
  }
  if (cnt > 0) acc.mo = Moments{double(cnt), K + s1 / cnt, fmax(s2 - s1 * s1 / cnt, 0.0)};
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    const Part q = shfl_down(acc, d);
    merge(acc, q);
  }
  if (lane == 0) s_warp[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    Part b = s_warp[0];
    for (int w = 1; w < kWarpsPerBlock; w++) merge(b, s_warp[w]);
    s_block = b;
  }
  cluster.sync();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    Part t = s_block;
    for (int b = 1; b < kBlocks; b++) merge(t, *cluster.map_shared_rank(&s_block, b));
    if (totals) {
      totals[0] = __dadd_rn(totals[0], t.cnt);
      totals[1] = __dadd_rn(totals[1], t.ret);
      totals[2] = __dadd_rn(totals[2], t.len);
      totals[3] = __dadd_rn(totals[3], t.rew);
    }
    if (norm) {
      double var = *ret_var;
      if (t.mo.n > 0.0) {   // RunningMeanStd.update_from_moments, operation for operation
        const double c0 = *ret_count, bc = t.mo.n, bm = t.mo.m, bv = t.mo.M2 / bc;
        const double mu = *ret_mean;
        const double delta = __dsub_rn(bm, mu), tot = __dadd_rn(c0, bc);
        const double m_a = __dmul_rn(var, c0), m_b = __dmul_rn(bv, bc);
        *ret_mean = __dadd_rn(mu, __ddiv_rn(__dmul_rn(delta, bc), tot));
        const double corr = __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), c0), bc), tot);
        var = __ddiv_rn(__dadd_rn(__dadd_rn(m_a, m_b), corr), tot);
        *ret_var = var;
        *ret_count = tot;
      }
      s_scale = sqrt(__dadd_rn(var, eps));
    }
  }
  cluster.sync();
  const double scale = norm ? *cluster.map_shared_rank(&s_scale, 0) : 1.0;
  for (int r = g; r < n; r += kAll) {
    const float rw = reward[r];
    if (norm) {   // VecNormalize.normalize_reward
      double v = double(rw) / scale;
      v = v < -clip_reward ? -clip_reward : (v > clip_reward ? clip_reward : v);
      reward_out[r] = float(v);
    } else {
      reward_out[r] = rw;
    }
  }
  cluster.sync();   // block 0's s_scale has been read by every block before it exits
}

// ------------------------------------------------------------------------------------------------ qs_ppo_gae
// RolloutBuffer.compute_returns_and_advantage in fp32, operation for operation (numpy's float32 arithmetic)
__global__ void k_ppo_gae(const float* __restrict__ rewards, const float* __restrict__ values,
                          const float* __restrict__ episode_starts, const float* __restrict__ last_values,
                          const uint8_t* __restrict__ last_dones, int n_steps, int n, float gamma, float gamma_lambda,
                          float* __restrict__ advantages, float* __restrict__ returns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float last_gae = 0.f;
  float next_value = last_values[e];
  float next_non_terminal = last_dones[e] ? 0.f : 1.f;
  for (int t = n_steps - 1; t >= 0; t--) {
    const size_t k = size_t(t) * n + e;
    const float v = values[k];
    const float delta = __fsub_rn(__fadd_rn(rewards[k], __fmul_rn(__fmul_rn(gamma, next_value), next_non_terminal)), v);
    last_gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gamma_lambda, next_non_terminal), last_gae));
    advantages[k] = last_gae;
    returns[k] = __fadd_rn(last_gae, v);
    next_value = v;
    next_non_terminal = __fsub_rn(1.f, episode_starts[k]);
  }
}

template <int kLayers>
int launch_act(const qs_ppo_args& p, const qs_ppo_arch& a, cudaStream_t s) {
  constexpr size_t smem = sizeof(float) * Layout<kLayers>::kSize;
  // above the 48 KB default with two hidden layers; the attribute belongs to a device, so it is set once per device
  static uint64_t configured = 0;   // bit d: set on device d
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess && (dev >= 64 || !((configured >> dev) & 1u))) {
    e = cudaFuncSetAttribute(k_ppo_act<kLayers>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e == cudaSuccess && dev < 64) configured |= uint64_t(1) << dev;
  }
  if (e != cudaSuccess) return qs::abi_fail(QS_ERR_CUDA, std::string("qs_ppo_act: ") + cudaGetErrorString(e));
  const unsigned grid = unsigned((p.n + kActThreads - 1) / kActThreads);
  k_ppo_act<kLayers><<<grid, kActThreads, smem, s>>>(p, a);
  return QS_OK;
}

}  // namespace

extern "C" int qs_ppo_act(const qs_ppo_args* args, const qs_ppo_arch* arch, void* stream) {
  using qs::abi_fail;
  if (!args || !arch) return abi_fail(QS_ERR_ARG, "qs_ppo_act: args and arch must be given");
  const qs_ppo_args p = *args;
  const qs_ppo_arch a = *arch;
  if (a.obs_dim < 1 || a.obs_dim > QS_MAX_OBS || a.act_dim < 1 || a.act_dim > QS_ARS_MAX_ACT || a.n_hidden < 0 ||
      a.n_hidden > 2 || (a.activation != QS_ARS_RELU && a.activation != QS_ARS_TANH))
    return abi_fail(QS_ERR_ARG, "qs_ppo_act: unsupported policy architecture");
  for (int l = 0; l < a.n_hidden; l++)
    if (a.hidden[l] < 1 || a.hidden[l] > QS_ARS_MAX_HIDDEN)
      return abi_fail(QS_ERR_ARG, "qs_ppo_act: hidden sizes must lie in [1, QS_ARS_MAX_HIDDEN]");
  if (p.n < 1) return abi_fail(QS_ERR_ARG, "qs_ppo_act: n must be at least 1");
  if (!p.obs || !p.theta || (p.obs_mean && !p.obs_var))
    return abi_fail(QS_ERR_ARG, "qs_ppo_act: obs, theta (and obs_var with obs_mean) must be given");
  if (p.prev_truncated && (!p.terminal_obs || !p.buf_rewards || !p.episode_start))
    return abi_fail(QS_ERR_ARG, "qs_ppo_act: the time-limit bootstrap needs terminal_obs, episode_start and buf_rewards");
  // the bootstrap writes buf_rewards row step - 1 and a sampling call writes row step
  if (p.step < 0 || p.step > p.n_steps || (!p.values_only && !p.deterministic && p.step == p.n_steps))
    return abi_fail(QS_ERR_ARG, "qs_ppo_act: step must lie in [0, n_steps) for a sampling call and in [0, n_steps] "
                                "otherwise");
  if (p.values_only) {
    if (!p.last_values) return abi_fail(QS_ERR_ARG, "qs_ppo_act: values_only needs last_values");
  } else if (p.deterministic) {
    if (!p.actions) return abi_fail(QS_ERR_ARG, "qs_ppo_act: deterministic needs actions");
  } else if (!p.actions || !p.buf_obs || !p.buf_actions || !p.buf_values || !p.buf_log_probs ||
             !p.buf_episode_starts || !p.episode_start) {
    return abi_fail(QS_ERR_ARG, "qs_ppo_act: a sampling call needs actions, episode_start and every buffer row");
  }
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int rc = a.n_hidden == 0 ? launch_act<0>(p, a, s) : (a.n_hidden == 1 ? launch_act<1>(p, a, s) : launch_act<2>(p, a, s));
  if (rc != QS_OK) return rc;
  qs::abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_ppo_act: ") + cudaGetErrorString(e));
  return QS_OK;
}

extern "C" int qs_ppo_reward(const float* reward, const uint8_t* done, int n, double* ret, double* ret_mean,
                             double* ret_var, double* ret_count, double gamma, double epsilon, double clip_reward,
                             float* reward_out, double* ep_return, int32_t* ep_length, double* totals, void* stream) {
  using qs::abi_fail;
  if (n < 1) return abi_fail(QS_ERR_ARG, "qs_ppo_reward: n must be at least 1");
  if (!reward || !done || !reward_out || !ep_return || !ep_length)
    return abi_fail(QS_ERR_ARG, "qs_ppo_reward: reward, done, reward_out, ep_return and ep_length must be given");
  const bool norm = ret || ret_mean || ret_var || ret_count;
  if (norm && (!ret || !ret_mean || !ret_var || !ret_count))
    return abi_fail(QS_ERR_ARG, "qs_ppo_reward: ret, ret_mean, ret_var and ret_count are given together");
  k_ppo_reward<<<kBlocks, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      reward, done, n, ret, norm ? ret_mean : nullptr, ret_var, ret_count, gamma, epsilon, clip_reward, reward_out,
      ep_return, ep_length, totals);
  qs::abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_ppo_reward: ") + cudaGetErrorString(e));
  return QS_OK;
}

extern "C" int qs_ppo_gae(const float* rewards, const float* values, const float* episode_starts,
                          const float* last_values, const uint8_t* last_dones, int n_steps, int n, double gamma,
                          double gae_lambda, float* advantages, float* returns, void* stream) {
  using qs::abi_fail;
  if (n < 1 || n_steps < 1) return abi_fail(QS_ERR_ARG, "qs_ppo_gae: n and n_steps must be at least 1");
  if (!rewards || !values || !episode_starts || !last_values || !last_dones || !advantages || !returns)
    return abi_fail(QS_ERR_ARG, "qs_ppo_gae: every array must be given");
  // numpy: a Python float meets a float32 array as float32; gamma * gae_lambda is formed in double first
  k_ppo_gae<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      rewards, values, episode_starts, last_values, last_dones, n_steps, n, float(gamma), float(gamma * gae_lambda),
      advantages, returns);
  qs::abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_ppo_gae: ") + cudaGetErrorString(e));
  return QS_OK;
}
