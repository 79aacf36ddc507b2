// qs_render.cu -- qs_render (include/qs_b200.h): camera images of robots on the ground plane, ray cast on the GPU.
//
// What is drawn is what the contact code collides: the plane z = 0 and the Go1's 18 collision primitives (trunk box,
// imu box, per leg a hip cylinder, thigh box, calf box and foot sphere), posed from a qs_get_state row with leg_kin and
// the shape constants of ModelConstT<float> (qs_model_host.h build_model).  Its own translation unit: the step's
// kernels and their compile are not touched.
//
// One block renders a tile of kTile consecutive pixels (row-major) of one image.  Its prologue poses the image's
// primitives and a bounding sphere around them into shared memory and inverts the camera's P V in fp64; then every
// thread casts one primary ray and, for a lit surface, one shadow ray.  The ray set-up (unprojection, the ground hit) is
// fp64 so that grazing views keep metric depth; the primitive tests are fp32.  Nothing depends on the other images of
// the batch or on which outputs are requested, so an image's bits do not depend on either.
#include <cuda_runtime.h>

#include <climits>
#include <string>

#include "qs_model_host.h"
#include "qs_physics.cuh"

namespace qs {
int abi_fail(int code, const std::string& msg);  // qs_kernels.cu: error text of qs_last_error
void abi_count_launch();                          // qs_kernels.cu: qs_launch_count
}  // namespace qs

using namespace qs;

namespace {

constexpr int kTile = 256;   // pixels per block = threads per block
constexpr int kPrims = 18;   // primitive i is URDF link i: trunk, imu, then hip / thigh / calf / foot of FR, FL, RR, RL

// The look of the image, in one place (restated by tests/test_render.py).  shade = albedo (ambient + (1 - ambient)
// max(0, n.L) s), s = 0 where a ray from hit + shadow_offset n toward L hits a robot primitive.
struct Style {
  float light[3];        // unit vector toward the light, not axis-aligned
  float ambient;
  float shadow_offset;   // m, along the surface normal
  float albedo[5][3];    // trunk / imu, hip, thigh, calf, foot (0-255)
  float ground[2][3];    // 1 m checkerboard: (floor x + floor y) even, odd
  float sky[3];
};
__constant__ Style kStyle = {
    {0.3f, -0.4f, 0.8660254f}, 0.35f, 1e-4f,
    {{80.f, 88.f, 104.f}, {214.f, 132.f, 44.f}, {66.f, 128.f, 196.f}, {150.f, 156.f, 164.f}, {40.f, 40.f, 44.f}},
    {{176.f, 176.f, 176.f}, {128.f, 128.f, 128.f}},
    {160.f, 196.f, 232.f}};

enum { SHAPE_BOX = 0, SHAPE_CYL = 1, SHAPE_SPHERE = 2 };
__host__ __device__ constexpr int prim_shape(int i) {
  return i < 2 ? SHAPE_BOX : ((i - 2) % 4 == 0 ? SHAPE_CYL : ((i - 2) % 4 == 3 ? SHAPE_SPHERE : SHAPE_BOX));
}
__host__ __device__ constexpr int prim_kind(int i) { return i < 2 ? 0 : 1 + (i - 2) % 4; }

struct Prim {
  float R[9];   // local -> world rotation, row-major
  float c[3];   // centre (world)
  float e[3];   // box: half extents; cylinder: radius, half length (axis = local z); sphere: radius
};
struct Setup {
  Prim prim[kPrims];
  double Minv[16];  // inverse(P V), row-major
  double V2[4];     // row 2 of V: eye z = V2 . (x, 1)
  float far_;       // far plane of the projection (the rays start on the near plane)
  float bs[4];      // bounding sphere of the primitives: centre, radius
  int robot;        // 0: the state row is not finite, no robot is drawn
};

__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
__device__ __forceinline__ void set_prim(Prim& p, const float* R, const float* pos, const float* Rb, const float* loc,
                                         float e0, float e1, float e2) {
  float w[3];
  m3_v(Rb, loc, w);
#pragma unroll
  for (int i = 0; i < 9; i++) p.R[i] = R[i];
#pragma unroll
  for (int i = 0; i < 3; i++) p.c[i] = pos[i] + w[i];
  p.e[0] = e0; p.e[1] = e1; p.e[2] = e2;
}

// general 4x4 inverse (row-major), cofactor expansion; a singular matrix gives non-finite entries, hence misses
__device__ void inverse4(const double* m, double* inv) {
  inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
  inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
  inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
  inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
  inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
  inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
  inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
  inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
  inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
  inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
  inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
  inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
  inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
  inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
  inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
  inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
  const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
  const double r = 1.0 / det;
  for (int i = 0; i < 16; i++) inv[i] *= r;
}

// Ray (o, d) against primitive i in its local frame: the entry / exit parameters of the solid [tn, tf] (tn > tf: no
// intersection) and the outward local normal at the entry.
__device__ __forceinline__ void intersect(int i, const Prim& p, const float* o, const float* d, float& tn, float& tf,
                                          float* nl) {
  float ol[3], dl[3];
  {
    const float v[3] = {o[0] - p.c[0], o[1] - p.c[1], o[2] - p.c[2]};
    m3t_v(p.R, v, ol);
    m3t_v(p.R, d, dl);
  }
  const int shape = prim_shape(i);
  if (shape == SHAPE_SPHERE) {
    const float r = p.e[0];
    const float b = dot3(ol, dl);
    const float q[3] = {ol[0] - b * dl[0], ol[1] - b * dl[1], ol[2] - b * dl[2]};   // closest approach, no cancellation
    const float disc = r * r - dot3(q, q);
    if (disc < 0.f) { tn = 1.f; tf = 0.f; return; }
    const float s = sqrtf(disc);
    tn = -b - s; tf = -b + s;
#pragma unroll
    for (int a = 0; a < 3; a++) nl[a] = (ol[a] + tn * dl[a]) / r;
  } else if (shape == SHAPE_BOX) {
    tn = -INFINITY; tf = INFINITY;
    int ax = 0;
#pragma unroll
    for (int a = 0; a < 3; a++) {
      const float inv = 1.f / dl[a];
      const float t1 = (-p.e[a] - ol[a]) * inv, t2 = (p.e[a] - ol[a]) * inv;
      const float lo = fminf(t1, t2), hi = fmaxf(t1, t2);
      if (lo > tn) { tn = lo; ax = a; }
      tf = fminf(tf, hi);
    }
    nl[0] = nl[1] = nl[2] = 0.f;
    nl[ax] = dl[ax] > 0.f ? -1.f : 1.f;
  } else {  // capped cylinder along local z
    const float r = p.e[0], hl = p.e[1];
    const float a2 = dl[0] * dl[0] + dl[1] * dl[1];
    float s0, s1;
    if (a2 > 1e-12f) {
      const float b = ol[0] * dl[0] + ol[1] * dl[1], cr = ol[0] * dl[1] - ol[1] * dl[0];
      const float disc = a2 * r * r - cr * cr;       // = b^2 - a2 (|o_xy|^2 - r^2), without the cancellation
      if (disc < 0.f) { tn = 1.f; tf = 0.f; return; }
      const float s = sqrtf(disc);
      s0 = (-b - s) / a2; s1 = (-b + s) / a2;
    } else {
      if (ol[0] * ol[0] + ol[1] * ol[1] > r * r) { tn = 1.f; tf = 0.f; return; }
      s0 = -INFINITY; s1 = INFINITY;
    }
    const float inv = 1.f / dl[2];
    const float t1 = (-hl - ol[2]) * inv, t2 = (hl - ol[2]) * inv;
    const float z0 = fminf(t1, t2), z1 = fmaxf(t1, t2);
    tn = fmaxf(s0, z0); tf = fminf(s1, z1);
    if (s0 >= z0) {
      const float x = ol[0] + tn * dl[0], y = ol[1] + tn * dl[1];
      const float rn = rsqrtf(x * x + y * y);
      nl[0] = x * rn; nl[1] = y * rn; nl[2] = 0.f;
    } else {
      nl[0] = 0.f; nl[1] = 0.f; nl[2] = dl[2] > 0.f ? -1.f : 1.f;
    }
  }
}

// does the ray (o, d), t >= 0, come within the (slightly inflated) bounding sphere?
__device__ __forceinline__ bool near_robot(const Setup& S, const float* o, const float* d) {
  const float oc[3] = {o[0] - S.bs[0], o[1] - S.bs[1], o[2] - S.bs[2]};
  const float r = S.bs[3];
  const float c = dot3(oc, oc) - r * r;
  if (c <= 0.f) return true;
  const float b = dot3(oc, d);
  if (b >= 0.f) return false;
  const float q[3] = {oc[0] - b * d[0], oc[1] - b * d[1], oc[2] - b * d[2]};
  return dot3(q, q) <= r * r;
}

__global__ void __launch_bounds__(kTile) k_render(const __grid_constant__ ModelConstT<float> M,
                                                  const float* __restrict__ states, const float* __restrict__ cams,
                                                  int tiles, int W, int H, uint8_t* __restrict__ rgb,
                                                  float* __restrict__ depth, int32_t* __restrict__ seg) {
  __shared__ Setup S;
  __shared__ uint32_t rgb_tile[kTile * 3 / 4];
  const int img = blockIdx.x / tiles, tile = blockIdx.x - img * tiles;
  const int tid = threadIdx.x;
  const float* st = states + size_t(img) * QS_STATE_DIM;
  const int finite = __syncthreads_and(tid < QS_STATE_DIM ? isfinite(st[tid]) : 1);
  if (tid < 5 && finite) {
    float pos[3] = {st[0], st[1], st[2]}, Rb[9];
    quat_to_R(st + 3, Rb);
    if (tid < 4) {   // leg tid: hip cylinder (rolled 90 deg about x in the URDF), thigh box, calf box, foot sphere
      const int k = tid;
      LegKin<float> K;
      leg_kin(k, st + 13 + 3 * k, M, K);
      float RH[9], RT[9], RC[9], R[9];
      link_rotations(K, RH, RT, RC);
      const float Rroll[9] = {RH[0], RH[2], -RH[1], RH[3], RH[5], -RH[4], RH[6], RH[8], -RH[7]};
      mat3_mul(Rb, Rroll, R);
      set_prim(S.prim[2 + 4 * k], R, pos, Rb, K.r1, M.hip_r, M.hip_hl, 0.f);
      float loc[3];
      m3_v(RT, M.thigh_c, loc);
      for (int a = 0; a < 3; a++) loc[a] += K.r2[a];
      mat3_mul(Rb, RT, R);
      set_prim(S.prim[3 + 4 * k], R, pos, Rb, loc, M.thigh_half[0], M.thigh_half[1], M.thigh_half[2]);
      m3_v(RC, M.calf_c, loc);
      for (int a = 0; a < 3; a++) loc[a] += K.r3[a];
      mat3_mul(Rb, RC, R);
      set_prim(S.prim[4 + 4 * k], R, pos, Rb, loc, M.calf_half[0], M.calf_half[1], M.calf_half[2]);
      set_prim(S.prim[5 + 4 * k], Rb, pos, Rb, K.r4, M.foot_radius, 0.f, 0.f);
    } else {
      const float zero[3] = {0.f, 0.f, 0.f};
      set_prim(S.prim[0], Rb, pos, Rb, zero, M.trunk_half[0], M.trunk_half[1], M.trunk_half[2]);
      set_prim(S.prim[1], Rb, pos, Rb, M.imu_pos, M.imu_half, M.imu_half, M.imu_half);
    }
  } else if (tid == 32) {   // camera: inverse(P V) in fp64, near / far of the projection
    const float* cam = cams + size_t(img) * QS_CAM_DIM;
    double V[16], P[16], PV[16];   // row-major from pybullet's column-major lists
    for (int r = 0; r < 4; r++)
      for (int c = 0; c < 4; c++) { V[4 * r + c] = cam[4 * c + r]; P[4 * r + c] = cam[16 + 4 * c + r]; }
    for (int r = 0; r < 4; r++)
      for (int c = 0; c < 4; c++)
        PV[4 * r + c] = P[4 * r] * V[c] + P[4 * r + 1] * V[4 + c] + P[4 * r + 2] * V[8 + c] + P[4 * r + 3] * V[12 + c];
    inverse4(PV, S.Minv);   // OpenGL perspective: P[2][3] / (P[2][2] + 1) is the far plane
    for (int c = 0; c < 4; c++) S.V2[c] = V[8 + c];
    S.far_ = float(P[11] / (P[10] + 1.0));
  }
  __syncthreads();
  if (tid == 0) {
    S.robot = finite;
    if (finite) {   // centred on the base, radius covering every primitive, inflated: only a cull
      float r = 0.f;
      for (int i = 0; i < kPrims; i++) {
        const Prim& p = S.prim[i];
        const float dc[3] = {p.c[0] - S.prim[0].c[0], p.c[1] - S.prim[0].c[1], p.c[2] - S.prim[0].c[2]};
        const int sh = prim_shape(i);
        const float ext = sh == SHAPE_SPHERE ? p.e[0]
                        : sh == SHAPE_CYL    ? sqrtf(p.e[0] * p.e[0] + p.e[1] * p.e[1])
                                             : sqrtf(p.e[0] * p.e[0] + p.e[1] * p.e[1] + p.e[2] * p.e[2]);
        r = fmaxf(r, sqrtf(dot3(dc, dc)) + ext);
      }
      for (int a = 0; a < 3; a++) S.bs[a] = S.prim[0].c[a];
      S.bs[3] = r * 1.01f + 1e-3f;
      const float qn = st[3] * st[3] + st[4] * st[4] + st[5] * st[5] + st[6] * st[6];
      S.robot = qn > 0.f && isfinite(qn) && isfinite(r);   // a zero or overflowing quaternion poses nothing
    }
  }
  __syncthreads();

  const int HW = W * H;
  const int pix = tile * kTile + tid;
  if (pix < HW) {
    const int row = pix / W, col = pix - row * W;
    // the ray through the pixel centre, from the near plane to the far plane (fp64 set-up)
    const double x = 2.0 * (col + 0.5) / W - 1.0, y = 1.0 - 2.0 * (row + 0.5) / H;
    double hn[4], hf[4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const double* m = S.Minv + 4 * r;
      const double b = m[0] * x + m[1] * y + m[3];
      hn[r] = b - m[2];
      hf[r] = b + m[2];
    }
    const double on[3] = {hn[0] / hn[3], hn[1] / hn[3], hn[2] / hn[3]};
    double dd[3] = {hf[0] / hf[3] - on[0], hf[1] / hf[3] - on[1], hf[2] / hf[3] - on[2]};
    const double il = 1.0 / sqrt(dd[0] * dd[0] + dd[1] * dd[1] + dd[2] * dd[2]);
    dd[0] *= il; dd[1] *= il; dd[2] *= il;
    const double z0 = -(S.V2[0] * on[0] + S.V2[1] * on[1] + S.V2[2] * on[2] + S.V2[3]);   // eye depth at t = 0
    const double g = -(S.V2[0] * dd[0] + S.V2[1] * dd[1] + S.V2[2] * dd[2]);             // ... per unit of t
    const float far_ = S.far_;
    const double tmax = (double(far_) - z0) / g;
    // ground: the plane z = 0, from either side
    double tbest = INFINITY;
    int hit = -2;   // -2 sky, -1 ground, i >= 0 primitive i
    {
      const double t = -on[2] / dd[2];
      if (t >= 0.0 && t <= tmax) { tbest = t; hit = -1; }
    }
    const float o[3] = {float(on[0]), float(on[1]), float(on[2])}, d[3] = {float(dd[0]), float(dd[1]), float(dd[2])};
    float n[3] = {0.f, 0.f, 1.f};
    if (S.robot && near_robot(S, o, d)) {
      float tb = hit == -1 ? float(tbest) : float(tmax);
      for (int i = 0; i < kPrims; i++) {
        float tn, tf, nl[3];
        intersect(i, S.prim[i], o, d, tn, tf, nl);
        if (tn <= tf && tn >= 0.f && tn < tb) {   // entry point in front of the near plane and before the best so far
          tb = tn; hit = i;
          m3_v(S.prim[i].R, nl, n);
        }
      }
      if (hit >= 0) tbest = tb;
    }
    const float dep = hit == -2 ? far_ : float(z0 + tbest * g);
    if (depth) depth[size_t(img) * HW + pix] = dep;
    if (seg) seg[size_t(img) * HW + pix] = hit == -2 ? -1 : (hit == -1 ? 0 : 1 + ((hit + 1) << 24));
    if (rgb) {
      float c[3];
      if (hit == -2) {
        c[0] = kStyle.sky[0]; c[1] = kStyle.sky[1]; c[2] = kStyle.sky[2];
      } else {
        float p[3];
        const float* alb;
        if (hit == -1) {
          const double gx = on[0] + tbest * dd[0], gy = on[1] + tbest * dd[1];
          p[0] = float(gx); p[1] = float(gy); p[2] = 0.f;
          alb = kStyle.ground[(static_cast<long long>(floor(gx)) + static_cast<long long>(floor(gy))) & 1];
        } else {
#pragma unroll
          for (int a = 0; a < 3; a++) p[a] = o[a] + float(tbest) * d[a];
          alb = kStyle.albedo[prim_kind(hit)];
        }
        const float* L = kStyle.light;
        const float ndl = fmaxf(0.f, dot3(n, L));
        float s = 0.f;
        if (ndl > 0.f) {
          s = 1.f;
          const float so[3] = {p[0] + kStyle.shadow_offset * n[0], p[1] + kStyle.shadow_offset * n[1],
                               p[2] + kStyle.shadow_offset * n[2]};
          if (S.robot && near_robot(S, so, L)) {
            for (int i = 0; i < kPrims; i++) {
              float tn, tf, nl[3];
              intersect(i, S.prim[i], so, L, tn, tf, nl);
              if (tn <= tf && tf >= 0.f) { s = 0.f; break; }
            }
          }
        }
        const float shade = kStyle.ambient + (1.f - kStyle.ambient) * ndl * s;
#pragma unroll
        for (int a = 0; a < 3; a++) c[a] = alb[a] * shade;
      }
      uint8_t* t8 = reinterpret_cast<uint8_t*>(rgb_tile);
#pragma unroll
      for (int a = 0; a < 3; a++) t8[3 * tid + a] = uint8_t(__float2int_rn(fminf(fmaxf(c[a], 0.f), 255.f)));
    }
  }
  if (rgb) {   // the tile's bytes go out as coalesced words (bytes when an image is not a whole number of words)
    __syncthreads();
    const int npix = min(kTile, HW - tile * kTile);
    const size_t base = (size_t(img) * HW + size_t(tile) * kTile) * 3;
    if ((HW & 3) == 0) {
      uint32_t* out = reinterpret_cast<uint32_t*>(rgb + base);
      for (int i = tid; i < npix * 3 / 4; i += kTile) out[i] = rgb_tile[i];
    } else {
      const uint8_t* t8 = reinterpret_cast<const uint8_t*>(rgb_tile);
      for (int i = tid; i < npix * 3; i += kTile) rgb[base + i] = t8[i];
    }
  }
}

}  // namespace

extern "C" int qs_render(const float* states, const float* cams, int k, int width, int height, uint8_t* rgb,
                         float* depth, int32_t* seg, void* stream) {
  if (k < 1) return abi_fail(QS_ERR_ARG, "qs_render: k must be at least 1");
  if (width < 1 || width > 4096 || height < 1 || height > 4096)
    return abi_fail(QS_ERR_ARG, "qs_render: width and height must lie in [1, 4096]");
  if (!rgb && !depth && !seg) return abi_fail(QS_ERR_ARG, "qs_render: no output requested (rgb, depth and seg are NULL)");
  if (!states || !cams) return abi_fail(QS_ERR_ARG, "qs_render: states or cams is NULL");
  const int tiles = (width * height + kTile - 1) / kTile;
  if (int64_t(k) * tiles > INT_MAX) return abi_fail(QS_ERR_ARG, "qs_render: too many pixels in one call");
  static const ModelConstT<float> M = [] {
    ModelConstT<float> m;
    host::build_model(m, 0.02);   // the breaking threshold only sets the *_thresh fields, which are not drawn
    return m;
  }();
  k_render<<<unsigned(int64_t(k) * tiles), kTile, 0, static_cast<cudaStream_t>(stream)>>>(M, states, cams, tiles, width,
                                                                                          height, rgb, depth, seg);
  abi_count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return abi_fail(QS_ERR_CUDA, std::string("qs_render: ") + cudaGetErrorString(e));
  return QS_OK;
}
