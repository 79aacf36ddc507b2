// qs_physics.cuh -- one physics tick for one env held in one thread's registers.
//
// Replaces pybullet.stepSimulation() (reference: quadruped_gym_env.py:218-219)
// for the Go1 URDF.  Same model and step semantics as the CPU oracle
// (oracle/qso_physics.c), different formulation, chosen for a one-env-per-thread
// GPU mapping:
//   * merged 13-body model (fixed links folded), everything expressed in the
//     BASE frame about the base origin, so composite inertias are plain sums;
//   * per leg: 3x3 joint-space inertia M_kk, coupling F_k (3x6), bias by
//     Newton-Euler; the base sees the Schur complement
//     S = M_bb - sum_k F_k^T M_kk^-1 F_k  (= its articulated-body inertia);
//   * contacts: PGS in a reduced space.  With S = L L^T, G_k = J_b - J_kk B_k,
//     Y_k = L^-1 G_k^T and H_k = J_kk M_kk^-1 J_kk^T the Delassus block is
//     A_kl = Y_k^T Y_l + delta_kl H_k, so a sweep needs one 6-vector z = sum Y lam
//     instead of Bullet's 18-vector; row order, clamps, cone projection, warm
//     start and early exit are Bullet's (see the oracle for the restatement).
#pragma once
#include "qs_robot.cuh"
#include "qs_packed.cuh"

namespace qs {

template <typename T> QS_DEV void cross3(const T* a, const T* b, T* o) {
  const T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}
template <typename T> QS_DEV void cross3_add(const T* a, const T* b, T* o) {   // accumulator first: two fused multiply-adds each
  const T x = o[0] + a[1] * b[2] - a[2] * b[1], y = o[1] + a[2] * b[0] - a[0] * b[2], z = o[2] + a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}
template <typename T> QS_DEV T dot3(const T* a, const T* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename T, typename U> QS_DEV void m3_v(const T* R, const U* v, T* o) {  // o = R v
  const T x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
  const T y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
  const T z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}
template <typename T> QS_DEV void m3t_v(const T* R, const T* v, T* o) {  // o = R^T v
  const T x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
  const T y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
  const T z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}
template <typename T> QS_DEV void sym3_mul(const T* I, const T* w, T* o) {
  o[0] = I[0] * w[0] + I[1] * w[1] + I[2] * w[2];
  o[1] = I[1] * w[0] + I[3] * w[1] + I[4] * w[2];
  o[2] = I[2] * w[0] + I[4] * w[1] + I[5] * w[2];
}

// rigid-body (or composite) spatial inertia about the base origin, base axes
template <typename T> struct SpI {
  T m, h[3], I[6];
};
// momentum of velocity (w, v):  L = I w + h x v,  p = m v - h x w
template <typename T> QS_DEV void spi_apply(const SpI<T>& A, const T* w, const T* v, T* L, T* p) {
  sym3_mul(A.I, w, L);
  cross3_add(A.h, v, L);
  T t[3];
  cross3(A.h, w, t);
  p[0] = A.m * v[0] - t[0]; p[1] = A.m * v[1] - t[1]; p[2] = A.m * v[2] - t[2];
}
// the same for the joint axes' motion vectors: w = (1,0,0) (hip) and w = (0, c, s) (thigh, calf)
template <typename T> QS_DEV void spi_apply_x(const SpI<T>& A, const T* v, T* L, T* p) {
  L[0] = A.I[0]; L[1] = A.I[1]; L[2] = A.I[2];
  cross3_add(A.h, v, L);
  p[0] = A.m * v[0]; p[1] = A.m * v[1] - A.h[2]; p[2] = A.m * v[2] + A.h[1];          // h x w = (0, h2, -h1)
}
template <typename T> QS_DEV void spi_apply_yz(const SpI<T>& A, T c, T s, const T* v, T* L, T* p) {
  L[0] = A.I[1] * c + A.I[2] * s; L[1] = A.I[3] * c + A.I[4] * s; L[2] = A.I[4] * c + A.I[5] * s;
  cross3_add(A.h, v, L);
  p[0] = A.m * v[0] - (A.h[1] * s - A.h[2] * c);                                       // h x w = (h1 s - h2 c, -h0 s, h0 c)
  p[1] = A.m * v[1] + A.h[0] * s;
  p[2] = A.m * v[2] - A.h[0] * c;
}
template <typename T> QS_DEV void spi_add(SpI<T>& a, const SpI<T>& b) {
  a.m += b.m;
#pragma unroll
  for (int i = 0; i < 3; i++) a.h[i] += b.h[i];
#pragma unroll
  for (int i = 0; i < 6; i++) a.I[i] += b.I[i];
}
// the robot's composite inertia takes a leg's, or both legs' of a pair
template <typename A, typename T> QS_DEV void spi_acc(SpI<A>& a, const SpI<T>& b) {
  acc_add(a.m, b.m);
#pragma unroll
  for (int i = 0; i < 3; i++) acc_add(a.h[i], b.h[i]);
#pragma unroll
  for (int i = 0; i < 6; i++) acc_add(a.I[i], b.I[i]);
}
// inertia of a body given in its link frame (mass, com, Ic about com) placed at
// rotation R (link->base) and origin r (base coords)
template <typename T>
QS_DEV void body_spi(T m, const T* com, const T* Ic, const T* R, const T* r, SpI<T>& o) {
  T c[3];
  m3_v(R, com, c);
  c[0] += r[0]; c[1] += r[1]; c[2] += r[2];
  T t[9];  // t = R * Ic
#pragma unroll
  for (int i = 0; i < 3; i++) {
    t[3 * i + 0] = R[3 * i] * Ic[0] + R[3 * i + 1] * Ic[1] + R[3 * i + 2] * Ic[2];
    t[3 * i + 1] = R[3 * i] * Ic[1] + R[3 * i + 1] * Ic[3] + R[3 * i + 2] * Ic[4];
    t[3 * i + 2] = R[3 * i] * Ic[2] + R[3 * i + 1] * Ic[4] + R[3 * i + 2] * Ic[5];
  }
  const T cc = dot3(c, c);
  o.I[0] = t[0] * R[0] + t[1] * R[1] + t[2] * R[2] + m * (cc - c[0] * c[0]);
  o.I[1] = t[0] * R[3] + t[1] * R[4] + t[2] * R[5] - m * c[0] * c[1];
  o.I[2] = t[0] * R[6] + t[1] * R[7] + t[2] * R[8] - m * c[0] * c[2];
  o.I[3] = t[3] * R[3] + t[4] * R[4] + t[5] * R[5] + m * (cc - c[1] * c[1]);
  o.I[4] = t[3] * R[6] + t[4] * R[7] + t[5] * R[8] - m * c[1] * c[2];
  o.I[5] = t[6] * R[6] + t[7] * R[7] + t[8] * R[8] + m * (cc - c[2] * c[2]);
  o.m = m;
  o.h[0] = m * c[0]; o.h[1] = m * c[1]; o.h[2] = m * c[2];
}

// The same for a link whose inertia about its com is DIAGONAL in the link frame (hip and thigh: single URDF links with
// bounding-box inertias, qs_model_host.h; the calf + foot body is not): I = sum_k d_k r_k r_k^T over the columns r_k of R,
// 27 multiply-adds instead of 45 -- and none of them multiplies one of the three structural zeros of Ic, which IEEE
// rules forbid the compiler to drop.
template <typename T>
QS_DEV void body_spi_diag(T m, const T* com, const T* Ic, const T* R, const T* r, SpI<T>& o) {
  T c[3];
  m3_v(R, com, c);
  c[0] += r[0]; c[1] += r[1]; c[2] += r[2];
  const T d0 = Ic[0], d1 = Ic[3], d2 = Ic[5];
  const T t0 = R[0] * d0, t1 = R[1] * d1, t2 = R[2] * d2;   // row 0 of R D
  const T t3 = R[3] * d0, t4 = R[4] * d1, t5 = R[5] * d2;   // row 1
  const T t6 = R[6] * d0, t7 = R[7] * d1, t8 = R[8] * d2;   // row 2
  const T cc = dot3(c, c);
  o.I[0] = t0 * R[0] + t1 * R[1] + t2 * R[2] + m * (cc - c[0] * c[0]);
  o.I[1] = t0 * R[3] + t1 * R[4] + t2 * R[5] - m * c[0] * c[1];
  o.I[2] = t0 * R[6] + t1 * R[7] + t2 * R[8] - m * c[0] * c[2];
  o.I[3] = t3 * R[3] + t4 * R[4] + t5 * R[5] + m * (cc - c[1] * c[1]);
  o.I[4] = t3 * R[6] + t4 * R[7] + t5 * R[8] - m * c[1] * c[2];
  o.I[5] = t6 * R[6] + t7 * R[7] + t8 * R[8] + m * (cc - c[2] * c[2]);
  o.m = m;
  o.h[0] = m * c[0]; o.h[1] = m * c[1]; o.h[2] = m * c[2];
}
// ... and for the hip link, whose rotation is about x by the hip angle (R = [1 0 0; 0 c -s; 0 s c])
template <typename T>
QS_DEV void body_spi_hip(T m, const T* com, const T* Ic, T c1, T s1, const T* r, SpI<T>& o) {
  const T c[3] = {com[0] + r[0], c1 * com[1] - s1 * com[2] + r[1], s1 * com[1] + c1 * com[2] + r[2]};
  const T d0 = Ic[0], d1 = Ic[3], d2 = Ic[5];
  const T cc = dot3(c, c);
  o.I[0] = d0 + m * (cc - c[0] * c[0]);
  o.I[1] = -m * c[0] * c[1];
  o.I[2] = -m * c[0] * c[2];
  o.I[3] = c1 * c1 * d1 + s1 * s1 * d2 + m * (cc - c[1] * c[1]);
  o.I[4] = c1 * s1 * (d1 - d2) - m * c[1] * c[2];
  o.I[5] = s1 * s1 * d1 + c1 * c1 * d2 + m * (cc - c[2] * c[2]);
  o.m = m;
  o.h[0] = m * c[0]; o.h[1] = m * c[1]; o.h[2] = m * c[2];
}

// upper-triangular index of a symmetric 6x6 stored in 21 entries
__host__ __device__ constexpr int s6(int i, int j) { return i <= j ? i * (11 - i) / 2 + j : j * (11 - j) / 2 + i; }

// a value parked in memory comes back: a volatile read for the machine types (the compiler must not keep the register
// alive instead), a plain one for the instrumented scalar of tools/count_flops.cu
template <typename T> QS_DEV T reload(const T& x) {
  if constexpr (std::is_arithmetic<T>::value) return *static_cast<const volatile T*>(&x);
  else return x;
}

template <typename T> struct EnvState {
  T pos[3], quat[4], vlin[3], vang[3], q[12], qd[12];
};
template <typename T> struct ContactState {
  T lam_n[4];   // normal impulse of the last tick per foot (N s); force = lam/dt
  int mask;     // bits 0-3: foot manifold point exists (quadruped.py:250-257)
  int invalid;  // number of non-foot shapes touching the ground (quadruped.py:243-249)
  int work_contacts;   // sum over ticks of active foot contacts        } algorithmic-work counters
  int work_row_iters;  // sum over ticks of contacts x PGS sweeps run   } (bench.py roofline)
};

// Per-env mass properties (EnvRandomizerMasses, env_randomizers/env_randomizer.py:19-84): column `idx` of a
// [EM_ROWS][stride] float array holding what differs from the nominal model M -- the three leg-link masses
// (the same for the four legs, :62-71), the calf+foot body re-merged for that calf mass, and body 0 (base + trunk +
// imu + payload block, :73-84 and :56-60) about the base origin.  base == nullptr: the nominal model.  The pointer
// and the stride are uniform (kernel parameters); only `idx` is per thread.
struct EnvModelRef {
  const float* base;
  int stride, idx;
};
enum { EM_HIP_M = 0, EM_THIGH_M = 1, EM_CALF_M = 2, EM_CALF_COM = 3, EM_CALF_IC = 6, EM_TRUNK_M = 12, EM_TRUNK_H = 13,
       EM_TRUNK_I = 16, EM_ROWS = 22 };
template <typename T> QS_DEV T em_get(const EnvModelRef& em, int row) { return T(em.base[size_t(row) * em.stride + em.idx]); }

template <typename T> struct LegKin {
  T s1, c1, s2, c2, s23, c23;
  T a2[3];                     // thigh/calf joint axis (base coords); hip axis is x
  T r1[3], r2[3], r3[3], r4[3];  // joint origins and foot centre (base coords)
};

template <typename T, typename ML> QS_DEV void leg_kin(int k, const T* q, const ML& M, LegKin<T>& K) {
  T s3, c3;
  sincos_tick(q[0], &K.s1, &K.c1);
  sincos_tick(q[1], &K.s2, &K.c2);
  sincos_tick(q[2], &s3, &c3);
  K.c23 = K.c2 * c3 - K.s2 * s3;
  K.s23 = K.s2 * c3 + K.c2 * s3;
  K.a2[0] = T(0); K.a2[1] = K.c1; K.a2[2] = K.s1;
  const T l = M.link_len, dy = M.thigh_off_y[k];
#pragma unroll
  for (int i = 0; i < 3; i++) K.r1[i] = M.hip_pos[k][i];
  K.r2[0] = K.r1[0]; K.r2[1] = K.r1[1] + dy * K.c1; K.r2[2] = K.r1[2] + dy * K.s1;
  K.r3[0] = K.r2[0] - l * K.s2; K.r3[1] = K.r2[1] + l * K.s1 * K.c2; K.r3[2] = K.r2[2] - l * K.c1 * K.c2;
  K.r4[0] = K.r3[0] - l * K.s23; K.r4[1] = K.r3[1] + l * K.s1 * K.c23; K.r4[2] = K.r3[2] - l * K.c1 * K.c23;
}

// contact Jacobian rows of foot k for direction d (base coords) at point pc:
// base part (pc x d, d), joint part a_j . ((pc - r_j) x d)
template <typename T>
QS_DEV void foot_jac_dir(const LegKin<T>& K, const T* pc, const T* d, T* Jb /*6*/, T* Jk /*3*/) {
  cross3(pc, d, Jb);
  Jb[3] = d[0]; Jb[4] = d[1]; Jb[5] = d[2];
  T u[3], t[3];
  u[0] = pc[0] - K.r1[0]; u[1] = pc[1] - K.r1[1]; u[2] = pc[2] - K.r1[2];
  cross3(u, d, t);
  Jk[0] = t[0];  // hip axis = x
  u[0] = pc[0] - K.r2[0]; u[1] = pc[1] - K.r2[1]; u[2] = pc[2] - K.r2[2];
  cross3(u, d, t);
  Jk[1] = K.c1 * t[1] + K.s1 * t[2];   // a2 = (0, c1, s1)
  u[0] = pc[0] - K.r3[0]; u[1] = pc[1] - K.r3[1]; u[2] = pc[2] - K.r3[2];
  cross3(u, d, t);
  Jk[2] = K.c1 * t[1] + K.s1 * t[2];
}

// f += I A + V x* (I V) for one body; V = (Vw, Vv), A = (Aw, Av)
template <typename T>
QS_DEV void body_force(const SpI<T>& I, const T* Vw, const T* Vv, const T* Aw, const T* Av, T* fn, T* fl) {
  T L[3], p[3], La[3], pa[3];
  spi_apply(I, Vw, Vv, L, p);
  spi_apply(I, Aw, Av, La, pa);
  // crf(V)(L,p) = (w x L + v x p, w x p)
  cross3_add(Vw, L, La);
  cross3_add(Vv, p, La);
  cross3_add(Vw, p, pa);
#pragma unroll
  for (int i = 0; i < 3; i++) { fn[i] += La[i]; fl[i] += pa[i]; }
}

template <typename T> QS_DEV T clamp_vel(T v, T mx) { return fmin_t(fmax_t(v, T(-mx)), mx); }

// External push on the base (Bullet applyExternalForce(robot, -1, f, pos + R p, WORLD_FRAME)): force f in the world frame
// (N) at the point p, base frame, from the base origin (m).
template <typename T> struct ExtWrench { T f[3]; T p[3]; };
// The push as a spatial force in base coordinates about the base origin, (p x Rb^T f, Rb^T f), taken off the Newton-Euler
// bias force fb: it acts on the body, the bias enters the base's equation with the opposite sign.
template <typename T> QS_DEV void sub_ext_wrench(const T* Rb, const ExtWrench<T>& w, T* fb) {
  T Fb[3], Nb[3];
  m3t_v(Rb, w.f, Fb);
  cross3(w.p, Fb, Nb);
#pragma unroll
  for (int i = 0; i < 3; i++) { fb[i] -= Nb[i]; fb[3 + i] -= Fb[i]; }
}


// ------------------------------------------------------------------------------------------
// Shared pieces of a tick
// ------------------------------------------------------------------------------------------
template <typename T> struct TickCtx {
  T Rb[9], wb[3], vb[3], nb[3], A0[3], wxv[3];
  T tdir[3][3];  // contact frame in base coords: normal, t1 = -y_world, t2 = x_world (btPlaneSpace1 of (0,0,1))
};

template <typename T> QS_DEV void tick_ctx(const EnvState<T>& st, const SolverConst& SC, TickCtx<T>& X) {
  {  // quat_to_R (qs_robot.cuh) with the tick's reciprocal-multiply division
    const T x = st.quat[0], y = st.quat[1], z = st.quat[2], w = st.quat[3];
    const T s = div_t(T(2), T(x * x + y * y + z * z + w * w));
    X.Rb[0] = T(1) - s * (y * y + z * z); X.Rb[1] = s * (x * y - w * z); X.Rb[2] = s * (x * z + w * y);
    X.Rb[3] = s * (x * y + w * z); X.Rb[4] = T(1) - s * (x * x + z * z); X.Rb[5] = s * (y * z - w * x);
    X.Rb[6] = s * (x * z - w * y); X.Rb[7] = s * (y * z + w * x); X.Rb[8] = T(1) - s * (x * x + y * y);
  }
  m3t_v(X.Rb, st.vang, X.wb);
  m3t_v(X.Rb, st.vlin, X.vb);
  const T gacc = T(-SC.gravity_z);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    X.nb[i] = X.Rb[6 + i];          // world z in base coords
    X.A0[i] = gacc * X.Rb[6 + i];   // fictitious base acceleration = -gravity
    X.tdir[0][i] = X.Rb[6 + i];
    X.tdir[1][i] = -X.Rb[3 + i];
    X.tdir[2][i] = X.Rb[i];
  }
  cross3(X.wb, X.vb, X.wxv);
}

template <typename T> QS_DEV void link_rotations(const LegKin<T>& K, T* RH, T* RT, T* RC) {
  RH[0] = T(1); RH[1] = T(0); RH[2] = T(0); RH[3] = T(0); RH[4] = K.c1; RH[5] = -K.s1; RH[6] = T(0); RH[7] = K.s1; RH[8] = K.c1;
  RT[0] = K.c2; RT[1] = T(0); RT[2] = K.s2; RT[3] = K.s1 * K.s2; RT[4] = K.c1; RT[5] = -K.s1 * K.c2;
  RT[6] = -K.c1 * K.s2; RT[7] = K.s1; RT[8] = K.c1 * K.c2;
  RC[0] = K.c23; RC[1] = T(0); RC[2] = K.s23; RC[3] = K.s1 * K.s23; RC[4] = K.c1; RC[5] = -K.s1 * K.c23;
  RC[6] = -K.c1 * K.s23; RC[7] = K.s1; RC[8] = K.c1 * K.c23;
}

// body 0 (base + trunk + imu, plus the payload block when the masses are randomized) about the base origin
template <typename T, bool kEM> QS_DEV void trunk_spi(const ModelConstT<T>& M, const EnvModelRef& em, SpI<T>& tot) {
  if (kEM && em.base) {
    tot.m = em_get<T>(em, EM_TRUNK_M);
#pragma unroll
    for (int i = 0; i < 3; i++) tot.h[i] = em_get<T>(em, EM_TRUNK_H + i);
#pragma unroll
    for (int i = 0; i < 6; i++) tot.I[i] = em_get<T>(em, EM_TRUNK_I + i);
  } else {
    tot.m = M.trunk_m;
#pragma unroll
    for (int i = 0; i < 3; i++) tot.h[i] = M.trunk_h[i];
#pragma unroll
    for (int i = 0; i < 6; i++) tot.I[i] = M.trunk_I[i];
  }
}

// Per-leg dynamics: joint-space inertia inverse Mi (sym 3x3: 00 01 02 11 12 22),
// Bm = M_kk^-1 F_k (3x6), ev = M_kk^-1 (tau - h) + B_lin (w x v); accumulates the
// Schur complement S6 -= F^T B, the base force fb += f_leg + F^T d and the
// composite inertia tot += I_leg.
//
// The three bodies are visited ROOT TO TIP and each is finished before the next starts: its inertia, velocity and bias
// acceleration are built, its bias wrench is projected on the joints at or above it (h_j = S_j . sum_{i >= j} f_i) and
// its momentum columns I_i S_j are added to F_j (= I^c_j S_j by linearity).  Against the textbook order (velocities
// down, forces and composite inertias up) this costs three more projections and three more I S products, ~5 % of
// the function, and keeps ONE body's inertia and ONE pair of velocity / acceleration vectors alive instead of three:
// what lets the pair instantiation (two legs per thread, twice the registers per value) fit the register file.
//
// T = a scalar and k = a leg, or T = a pair of scalars and k = a pair of legs (M = ModelLegPairsT); the sums over the
// legs (S6, fb, tot) are scalars of type A either way.
template <typename T> QS_DEV void body_force_set(const SpI<T>& I, const T* Vw, const T* Vv, const T* Aw, const T* Av, T* fn, T* fl) {
  T L[3], p[3];
  spi_apply(I, Vw, Vv, L, p);
  spi_apply(I, Aw, Av, fn, fl);
  // crf(V)(L,p) = (w x L + v x p, w x p)
  cross3_add(Vw, L, fn);
  cross3_add(Vv, p, fn);
  cross3_add(Vw, p, fl);
}
template <typename T, bool kEM, typename ML, typename A>
QS_DEV void leg_dynamics(int k, const T* q, const T* qd, const T* tau3, const TickCtx<T>& X, const ML& M,
                         const LegKin<T>& K, T* Mi, T* Bm, T* ev, A* S6, A* fb, SpI<A>& tot, const EnvModelRef& em) {
  const T* wb = X.wb;
  const T* vb = X.vb;
  const bool rand_m = kEM && em.base;  // randomized masses: changeDynamics(mass=) keeps each link's inertia diagonal and inertial frame
  const T c1 = K.c1, s1 = K.s1;
  (void)q;
  // motion subspaces S_j = (a_j, r_j x a_j).  The axes have structural zeros -- hip a1 = (1,0,0), thigh / calf
  // a2 = (0, c1, s1) -- and a product with a zero is an instruction the compiler has to keep (0 * x is not 0 for every x
  // under IEEE rules): the products below are written out for those axes.
  const T S1v1 = K.r1[2], S1v2 = -K.r1[1];                                               // r1 x a1 = (0, r1z, -r1y)
  const T S2v[3] = {K.r2[1] * s1 - K.r2[2] * c1, -K.r2[0] * s1, K.r2[0] * c1};           // r2 x a2
  const T S3v[3] = {K.r3[1] * s1 - K.r3[2] * c1, -K.r3[0] * s1, K.r3[0] * c1};           // r3 x a2
  const T S1v[3] = {T(0), S1v1, S1v2};
  // x-axis and (0, p, q) cross products: u x (w0,0,0) = (0, u2 w0, -u1 w0);  u x (0,p,q) = (u1 q - u2 p, -u0 q, u0 p)
  T F1[6], F2[6], F3[6], fn[3], fl[3], bn[3], bl[3], g[6];
  T Vw[3], Vv[3], Aw[3], Av[3];
  SpI<T> I;
  T h1, h2, h3;

  // ---- hip link
  {
    const T m1w0 = qd[0];                                         // m1w = (qd0, 0, 0)
    const T m1v1 = S1v1 * m1w0, m1v2 = S1v2 * m1w0;               // m1v = (0, .., ..)
    Aw[0] = T(0); Aw[1] = wb[2] * m1w0; Aw[2] = -wb[1] * m1w0;                           // wb x m1w
    Av[0] = wb[1] * m1v2 - wb[2] * m1v1 + X.A0[0];                                       // wb x m1v + vb x m1w + A0
    Av[1] = -wb[0] * m1v2 + vb[2] * m1w0 + X.A0[1];
    Av[2] = wb[0] * m1v1 - vb[1] * m1w0 + X.A0[2];
    Vw[0] = wb[0] + m1w0; Vw[1] = wb[1]; Vw[2] = wb[2];
    Vv[0] = vb[0]; Vv[1] = vb[1] + m1v1; Vv[2] = vb[2] + m1v2;
    body_spi_hip(rand_m ? em_get<T>(em, EM_HIP_M) : T(M.body_m[k][0]), M.body_com[k][0], M.body_Ic[k][0], c1, s1, K.r1, I);
    body_force_set(I, Vw, Vv, Aw, Av, fn, fl);
    h1 = fn[0] + S1v1 * fl[1] + S1v2 * fl[2];
    spi_apply_x(I, S1v, F1, F1 + 3);
    spi_acc(tot, I);
  }
  // ---- thigh
  {
    const T w1 = c1 * qd[1], w2 = s1 * qd[1];                     // m2w = (0, w1, w2)
    const T m2v[3] = {S2v[0] * qd[1], S2v[1] * qd[1], S2v[2] * qd[1]};
    Aw[0] = Aw[0] + Vw[1] * w2 - Vw[2] * w1;                                             // + V1w x m2w
    Aw[1] = Aw[1] - Vw[0] * w2;
    Aw[2] = Aw[2] + Vw[0] * w1;
    cross3_add(Vw, m2v, Av);                                                             // + V1w x m2v
    Av[0] = Av[0] + Vv[1] * w2 - Vv[2] * w1;                                             // + V1v x m2w
    Av[1] = Av[1] - Vv[0] * w2;
    Av[2] = Av[2] + Vv[0] * w1;
    Vw[1] = Vw[1] + w1; Vw[2] = Vw[2] + w2;
#pragma unroll
    for (int i = 0; i < 3; i++) Vv[i] = Vv[i] + m2v[i];
    // thigh link rotation: Rx(q1) Ry(q2)
    const T RT[9] = {K.c2, T(0), K.s2, s1 * K.s2, c1, -s1 * K.c2, -c1 * K.s2, s1, c1 * K.c2};
    body_spi_diag(rand_m ? em_get<T>(em, EM_THIGH_M) : T(M.body_m[k][1]), M.body_com[k][1], M.body_Ic[k][1], RT, K.r2, I);
    body_force_set(I, Vw, Vv, Aw, Av, bn, bl);
    h1 = h1 + bn[0] + S1v1 * bl[1] + S1v2 * bl[2];
    h2 = c1 * bn[1] + s1 * bn[2] + dot3(S2v, bl);
#pragma unroll
    for (int i = 0; i < 3; i++) { fn[i] = fn[i] + bn[i]; fl[i] = fl[i] + bl[i]; }
    spi_apply_x(I, S1v, g, g + 3);
#pragma unroll
    for (int i = 0; i < 6; i++) F1[i] = F1[i] + g[i];
    spi_apply_yz(I, c1, s1, S2v, F2, F2 + 3);
    spi_acc(tot, I);
  }
  // ---- calf + foot
  {
    const T w1 = c1 * qd[2], w2 = s1 * qd[2];                     // m3w = (0, w1, w2)
    const T m3v[3] = {S3v[0] * qd[2], S3v[1] * qd[2], S3v[2] * qd[2]};
    Aw[0] = Aw[0] + Vw[1] * w2 - Vw[2] * w1;                                             // + V2w x m3w
    Aw[1] = Aw[1] - Vw[0] * w2;
    Aw[2] = Aw[2] + Vw[0] * w1;
    cross3_add(Vw, m3v, Av);                                                             // + V2w x m3v
    Av[0] = Av[0] + Vv[1] * w2 - Vv[2] * w1;                                             // + V2v x m3w
    Av[1] = Av[1] - Vv[0] * w2;
    Av[2] = Av[2] + Vv[0] * w1;
    Vw[1] = Vw[1] + w1; Vw[2] = Vw[2] + w2;
#pragma unroll
    for (int i = 0; i < 3; i++) Vv[i] = Vv[i] + m3v[i];
    const T RC[9] = {K.c23, T(0), K.s23, s1 * K.s23, c1, -s1 * K.c23, -c1 * K.s23, s1, c1 * K.c23};
    if (rand_m) {
      T cc[3], ci[6];
#pragma unroll
      for (int i = 0; i < 3; i++) cc[i] = em_get<T>(em, EM_CALF_COM + i);
#pragma unroll
      for (int i = 0; i < 6; i++) ci[i] = em_get<T>(em, EM_CALF_IC + i);
      body_spi(em_get<T>(em, EM_CALF_M), cc, ci, RC, K.r3, I);
    } else {
      body_spi(T(M.body_m[k][2]), M.body_com[k][2], M.body_Ic[k][2], RC, K.r3, I);
    }
    body_force_set(I, Vw, Vv, Aw, Av, bn, bl);
    h1 = h1 + bn[0] + S1v1 * bl[1] + S1v2 * bl[2];
    const T a2bn = c1 * bn[1] + s1 * bn[2];
    h2 = h2 + a2bn + dot3(S2v, bl);
    h3 = a2bn + dot3(S3v, bl);
#pragma unroll
    for (int i = 0; i < 3; i++) { fn[i] = fn[i] + bn[i]; fl[i] = fl[i] + bl[i]; }
    spi_apply_x(I, S1v, g, g + 3);
#pragma unroll
    for (int i = 0; i < 6; i++) F1[i] = F1[i] + g[i];
    spi_apply_yz(I, c1, s1, S2v, g, g + 3);
#pragma unroll
    for (int i = 0; i < 6; i++) F2[i] = F2[i] + g[i];
    spi_apply_yz(I, c1, s1, S3v, F3, F3 + 3);
    spi_acc(tot, I);
  }

  // ---- joint-space inertia M_ij = S_i . F_j
  const T a2F3 = c1 * F3[1] + s1 * F3[2];
  const T M33 = a2F3 + dot3(S3v, F3 + 3);
  const T M23 = a2F3 + dot3(S2v, F3 + 3);
  const T M13 = F3[0] + S1v1 * F3[4] + S1v2 * F3[5];
  const T M22 = c1 * F2[1] + s1 * F2[2] + dot3(S2v, F2 + 3);
  const T M12 = F2[0] + S1v1 * F2[4] + S1v2 * F2[5];
  const T M11 = F1[0] + S1v1 * F1[4] + S1v2 * F1[5];
  // inverse of the symmetric 3x3 (adjugate)
  const T c00 = M22 * M33 - M23 * M23, c01 = M13 * M23 - M12 * M33, c02 = M12 * M23 - M13 * M22;
  const T c11 = M11 * M33 - M13 * M13, c12 = M12 * M13 - M11 * M23, c22 = M11 * M22 - M12 * M12;
  const T idet = div_t(T(1), T(M11 * c00 + M12 * c01 + M13 * c02));
  Mi[0] = c00 * idet; Mi[1] = c01 * idet; Mi[2] = c02 * idet; Mi[3] = c11 * idet; Mi[4] = c12 * idet; Mi[5] = c22 * idet;
  const T t1 = tau3[0] - h1, t2 = tau3[1] - h2, t3 = tau3[2] - h3;
  const T d0 = Mi[0] * t1 + Mi[1] * t2 + Mi[2] * t3;
  const T d1 = Mi[1] * t1 + Mi[3] * t2 + Mi[4] * t3;
  const T d2 = Mi[2] * t1 + Mi[4] * t2 + Mi[5] * t3;
#pragma unroll
  for (int c = 0; c < 6; c++) {
    Bm[c] = Mi[0] * F1[c] + Mi[1] * F2[c] + Mi[2] * F3[c];
    Bm[6 + c] = Mi[1] * F1[c] + Mi[3] * F2[c] + Mi[4] * F3[c];
    Bm[12 + c] = Mi[2] * F1[c] + Mi[4] * F2[c] + Mi[5] * F3[c];
  }
  ev[0] = d0 + Bm[3] * X.wxv[0] + Bm[4] * X.wxv[1] + Bm[5] * X.wxv[2];
  ev[1] = d1 + Bm[9] * X.wxv[0] + Bm[10] * X.wxv[1] + Bm[11] * X.wxv[2];
  ev[2] = d2 + Bm[15] * X.wxv[0] + Bm[16] * X.wxv[1] + Bm[17] * X.wxv[2];
#pragma unroll
  for (int a = 0; a < 6; a++) {
#pragma unroll
    for (int b = a; b < 6; b++) acc_add(S6[s6(a, b)], T(-(F1[a] * Bm[b] + F2[a] * Bm[6 + b] + F3[a] * Bm[12 + b])));
    acc_add(fb[a], T((a < 3 ? fn[a] : fl[a - 3]) + F1[a] * d0 + F2[a] * d1 + F3[a] * d2));
  }
}

// support-function gap of the leg's non-foot shapes (hip cylinder, thigh box, calf box)
// (pz = height of the base origin; MC = the scalar model: for a pair of legs its constants are broadcast)
template <typename T, typename S, typename MC>
QS_DEV void leg_shape_gaps(S pz, const TickCtx<T>& X, const MC& M, const LegKin<T>& K,
                           const T* RT, const T* RC, T* zh, T* zt, T* zc) {
  const T* nb = X.nb;
  const T nz = dot3(nb, K.a2);
  *zh = pz + dot3(nb, K.r1) - (abs_t(nz) * M.hip_hl + M.hip_r * sqrt_t(tmax(T(T(1) - nz * nz), T(0))));
  T c[3];
  m3_v(RT, M.thigh_c, c);
  *zt = pz + dot3(nb, K.r2) + dot3(nb, c) -
        (abs_t(nb[0] * RT[0] + nb[1] * RT[3] + nb[2] * RT[6]) * M.thigh_half[0] +
         abs_t(nb[0] * RT[1] + nb[1] * RT[4] + nb[2] * RT[7]) * M.thigh_half[1] +
         abs_t(nb[0] * RT[2] + nb[1] * RT[5] + nb[2] * RT[8]) * M.thigh_half[2]);
  m3_v(RC, M.calf_c, c);
  *zc = pz + dot3(nb, K.r3) + dot3(nb, c) -
        (abs_t(nb[0] * RC[0] + nb[1] * RC[3] + nb[2] * RC[6]) * M.calf_half[0] +
         abs_t(nb[0] * RC[1] + nb[1] * RC[4] + nb[2] * RC[7]) * M.calf_half[1] +
         abs_t(nb[0] * RC[2] + nb[1] * RC[5] + nb[2] * RC[8]) * M.calf_half[2]);
}
template <typename T>
QS_DEV void trunk_shape_gaps(const EnvState<T>& st, const TickCtx<T>& X, const ModelConstT<T>& M, T* zt, T* zi) {
  const T* nb = X.nb;
  *zt = st.pos[2] - (abs_t(nb[0]) * M.trunk_half[0] + abs_t(nb[1]) * M.trunk_half[1] + abs_t(nb[2]) * M.trunk_half[2]);
  *zi = st.pos[2] + dot3(nb, M.imu_pos) - (abs_t(nb[0]) + abs_t(nb[1]) + abs_t(nb[2])) * M.imu_half;
}

// base block: S6 += mat6(tot); in-place Cholesky (L(i,j), j<=i at s6(j,i)), Ld = 1/diag
template <typename T> QS_DEV void base_factor(const SpI<T>& tot, T* S6, T* Ld) {
  const T* I = tot.I;
  const T* h = tot.h;
  S6[s6(0, 0)] += I[0]; S6[s6(0, 1)] += I[1]; S6[s6(0, 2)] += I[2];
  S6[s6(1, 1)] += I[3]; S6[s6(1, 2)] += I[4]; S6[s6(2, 2)] += I[5];
  S6[s6(0, 4)] += -h[2]; S6[s6(0, 5)] += h[1];
  S6[s6(1, 3)] += h[2];  S6[s6(1, 5)] += -h[0];
  S6[s6(2, 3)] += -h[1]; S6[s6(2, 4)] += h[0];
  S6[s6(3, 3)] += tot.m; S6[s6(4, 4)] += tot.m; S6[s6(5, 5)] += tot.m;
#pragma unroll
  for (int j = 0; j < 6; j++) {
    T dj = S6[s6(j, j)];
#pragma unroll
    for (int k2 = 0; k2 < j; k2++) dj -= S6[s6(k2, j)] * S6[s6(k2, j)];
    const T inv = rsqrt_pos(dj);
    Ld[j] = inv;
    S6[s6(j, j)] = dj * inv;
#pragma unroll
    for (int i = j + 1; i < 6; i++) {
      T v = S6[s6(j, i)];
#pragma unroll
      for (int k2 = 0; k2 < j; k2++) v -= S6[s6(k2, i)] * S6[s6(k2, j)];
      S6[s6(j, i)] = v * inv;
    }
  }
}
template <typename S, typename T> QS_DEV void chol_fwd(const S* S6, const S* Ld, T* g) {  // g <- L^-1 g (g: scalars or pairs)
#pragma unroll
  for (int i = 0; i < 6; i++) {
    T v = g[i];
#pragma unroll
    for (int k2 = 0; k2 < i; k2++) v -= S6[s6(k2, i)] * g[k2];
    g[i] = v * Ld[i];
  }
}
template <typename T> QS_DEV void chol_bwd(const T* S6, const T* Ld, const T* y, T* x) {  // x = L^-T y
#pragma unroll
  for (int i = 5; i >= 0; i--) {
    T v = y[i];
#pragma unroll
    for (int k2 = i + 1; k2 < 6; k2++) v -= S6[s6(i, k2)] * x[k2];
    x[i] = v * Ld[i];
  }
}

// unconstrained update v += dt a with Bullet's per-coordinate clamp (applyDeltaVeeMultiDof);
// ab = classical base acceleration (spatial + w x v) in base coords
template <typename T>
QS_DEV bool base_velocity_update(EnvState<T>& st, const TickCtx<T>& X, const T* ab, T dt, T mcv, T* wb1, T* vb1) {
  bool clamped = false;
  T aw[3], av[3];
  m3_v(X.Rb, ab, aw);
  m3_v(X.Rb, ab + 3, av);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const T w1 = st.vang[i] + dt * aw[i], v1 = st.vlin[i] + dt * av[i];
    st.vang[i] = clamp_vel(w1, mcv);
    st.vlin[i] = clamp_vel(v1, mcv);
    clamped |= (st.vang[i] != w1) | (st.vlin[i] != v1);
  }
  m3t_v(X.Rb, st.vang, wb1);
  m3t_v(X.Rb, st.vlin, vb1);
  return clamped;
}

// positions from the new velocities (btMultiBody::stepPositionsMultiDof)
template <typename T> QS_DEV void integrate_positions(EnvState<T>& st, T dt) {
#pragma unroll
  for (int i = 0; i < 3; i++) st.pos[i] += dt * st.vlin[i];
  const T* om = st.vang;
  T ang = sqrt_pos(dot3(om, om));
  if (ang * dt > T(0.25 * QS_PI)) ang = div_t(T(0.25 * QS_PI), dt);
  // axis * sin(ang dt / 2) = om * (sin(x) / x) * dt / 2 with x = ang dt / 2 <= pi / 8: one branch-free form for every rate
  // (Bullet switches to a Taylor series below ang = 1e-3; the series used here is exact to rounding on the whole range)
  T sinc, cw;
  sinc_cos_small(T(T(0.5) * ang * dt), &sinc, &cw);
  const T sc = T(0.5) * dt * sinc;
  const T ax = om[0] * sc, ay = om[1] * sc, az = om[2] * sc;
  const T* q = st.quat;
  const T nw = cw * q[3] - ax * q[0] - ay * q[1] - az * q[2];
  const T nx = cw * q[0] + ax * q[3] + ay * q[2] - az * q[1];
  const T ny = cw * q[1] - ax * q[2] + ay * q[3] + az * q[0];
  const T nz = cw * q[2] + ax * q[1] - ay * q[0] + az * q[3];
  const T inv = rsqrt_pos(nx * nx + ny * ny + nz * nz + nw * nw);
  st.quat[0] = nx * inv; st.quat[1] = ny * inv; st.quat[2] = nz * inv; st.quat[3] = nw * inv;
#pragma unroll
  for (int i = 0; i < 12; i++) st.q[i] += dt * st.qd[i];
}

// ------------------------------------------------------------------------------------------
// FAST tick: foot contacts only (the overwhelmingly common case).
//
// Code-size discipline: the per-leg work is ONE rolled loop body (the instruction cache, not
// the FP32 pipe, bounded the fully unrolled version: ncu showed ~85% "no instruction" stalls),
// so per-leg results that later phases need go through a small per-thread scratch area
// (shared memory in the kernels, [slot][thread] layout => conflict-free); the PGS rows of the
// four feet live in registers because the sweep loop re-reads them up to 30 times.
//
// tau = joint torques of this tick (motor + spring).  cs: in = previous tick's contact
// impulses (warm start), out = this tick's.  Returns true WITHOUT touching the state when
// the tick needs the general solver (a joint at its limit, or a non-foot shape on the
// ground while SC.body_response is set); the caller then hands the env to physics_tick_general.
// ------------------------------------------------------------------------------------------
constexpr int QS_LEG_SCRATCH = 18 + 3 + 6 + 6 + 9 + 9;      // Bm, ev, Mi, sincos, W, (q, qd, tau)
constexpr int QS_PARK = 21;                                  // the caller's: motor command (12), spring k / b / rest (9)
constexpr int QS_TICK_SCRATCH = 4 * QS_LEG_SCRATCH + QS_PARK;  // floats per thread: 225 (2 blocks of 128 threads fill an SM's 228 KB)

// kStride > 0: the stride is a compile-time constant (the block size of the step / settle kernels), so every
// slot of a leg is an immediate offset from one per-leg base address; kStride = 0 reads it at run time.
// Layout: slot s of legs (2 kp, 2 kp + 1) of thread t are the two halves of ONE 64-bit word at
// [(kp * QS_LEG_SCRATCH + s) * 2 * stride + 2 t]: the pair passes read and write both legs with one LDS.64 / STS.64
// (consecutive threads -> consecutive words, conflict-free), a single leg's value is a 32-bit access at stride 2.
template <typename T, int kStride = 0> struct Scratch {
  T* p;        // the block's area
  int stride;  // threads of the block (ignored when kStride > 0)
  int tid = 0; // this thread
  QS_DEV int st() const { return kStride > 0 ? kStride : stride; }
  QS_DEV T& operator()(int leg, int slot) const {
    return p[((leg >> 1) * QS_LEG_SCRATCH + slot) * 2 * st() + 2 * tid + (leg & 1)];
  }
  QS_DEV PkT<T>& pair(int kp, int slot) const {
    return *reinterpret_cast<PkT<T>*>(p + (kp * QS_LEG_SCRATCH + slot) * 2 * st() + 2 * tid);
  }
  // what the tick loop's caller keeps here instead of in registers across the ticks (the tick itself never touches it)
  QS_DEV T& park(int i) const { return p[(4 * QS_LEG_SCRATCH + i) * st() + tid]; }
};
enum { SCR_BM = 0, SCR_EV = 18, SCR_MI = 21, SCR_SC = 27, SCR_W = 33, SCR_Q = 42, SCR_QD = 45, SCR_TAU = 48 };
// Once a foot's contact rows are built, EV / MI / SC / TAU of its leg are dead: the 18 floats of the rows'
// base part Y = L^-1 G^T live there during the PGS sweeps instead of in (spilling) registers.  (Not Q: the joint angles
// stay parked in the scratch for the whole tick and come back for the integration, so that they hold no registers
// in between.)
QS_DEV constexpr int scr_y(int i) { return i < 15 ? SCR_EV + i : SCR_TAU + (i - 15); }

template <typename T, typename ML> QS_DEV void leg_kin_from_sc(int k, const T* sc, const ML& M, LegKin<T>& K) {
  K.s1 = sc[0]; K.c1 = sc[1]; K.s2 = sc[2]; K.c2 = sc[3]; K.s23 = sc[4]; K.c23 = sc[5];
  K.a2[0] = T(0); K.a2[1] = K.c1; K.a2[2] = K.s1;
  const T l = M.link_len, dy = M.thigh_off_y[k];
#pragma unroll
  for (int i = 0; i < 3; i++) K.r1[i] = M.hip_pos[k][i];
  K.r2[0] = K.r1[0]; K.r2[1] = K.r1[1] + dy * K.c1; K.r2[2] = K.r1[2] + dy * K.s1;
  K.r3[0] = K.r2[0] - l * K.s2; K.r3[1] = K.r2[1] + l * K.s1 * K.c2; K.r3[2] = K.r2[2] - l * K.c1 * K.c2;
  K.r4[0] = K.r3[0] - l * K.s23; K.r4[1] = K.r3[1] + l * K.s1 * K.c23; K.r4[2] = K.r3[2] - l * K.c1 * K.c23;
}

// Returns TICK_DONE, or -- with the state untouched -- TICK_NEEDS_GENERAL (a joint at its limit, a body
// shape on the ground) or, for the kContacts = false variant (no foot-contact code at all: the flight
// kernel), TICK_NEEDS_CONTACT when a foot is within its contact threshold.
enum { TICK_DONE = 0, TICK_NEEDS_GENERAL = 1, TICK_NEEDS_CONTACT = 2 };
// kEM: read the per-env mass properties `em` (compiled out of the default kernels)
// M2 != nullptr (float / double only): the per-leg passes run on PAIRS of legs with packed arithmetic (qs_packed.cuh).
// kExt: `ext` != nullptr pushes the base in this tick (compiled out of the default kernels; a null `ext` runs the
// arithmetic of the default instantiation).
#ifndef QS_PACK_LEGS
#define QS_PACK_LEGS 1
#endif
template <typename T, bool kContacts = true, int kStride = 0, bool kEM = false, bool kExt = false>
__host__ __device__ int physics_tick(EnvState<T>& st, const T* tau, T mu, ContactState<T>& cs,
                                     const ModelConstT<T>& M, const SolverConst& SC, bool detect_invalid,
                                     const Scratch<T, kStride>& scr, const EnvModelRef em = EnvModelRef{nullptr, 0, 0},
                                     const ModelLegPairsT<T>* M2 = nullptr, const ExtWrench<T>* ext = nullptr) {
  constexpr bool kPack = QS_PACK_LEGS && std::is_floating_point<T>::value;
  const T dt = T(SC.dt);
  const T idt = div_t(T(1), dt);
  const T mcv = T(SC.max_coord_vel);
  TickCtx<T> X;
  tick_ctx(st, SC, X);
  const T* nb = X.nb;
  const T zero3[3] = {T(0), T(0), T(0)};

  // composite inertia of the whole robot and Newton-Euler base force, trunk first
  SpI<T> tot;
  trunk_spi<T, kEM>(M, em, tot);
  T fb[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  body_force(tot, X.wb, X.vb, zero3, X.A0, fb, fb + 3);
  if constexpr (kExt) {
    if (ext) sub_ext_wrench(X.Rb, *ext, fb);
  }
  T S6[21];
#pragma unroll
  for (int i = 0; i < 21; i++) S6[i] = T(0);

  int active = 0, invalid = 0;
  bool need_general = false;
  const bool watch_shapes = detect_invalid || SC.body_response;

  // joint state and torques go through the scratch so that the rolled loops can index them by leg
  if constexpr (kPack) {
#pragma unroll
    for (int kp = 0; kp < 2; kp++) {
#pragma unroll
      for (int j = 0; j < 3; j++) {
        scr.pair(kp, SCR_Q + j) = PkT<T>(st.q[6 * kp + j], st.q[6 * kp + 3 + j]);
        scr.pair(kp, SCR_QD + j) = PkT<T>(st.qd[6 * kp + j], st.qd[6 * kp + 3 + j]);
        scr.pair(kp, SCR_TAU + j) = PkT<T>(tau[6 * kp + j], tau[6 * kp + 3 + j]);
      }
    }
  } else {
#pragma unroll
  for (int k = 0; k < 4; k++) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
      scr(k, SCR_Q + j) = st.q[3 * k + j];
      scr(k, SCR_QD + j) = st.qd[3 * k + j];
      scr(k, SCR_TAU + j) = tau[3 * k + j];
    }
  }
  }

  // ---- pass A: one rolled loop over the legs, two at a time when packed
  if constexpr (kPack) {
    using P = PkT<T>;
    TickCtx<P> X2;   // the base's quantities are the same for both legs of a pair: broadcast operands
#pragma unroll
    for (int i = 0; i < 3; i++) {
      X2.wb[i] = P(X.wb[i]); X2.vb[i] = P(X.vb[i]); X2.nb[i] = P(X.nb[i]); X2.A0[i] = P(X.A0[i]); X2.wxv[i] = P(X.wxv[i]);
    }
#pragma unroll 1
    for (int kp = 0; kp < 2; kp++) {
      const int k0 = 2 * kp, k1 = k0 + 1;
      P q[3], qd[3], tk[3];
#pragma unroll
      for (int j = 0; j < 3; j++) {
        q[j] = scr.pair(kp, SCR_Q + j);
        qd[j] = scr.pair(kp, SCR_QD + j);
        tk[j] = scr.pair(kp, SCR_TAU + j);
      }
      LegKin<P> K;
      leg_kin(kp, q, *M2, K);
      // everything that only needs the kinematics comes first, so that it is dead while the dynamics run
      const P sc6[6] = {K.s1, K.c1, K.s2, K.c2, K.s23, K.c23};
#pragma unroll
      for (int i = 0; i < 6; i++) scr.pair(kp, SCR_SC + i) = sc6[i];
      if (SC.enable_limits) {
#pragma unroll
        for (int j = 0; j < 3; j++)
          need_general |= (q[j].x <= M.joint_lo[j]) | (q[j].x >= M.joint_hi[j]) | (q[j].y <= M.joint_lo[j]) | (q[j].y >= M.joint_hi[j]);
      }
      // collision detection on the poses at the start of the tick
      const P gap = st.pos[2] + dot3(X2.nb, K.r4) - M.foot_radius;
      if (gap.x < M.foot_thresh) active |= 1 << k0;
      if (gap.y < M.foot_thresh) active |= 1 << k1;
      if (watch_shapes) {
        P RH[9], RT[9], RC[9], zh, zt, zc;
        link_rotations(K, RH, RT, RC);
        leg_shape_gaps(st.pos[2], X2, M, K, RT, RC, &zh, &zt, &zc);
        invalid += (zh.x < M.hip_thresh) + (zt.x < M.thigh_thresh) + (zc.x < M.calf_thresh) +
                   (zh.y < M.hip_thresh) + (zt.y < M.thigh_thresh) + (zc.y < M.calf_thresh);
      }
      P Mi[6], Bm[18], ev[3];
      leg_dynamics<P, kEM>(kp, q, qd, tk, X2, *M2, K, Mi, Bm, ev, S6, fb, tot, em);
#pragma unroll
      for (int i = 0; i < 18; i++) scr.pair(kp, SCR_BM + i) = Bm[i];
#pragma unroll
      for (int i = 0; i < 3; i++) scr.pair(kp, SCR_EV + i) = ev[i];
#pragma unroll
      for (int i = 0; i < 6; i++) scr.pair(kp, SCR_MI + i) = Mi[i];
    }
  } else {
#pragma unroll 1
  for (int k = 0; k < 4; k++) {
    const T q[3] = {scr(k, SCR_Q), scr(k, SCR_Q + 1), scr(k, SCR_Q + 2)};
    const T qd[3] = {scr(k, SCR_QD), scr(k, SCR_QD + 1), scr(k, SCR_QD + 2)};
    const T tk[3] = {scr(k, SCR_TAU), scr(k, SCR_TAU + 1), scr(k, SCR_TAU + 2)};
    LegKin<T> K;
    leg_kin(k, q, M, K);
    T Mi[6], Bm[18], ev[3];
    leg_dynamics<T, kEM>(k, q, qd, tk, X, M, K, Mi, Bm, ev, S6, fb, tot, em);
#pragma unroll
    for (int i = 0; i < 18; i++) scr(k, SCR_BM + i) = Bm[i];
#pragma unroll
    for (int i = 0; i < 3; i++) scr(k, SCR_EV + i) = ev[i];
#pragma unroll
    for (int i = 0; i < 6; i++) scr(k, SCR_MI + i) = Mi[i];
    scr(k, SCR_SC + 0) = K.s1; scr(k, SCR_SC + 1) = K.c1; scr(k, SCR_SC + 2) = K.s2;
    scr(k, SCR_SC + 3) = K.c2; scr(k, SCR_SC + 4) = K.s23; scr(k, SCR_SC + 5) = K.c23;
    if (SC.enable_limits) {
#pragma unroll
      for (int j = 0; j < 3; j++) need_general |= (q[j] <= M.joint_lo[j]) | (q[j] >= M.joint_hi[j]);
    }
    // collision detection on the poses at the start of the tick
    const T gap = st.pos[2] + dot3(nb, K.r4) - M.foot_radius;
    if (gap < M.foot_thresh) active |= 1 << k;
    if (watch_shapes) {
      // non-foot shapes vs the plane: support-function distance below the link's
      // contact breaking threshold (quadruped.py:243-249 -> invalid contact)
      T RH[9], RT[9], RC[9], zh, zt, zc;
      link_rotations(K, RH, RT, RC);
      leg_shape_gaps(st.pos[2], X, M, K, RT, RC, &zh, &zt, &zc);
      invalid += (zh < M.hip_thresh) + (zt < M.thigh_thresh) + (zc < M.calf_thresh);
    }
  }
  }
  if (watch_shapes) {
    T zt, zi;
    trunk_shape_gaps(st, X, M, &zt, &zi);
    invalid += (zt < M.trunk_thresh) + (zi < M.imu_thresh);
    if (SC.body_response && invalid > 0) need_general = true;
  }
  if (need_general) return TICK_NEEDS_GENERAL;
  if (!kContacts && active) return TICK_NEEDS_CONTACT;

  // ---- base: S = M_bb - sum F^T B, Cholesky, solve
  T Ld[6];
  base_factor(tot, S6, Ld);
  T ab[6];
  {
    T y[6];
#pragma unroll
    for (int i = 0; i < 6; i++) y[i] = -fb[i];
    chol_fwd(S6, Ld, y);
    chol_bwd(S6, Ld, y, ab);
  }
  // classical acceleration of the base origin: spatial + w x v
  ab[3] += X.wxv[0]; ab[4] += X.wxv[1]; ab[5] += X.wxv[2];

  // ---- v += dt a, clamped like btMultiBody::applyDeltaVeeMultiDof
  T wb1[3], vb1[3];
  base_velocity_update(st, X, ab, dt, mcv, wb1, vb1);
  if constexpr (kPack) {
    using P = PkT<T>;
#pragma unroll 1
    for (int kp = 0; kp < 2; kp++) {
      const int k0 = 2 * kp, k1 = k0 + 1;
#pragma unroll
      for (int j = 0; j < 3; j++) {
        P acc = scr.pair(kp, SCR_EV + j);
#pragma unroll
        for (int c = 0; c < 6; c++) acc -= scr.pair(kp, SCR_BM + 6 * j + c) * P(ab[c]);
        scr.pair(kp, SCR_QD + j) = clamp_vel(P(scr.pair(kp, SCR_QD + j) + P(dt) * acc), P(mcv));
      }
    }
  } else {
#pragma unroll 1
  for (int k = 0; k < 4; k++) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
      T acc = scr(k, SCR_EV + j);
#pragma unroll
      for (int c = 0; c < 6; c++) acc -= scr(k, SCR_BM + 6 * j + c) * ab[c];
      scr(k, SCR_QD + j) = clamp_vel(scr(k, SCR_QD + j) + dt * acc, mcv);
    }
  }
  }

  bool in_contact = false;
  if constexpr (kContacts) in_contact = active != 0;
  if constexpr (kContacts) if (in_contact) {
    // ---- contact rows of the active feet (rolled loop), results routed into registers
    T H[4][6], rhs[4][3], dinv[4][3], diag[4][3], lam[4][3];
    T z[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
    // a foot without contact is an all-zero set of rows: the sweeps below then need no branch per foot (their
    // instructions are free to overlap across the feet), and zeros stay zeros through them
#pragma unroll
    for (int k = 0; k < 4; k++) {
#pragma unroll
      for (int i = 0; i < 3; i++) lam[k][i] = rhs[k][i] = dinv[k][i] = diag[k][i] = T(0);
#pragma unroll
      for (int i = 0; i < 6; i++) H[k][i] = T(0);
    }
    if constexpr (kPack) {
      // two feet at a time (qs_packed.cuh).  A pair with one foot down runs the arithmetic on both and keeps the rows of
      // that foot only (the idle leg's inputs are valid numbers: pass A fills them for every leg).
      using P = PkT<T>;
      P nbp[3], tdp[3][3], wb1p[3], vb1p[3];
#pragma unroll
      for (int i = 0; i < 3; i++) {
        nbp[i] = P(nb[i]); wb1p[i] = P(wb1[i]); vb1p[i] = P(vb1[i]);
        tdp[0][i] = P(X.tdir[0][i]); tdp[1][i] = P(X.tdir[1][i]); tdp[2][i] = P(X.tdir[2][i]);
      }
#pragma unroll 1
      for (int kp = 0; kp < 2; kp++) {
        const int k0 = 2 * kp, k1 = k0 + 1;
        const bool a0 = active & (1 << k0), a1 = active & (1 << k1);
        if (!a0 && !a1) {
#pragma unroll
          for (int i = 0; i < 18; i++) scr.pair(kp, scr_y(i)) = P(T(0));
          continue;
        }
        P sc[6], Mi[6], Bm[18];
#pragma unroll
        for (int i = 0; i < 6; i++) { sc[i] = scr.pair(kp, SCR_SC + i); Mi[i] = scr.pair(kp, SCR_MI + i); }
#pragma unroll
        for (int i = 0; i < 18; i++) Bm[i] = scr.pair(kp, SCR_BM + i);
        LegKin<P> K;
        leg_kin_from_sc(kp, sc, *M2, K);
        const P gap = st.pos[2] + dot3(nbp, K.r4) - M.foot_radius;
        const P pc[3] = {K.r4[0] - M.foot_radius * nbp[0], K.r4[1] - M.foot_radius * nbp[1], K.r4[2] - M.foot_radius * nbp[2]};
        const P qk[3] = {scr.pair(kp, SCR_QD), scr.pair(kp, SCR_QD + 1), scr.pair(kp, SCR_QD + 2)};
        P y[18], h[6], r3[3], di[3], dg[3], Jk[3][3], Wl[9];
#pragma unroll
        for (int dd = 0; dd < 3; dd++) {
          P Jb[6];
          foot_jac_dir(K, pc, tdp[dd], Jb, Jk[dd]);
          r3[dd] = Jb[0] * wb1p[0] + Jb[1] * wb1p[1] + Jb[2] * wb1p[2] + Jb[3] * vb1p[0] + Jb[4] * vb1p[1] + Jb[5] * vb1p[2] +
                   Jk[dd][0] * qk[0] + Jk[dd][1] * qk[1] + Jk[dd][2] * qk[2];
#pragma unroll
          for (int c = 0; c < 6; c++)
            y[6 * dd + c] = Jb[c] - (Jk[dd][0] * Bm[c] + Jk[dd][1] * Bm[6 + c] + Jk[dd][2] * Bm[12 + c]);
          Wl[0 * 3 + dd] = Mi[0] * Jk[dd][0] + Mi[1] * Jk[dd][1] + Mi[2] * Jk[dd][2];
          Wl[1 * 3 + dd] = Mi[1] * Jk[dd][0] + Mi[3] * Jk[dd][1] + Mi[4] * Jk[dd][2];
          Wl[2 * 3 + dd] = Mi[2] * Jk[dd][0] + Mi[4] * Jk[dd][1] + Mi[5] * Jk[dd][2];
        }
#define QS_H(a, b) (Jk[a][0] * Wl[0 * 3 + b] + Jk[a][1] * Wl[1 * 3 + b] + Jk[a][2] * Wl[2 * 3 + b])
        h[0] = QS_H(0, 0); h[1] = QS_H(0, 1); h[2] = QS_H(0, 2);
        h[3] = QS_H(1, 1); h[4] = QS_H(1, 2); h[5] = QS_H(2, 2);
#undef QS_H
#pragma unroll
        for (int i = 0; i < 9; i++) scr.pair(kp, SCR_W + i) = Wl[i];
        {
          const T slop = T(SC.linear_slop), erp = T(SC.contact_erp);
          const T d0 = gap.x + slop, d1 = gap.y + slop;
          T pe0 = T(0), ve0 = -r3[0].x, pe1 = T(0), ve1 = -r3[0].y;
          if (d0 > T(0)) ve0 -= d0 * idt; else pe0 = -d0 * erp * idt;
          if (d1 > T(0)) ve1 -= d1 * idt; else pe1 = -d1 * erp * idt;
          r3[0] = P(pe0 + ve0, pe1 + ve1);
          r3[1] = -r3[1];
          r3[2] = -r3[2];
        }
        const P hd[3] = {h[0], h[3], h[5]};
#pragma unroll
        for (int dd = 0; dd < 3; dd++) {
          chol_fwd(S6, Ld, y + 6 * dd);
          P nn = y[6 * dd] * y[6 * dd];
#pragma unroll
          for (int i = 1; i < 6; i++) nn += y[6 * dd + i] * y[6 * dd + i];
          dg[dd] = nn + hd[dd];
          di[dd] = div_t(P(T(1)), dg[dd]);
        }
        // warm start of the normal impulses (Bullet m_warmstartingFactor), foot k0 then foot k1 as in the scalar order
        T l00 = T(0), l01 = T(0);
        if (a0 && (cs.mask & (1 << k0))) {
          l00 = cs.lam_n[k0] * T(SC.warmstart);
#pragma unroll
          for (int i = 0; i < 6; i++) z[i] += y[i].x * l00;
        }
        if (a1 && (cs.mask & (1 << k1))) {
          l01 = cs.lam_n[k1] * T(SC.warmstart);
#pragma unroll
          for (int i = 0; i < 6; i++) z[i] += y[i].y * l01;
        }
#pragma unroll
        for (int i = 0; i < 18; i++) scr.pair(kp, scr_y(i)) = P(a0 ? y[i].x : T(0), a1 ? y[i].y : T(0));
#define QS_ROUTE2(KA, KB)                                                                                                \
  {                                                                                                                     \
    _Pragma("unroll") for (int i = 0; i < 6; i++) { H[KA][i] = a0 ? h[i].x : T(0); H[KB][i] = a1 ? h[i].y : T(0); }       \
    _Pragma("unroll") for (int i = 0; i < 3; i++) {                                                                       \
      rhs[KA][i] = a0 ? r3[i].x : T(0); dinv[KA][i] = a0 ? di[i].x : T(0); diag[KA][i] = a0 ? dg[i].x : T(0);             \
      rhs[KB][i] = a1 ? r3[i].y : T(0); dinv[KB][i] = a1 ? di[i].y : T(0); diag[KB][i] = a1 ? dg[i].y : T(0);             \
    }                                                                                                                   \
    lam[KA][0] = l00; lam[KB][0] = l01;                                                                                 \
  }
        if (kp == 0) QS_ROUTE2(0, 1) else QS_ROUTE2(2, 3)
#undef QS_ROUTE2
      }
    } else {
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
      if (!(active & (1 << k))) {
#pragma unroll
        for (int i = 0; i < 18; i++) scr(k, scr_y(i)) = T(0);   // (EV / MI / SC / TAU of an idle leg are dead by now)
        continue;
      }
      T sc[6], Mi[6], Bm[18];
#pragma unroll
      for (int i = 0; i < 6; i++) { sc[i] = scr(k, SCR_SC + i); Mi[i] = scr(k, SCR_MI + i); }
#pragma unroll
      for (int i = 0; i < 18; i++) Bm[i] = scr(k, SCR_BM + i);
      LegKin<T> K;
      leg_kin_from_sc(k, sc, M, K);
      const T gap = st.pos[2] + dot3(nb, K.r4) - M.foot_radius;
      const T pc[3] = {K.r4[0] - M.foot_radius * nb[0], K.r4[1] - M.foot_radius * nb[1],
                       K.r4[2] - M.foot_radius * nb[2]};
      const T qk[3] = {scr(k, SCR_QD), scr(k, SCR_QD + 1), scr(k, SCR_QD + 2)};
      T y[18], h[6], r3[3], di[3], dg[3], Jk[3][3], Wl[9];
#pragma unroll
      for (int dd = 0; dd < 3; dd++) {
        T Jb[6];
        foot_jac_dir(K, pc, X.tdir[dd], Jb, Jk[dd]);
        // J nu* evaluated directly on the updated velocities
        r3[dd] = Jb[0] * wb1[0] + Jb[1] * wb1[1] + Jb[2] * wb1[2] + Jb[3] * vb1[0] + Jb[4] * vb1[1] + Jb[5] * vb1[2] +
                 Jk[dd][0] * qk[0] + Jk[dd][1] * qk[1] + Jk[dd][2] * qk[2];
#pragma unroll
        for (int c = 0; c < 6; c++)
          y[6 * dd + c] = Jb[c] - (Jk[dd][0] * Bm[c] + Jk[dd][1] * Bm[6 + c] + Jk[dd][2] * Bm[12 + c]);
        Wl[0 * 3 + dd] = Mi[0] * Jk[dd][0] + Mi[1] * Jk[dd][1] + Mi[2] * Jk[dd][2];
        Wl[1 * 3 + dd] = Mi[1] * Jk[dd][0] + Mi[3] * Jk[dd][1] + Mi[4] * Jk[dd][2];
        Wl[2 * 3 + dd] = Mi[2] * Jk[dd][0] + Mi[4] * Jk[dd][1] + Mi[5] * Jk[dd][2];
      }
#define QS_H(a, b) (Jk[a][0] * Wl[0 * 3 + b] + Jk[a][1] * Wl[1 * 3 + b] + Jk[a][2] * Wl[2 * 3 + b])
      h[0] = QS_H(0, 0); h[1] = QS_H(0, 1); h[2] = QS_H(0, 2);
      h[3] = QS_H(1, 1); h[4] = QS_H(1, 2); h[5] = QS_H(2, 2);
#undef QS_H
#pragma unroll
      for (int i = 0; i < 9; i++) scr(k, SCR_W + i) = Wl[i];
      const T dist = gap + T(SC.linear_slop);
      T pos_err = T(0), vel_err = -r3[0];
      if (dist > T(0)) vel_err -= dist * idt; else pos_err = -dist * T(SC.contact_erp) * idt;
      r3[0] = pos_err + vel_err;
      r3[1] = -r3[1];
      r3[2] = -r3[2];
      const T hd[3] = {h[0], h[3], h[5]};
#pragma unroll
      for (int dd = 0; dd < 3; dd++) {
        chol_fwd(S6, Ld, y + 6 * dd);
        T nn = T(0);
#pragma unroll
        for (int i = 0; i < 6; i++) nn += y[6 * dd + i] * y[6 * dd + i];
        dg[dd] = nn + hd[dd];           // the row's diagonal of the Delassus matrix, and its inverse
        di[dd] = div_t(T(1), dg[dd]);
      }
      // warm start of the normal impulse (Bullet m_warmstartingFactor)
      T l0 = T(0);
      if (cs.mask & (1 << k)) {
        l0 = cs.lam_n[k] * T(SC.warmstart);
#pragma unroll
        for (int i = 0; i < 6; i++) z[i] += y[i] * l0;
      }
      // rows' base part to the leg's (now dead) scratch, the small per-foot blocks into the register
      // file (static indices only)
#pragma unroll
      for (int i = 0; i < 18; i++) scr(k, scr_y(i)) = y[i];
#define QS_ROUTE(KK)                                                                    \
  case KK: {                                                                            \
    _Pragma("unroll") for (int i = 0; i < 6; i++) H[KK][i] = h[i];                       \
    _Pragma("unroll") for (int i = 0; i < 3; i++) { rhs[KK][i] = r3[i]; dinv[KK][i] = di[i]; diag[KK][i] = dg[i]; } \
    lam[KK][0] = l0;                                                                    \
  } break;
      switch (k) { QS_ROUTE(0) QS_ROUTE(1) QS_ROUTE(2) default: QS_ROUTE(3) }
#undef QS_ROUTE
    }
    }

    // ---- projected Gauss-Seidel (rows: normals of all feet, then friction cones)
    //
    // The sweep is a chain: every row needs the z the row before it left.  Written naively that is, per row, a
    // nine-term dot product, the clamp and the update in sequence -- fourteen dependent instructions, and with two
    // warps per scheduler the chain, not the instruction count, is what a sweep costs (ncu: the dot product's FFMAs
    // carry the PGS's stall samples).  Same arithmetic, shorter chain:
    //  * normal rows: w_k = H_k lam_k + Yn_k . (z + sum_{l<k} Yn_l dI_l) = [H_k lam_k + Yn_k . z] + sum_{l<k} N_kl dI_l with
    //    the six couplings N_kl = Yn_k . Yn_l computed once per tick.  The brackets of the four feet are independent
    //    (computed side by side), and a row then hangs on its predecessor by ONE multiply-add;
    //  * friction rows: the dot product as two chains of three;
    //  * the residual uses the stored diagonal instead of a division.
    // Still Gauss-Seidel in Bullet's row order: each row sees every impulse change before it.
    const T thr = T(SC.residual_threshold);
    const int iters = SC.num_iterations;
    const int nact = (active & 1) + ((active >> 1) & 1) + ((active >> 2) & 1) + ((active >> 3) & 1);
    cs.work_contacts += nact;
    T N10, N20, N21, N30, N31, N32;
    {
      T Yn[4][6];
      if constexpr (kPack) {
#pragma unroll
        for (int kp = 0; kp < 2; kp++) {
#pragma unroll
          for (int i = 0; i < 6; i++) { const PkT<T> v = scr.pair(kp, scr_y(i)); Yn[2 * kp][i] = v.x; Yn[2 * kp + 1][i] = v.y; }
        }
      } else {
#pragma unroll
      for (int k = 0; k < 4; k++) {
#pragma unroll
        for (int i = 0; i < 6; i++) Yn[k][i] = scr(k, scr_y(i));
      }
      }
#define QS_N(a, b) ((Yn[a][0] * Yn[b][0] + Yn[a][1] * Yn[b][1] + Yn[a][2] * Yn[b][2]) + (Yn[a][3] * Yn[b][3] + Yn[a][4] * Yn[b][4] + Yn[a][5] * Yn[b][5]))
      N10 = QS_N(1, 0); N20 = QS_N(2, 0); N21 = QS_N(2, 1); N30 = QS_N(3, 0); N31 = QS_N(3, 1); N32 = QS_N(3, 2);
#undef QS_N
    }
    for (int it = 0; it < iters; it++) {
      T res = T(0);
      cs.work_row_iters += nact;
      PkT<T> yab[12];   // (pair builds) friction rows of the two feet of a pair
      {  // normal rows
        T Yn[4][6], bs[4], dIn[4];
        if constexpr (kPack) {
#pragma unroll
          for (int kp = 0; kp < 2; kp++) {
#pragma unroll
            for (int i = 0; i < 6; i++) { const PkT<T> v = scr.pair(kp, scr_y(i)); Yn[2 * kp][i] = v.x; Yn[2 * kp + 1][i] = v.y; }
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; k++) {
#pragma unroll
            for (int i = 0; i < 6; i++) Yn[k][i] = scr(k, scr_y(i));
          }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          bs[k] = rhs[k][0] - ((H[k][0] * lam[k][0] + H[k][1] * lam[k][1] + H[k][2] * lam[k][2] + Yn[k][0] * z[0] + Yn[k][1] * z[1] + Yn[k][2] * z[2]) +
                               (Yn[k][3] * z[3] + Yn[k][4] * z[4] + Yn[k][5] * z[5]));
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          T r = bs[k];
          if (k == 1) r = r - N10 * dIn[0];
          if (k == 2) r = r - N20 * dIn[0] - N21 * dIn[1];
          if (k == 3) r = r - N30 * dIn[0] - N31 * dIn[1] - N32 * dIn[2];
          T dI = r * dinv[k][0];
          const T sum = lam[k][0] + dI;
          const bool neg = sum < T(0);
          dI = neg ? -lam[k][0] : dI;
          lam[k][0] = neg ? T(0) : sum;
          dIn[k] = dI;
          const T dv = dI * diag[k][0];
          res = fmax_t(res, T(dv * dv));
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
#pragma unroll
          for (int i = 0; i < 6; i++) z[i] += Yn[k][i] * dIn[k];
        }
      }
#pragma unroll
      for (int k = 0; k < 4; k++) {
        T Ya[6], Yb[6];
        if constexpr (kPack) {   // one 64-bit read serves the two feet of a pair: the odd foot's values come from the even foot's reads
          if ((k & 1) == 0) {
#pragma unroll
            for (int i = 0; i < 6; i++) { yab[i] = scr.pair(k >> 1, scr_y(6 + i)); yab[6 + i] = scr.pair(k >> 1, scr_y(12 + i)); }
          }
#pragma unroll
          for (int i = 0; i < 6; i++) { Ya[i] = (k & 1) ? yab[i].y : yab[i].x; Yb[i] = (k & 1) ? yab[6 + i].y : yab[6 + i].x; }
        } else {
#pragma unroll
        for (int i = 0; i < 6; i++) { Ya[i] = scr(k, scr_y(6 + i)); Yb[i] = scr(k, scr_y(12 + i)); }
        }
        const T wa = (H[k][1] * lam[k][0] + H[k][3] * lam[k][1] + H[k][4] * lam[k][2] + Ya[0] * z[0] + Ya[1] * z[1] + Ya[2] * z[2]) +
                     (Ya[3] * z[3] + Ya[4] * z[4] + Ya[5] * z[5]);
        const T wbb = (H[k][2] * lam[k][0] + H[k][4] * lam[k][1] + H[k][5] * lam[k][2] + Yb[0] * z[0] + Yb[1] * z[1] + Yb[2] * z[2]) +
                      (Yb[3] * z[3] + Yb[4] * z[4] + Yb[5] * z[5]);
        T sa = lam[k][1] + (rhs[k][1] - wa) * dinv[k][1];
        T sb = lam[k][2] + (rhs[k][2] - wbb) * dinv[k][2];
        const T lim = mu * T(SC.mu_link) * lam[k][0];
        const T r2 = sa * sa + sb * sb;
        if (r2 >= lim * lim) {
          const T sc2 = r2 > T(0) ? lim * rsqrt_t(r2) : T(0);
          sa *= sc2; sb *= sc2;
        }
        const T dIa = sa - lam[k][1], dIb = sb - lam[k][2];
        lam[k][1] = sa; lam[k][2] = sb;
#pragma unroll
        for (int i = 0; i < 6; i++) z[i] += Ya[i] * dIa + Yb[i] * dIb;
        const T ra = dIa * diag[k][1], rb = dIb * diag[k][2];
        res = fmax_t(res, T(ra * ra + rb * rb));
      }
      if (res <= thr) break;
    }
    // ---- apply: base twist change L^-T z, joint change W lam - B dnu_b
    T dnu[6];
    chol_bwd(S6, Ld, z, dnu);
    T dw[3], dv[3];
    m3_v(X.Rb, dnu, dw);
    m3_v(X.Rb, dnu + 3, dv);
#pragma unroll
    for (int i = 0; i < 3; i++) {
      st.vang[i] = clamp_vel(st.vang[i] + dw[i], mcv);
      st.vlin[i] = clamp_vel(st.vlin[i] + dv[i], mcv);
    }
    if constexpr (kPack) {
      using P = PkT<T>;
#pragma unroll
      for (int kp = 0; kp < 2; kp++) {
        const int k0 = 2 * kp, k1 = k0 + 1;
        const bool on0 = active & (1 << k0), on1 = active & (1 << k1);
#pragma unroll
        for (int j = 0; j < 3; j++) {
          P acc = -(scr.pair(kp, SCR_BM + 6 * j) * P(dnu[0]));
#pragma unroll
          for (int c = 1; c < 6; c++) acc -= scr.pair(kp, SCR_BM + 6 * j + c) * P(dnu[c]);
          // (the W slots of an idle leg hold nothing meaningful: its impulses are zero, its W is read as zero)
#pragma unroll
          for (int c = 0; c < 3; c++) {
            const P w = scr.pair(kp, SCR_W + 3 * j + c);
            acc += P(on0 ? w.x : T(0), on1 ? w.y : T(0)) * P(lam[k0][c], lam[k1][c]);
          }
          const P v = clamp_vel(P(scr.pair(kp, SCR_QD + j) + acc), P(mcv));
          st.qd[3 * k0 + j] = v.x; st.qd[3 * k1 + j] = v.y;
        }
      }
    } else {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const bool on = active & (1 << k);
#pragma unroll
      for (int j = 0; j < 3; j++) {
        T acc = T(0);
#pragma unroll
        for (int c = 0; c < 6; c++) acc -= scr(k, SCR_BM + 6 * j + c) * dnu[c];
        if (on) acc += scr(k, SCR_W + 3 * j) * lam[k][0] + scr(k, SCR_W + 3 * j + 1) * lam[k][1] +
                       scr(k, SCR_W + 3 * j + 2) * lam[k][2];
        st.qd[3 * k + j] = clamp_vel(scr(k, SCR_QD + j) + acc, mcv);
      }
    }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) cs.lam_n[k] = lam[k][0];
  }
  if (!in_contact) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      cs.lam_n[k] = T(0);
#pragma unroll
      for (int j = 0; j < 3; j++) st.qd[3 * k + j] = scr(k, SCR_QD + j);
    }
  }
  cs.mask = active;
  cs.invalid = invalid;
  // the joint angles come back from the scratch (a volatile read: the compiler must not keep the twelve registers
  // alive across the tick instead)
#pragma unroll
  for (int k = 0; k < 4; k++) {
#pragma unroll
    for (int j = 0; j < 3; j++) st.q[3 * k + j] = reload(scr(k, SCR_Q + j));
  }
  integrate_positions(st, dt);
  return TICK_DONE;
}

// ------------------------------------------------------------------------------------------
// GENERAL tick (rare path): joint-limit rows, one contact point per collision shape
// (trunk, imu, hips, thighs, calves, feet) with normal + 2 friction rows each, solved by
// the same reduced-space PGS with one extra 3-vector per leg:
//   w_r = Y_r . z + Jk_r . delta_leg(r),   z += Y_r dI,   delta_leg += M_kk^-1 Jk_r^T dI.
// Row order is the oracle's (Bullet's): limits (alternating direction), all normals in
// link order (trunk, imu, then hip/thigh/calf/foot per leg), all friction cones.
// Rows live in local memory: this runs for the handful of envs the fast tick hands over.
// ------------------------------------------------------------------------------------------
constexpr int QS_MAX_CONTACTS = 2 + 4 * 4;   // every shape can touch at once: trunk, imu, and hip, thigh, calf, foot per leg
constexpr int QS_MAX_LIMITS = 12;

// A general row over u = [z(6), delta_leg0(3), ..., delta_leg3(3)]:  w = a . u,  u += b dI  with a = [Y, Jk in the
// leg's slot], b = [Y, M_kk^-1 Jk^T in the leg's slot].  Rows are stored SPARSE (Y, Jk, W and the leg: 16 words instead
// of the 36 of the dense form) and the twelve delta components live outside the registers, in an array the caller
// provides (`dl`, element c at dl[c * dl_stride]: this thread's column of a shared-memory area in k_step_slow), where
// indexing them by the row's leg costs nothing.  A row visit is 9 + 9 multiply-adds and 16 + 6 loads instead of 18 + 18
// and 36: this kernel is bound by the latency of ONE thread's dependent chain (round 2: -30 % on k_step_slow, which
// had become the step's critical path).
template <typename T> struct alignas(16) GenRow {
  T y[6], jk[3], w[3], dinv, rhs, lam;
  int leg;   // 0..3; rows of the trunk carry zero jk / w on leg 0
};

template <typename T>
QS_DEV void gen_build_row(GenRow<T>& r, int leg, const T* Jb, const T* Jk, const T* Mi, const T* Bm, const T* S6,
                          const T* Ld, const T* wb1, const T* vb1, const T* qd_leg, T* rel_out) {
  T rel = T(0);
  if (Jb) rel = Jb[0] * wb1[0] + Jb[1] * wb1[1] + Jb[2] * wb1[2] + Jb[3] * vb1[0] + Jb[4] * vb1[1] + Jb[5] * vb1[2];
  T Y[6];
#pragma unroll
  for (int c = 0; c < 6; c++) Y[c] = Jb ? Jb[c] : T(0);
  T hdiag = T(0);
  r.leg = leg >= 0 ? leg : 0;
#pragma unroll
  for (int c = 0; c < 3; c++) { r.jk[c] = T(0); r.w[c] = T(0); }
  if (leg >= 0) {
    const T W0 = Mi[0] * Jk[0] + Mi[1] * Jk[1] + Mi[2] * Jk[2];
    const T W1 = Mi[1] * Jk[0] + Mi[3] * Jk[1] + Mi[4] * Jk[2];
    const T W2 = Mi[2] * Jk[0] + Mi[4] * Jk[1] + Mi[5] * Jk[2];
#pragma unroll
    for (int c = 0; c < 6; c++) Y[c] -= Jk[0] * Bm[c] + Jk[1] * Bm[6 + c] + Jk[2] * Bm[12 + c];
    hdiag = Jk[0] * W0 + Jk[1] * W1 + Jk[2] * W2;
    rel += Jk[0] * qd_leg[0] + Jk[1] * qd_leg[1] + Jk[2] * qd_leg[2];
    r.jk[0] = Jk[0]; r.jk[1] = Jk[1]; r.jk[2] = Jk[2];
    r.w[0] = W0; r.w[1] = W1; r.w[2] = W2;
  }
  chol_fwd(S6, Ld, Y);
  T nn = T(0);
#pragma unroll
  for (int c = 0; c < 6; c++) { nn += Y[c] * Y[c]; r.y[c] = Y[c]; }
  r.dinv = div_t(T(1), nn + hdiag);
  r.lam = T(0);
  *rel_out = rel;
}

template <typename T> QS_DEV T gen_row_w(const GenRow<T>& r, const T* z, const T* dl, int ds) {
  const T* d = dl + 3 * r.leg * ds;
  const T w0 = r.y[0] * z[0] + r.y[3] * z[3] + r.jk[0] * d[0];
  const T w1 = r.y[1] * z[1] + r.y[4] * z[4] + r.jk[1] * d[ds];
  const T w2 = r.y[2] * z[2] + r.y[5] * z[5] + r.jk[2] * d[2 * ds];
  return (w0 + w1) + w2;
}
template <typename T> QS_DEV void gen_row_apply(const GenRow<T>& r, T dI, T* z, T* dl, int ds) {
#pragma unroll
  for (int c = 0; c < 6; c++) z[c] += r.y[c] * dI;
  T* d = dl + 3 * r.leg * ds;
  d[0] += r.w[0] * dI; d[ds] += r.w[1] * dI; d[2 * ds] += r.w[2] * dI;
}

// Jacobian of a point pc on body `level` (0 hip, 1 thigh, 2 calf/foot) of a leg
template <typename T>
QS_DEV void body_point_jac(const LegKin<T>& K, int level, const T* pc, const T* d, T* Jb, T* Jk) {
  foot_jac_dir(K, pc, d, Jb, Jk);
  if (level < 2) Jk[2] = T(0);
  if (level < 1) Jk[1] = T(0);
}

// kExt / ext: as physics_tick
template <typename T, bool kEM = false, bool kExt = false>
__host__ __device__ void physics_tick_general(EnvState<T>& st, const T* tau, T mu, ContactState<T>& cs,
                                              const ModelConstT<T>& M, const SolverConst& SC,
                                              const EnvModelRef em, T* dl /* 12 elements, stride dl_stride */, int dl_stride,
                                              const ExtWrench<T>* ext = nullptr) {
  const T dt = T(SC.dt);
  const T mcv = T(SC.max_coord_vel);
  TickCtx<T> X;
  tick_ctx(st, SC, X);
  const T* nb = X.nb;
  const T zero3[3] = {T(0), T(0), T(0)};
  SpI<T> tot;
  trunk_spi<T, kEM>(M, em, tot);
  T fb[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  body_force(tot, X.wb, X.vb, zero3, X.A0, fb, fb + 3);
  if constexpr (kExt) {
    if (ext) sub_ext_wrench(X.Rb, *ext, fb);
  }
  T S6[21];
  for (int i = 0; i < 21; i++) S6[i] = T(0);
  T Bm[4][18], ev[4][3], Mi[4][6];
  LegKin<T> K[4];
  // contact candidates in link order; level -1 = trunk body
  struct Cand { int leg, level, foot; T pc[3]; T gap; };
  Cand cand[QS_MAX_CONTACTS];
  int ncand = 0, invalid = 0, active = 0;
  // trunk box and imu box (link order: trunk, imu come first)
  {
    T zt, zi;
    trunk_shape_gaps(st, X, M, &zt, &zi);
    if (zt < M.trunk_thresh) {
      Cand& c = cand[ncand++];
      c.leg = -1; c.level = -1; c.foot = 0; c.gap = zt;
      for (int a = 0; a < 3; a++) c.pc[a] = (nb[a] > T(0) ? -M.trunk_half[a] : M.trunk_half[a]);
      invalid++;
    }
    if (zi < M.imu_thresh) {
      Cand& c = cand[ncand++];
      c.leg = -1; c.level = -1; c.foot = 0; c.gap = zi;
      for (int a = 0; a < 3; a++) c.pc[a] = M.imu_pos[a] + (nb[a] > T(0) ? -M.imu_half : M.imu_half);
      invalid++;
    }
  }
  for (int k = 0; k < 4; k++) {
    leg_kin(k, st.q + 3 * k, M, K[k]);
    T RH[9], RT[9], RC[9];
    link_rotations(K[k], RH, RT, RC);
    leg_dynamics<T, kEM>(k, st.q + 3 * k, st.qd + 3 * k, tau + 3 * k, X, M, K[k], Mi[k], Bm[k], ev[k], S6, fb, tot, em);
    T zh, zt, zc;
    leg_shape_gaps(st.pos[2], X, M, K[k], RT, RC, &zh, &zt, &zc);
    if (zh < M.hip_thresh) {  // lowest point of the lower rim of the hip cylinder (axis a2)
      Cand& c = cand[ncand++];
      c.leg = k; c.level = 0; c.foot = 0; c.gap = zh;
      const T nz = dot3(nb, K[k].a2);
      T dn[3] = {nb[0] - nz * K[k].a2[0], nb[1] - nz * K[k].a2[1], nb[2] - nz * K[k].a2[2]};
      const T n2 = dot3(dn, dn);
      T rad[3];
      if (n2 > T(1e-18)) { const T sc = M.hip_r * rsqrt_t(n2); for (int a = 0; a < 3; a++) rad[a] = -dn[a] * sc; }
      else { rad[0] = M.hip_r; rad[1] = T(0); rad[2] = T(0); }
      const T sg = nz > T(0) ? T(-1) : T(1);
      for (int a = 0; a < 3; a++) c.pc[a] = K[k].r1[a] + sg * M.hip_hl * K[k].a2[a] + rad[a];
      invalid++;
    }
    if (zt < M.thigh_thresh || zc < M.calf_thresh) {
      for (int b = 0; b < 2; b++) {
        const bool hit = b == 0 ? (zt < M.thigh_thresh) : (zc < M.calf_thresh);
        if (!hit) continue;
        const T* R = b == 0 ? RT : RC;
        const T* half = b == 0 ? M.thigh_half : M.calf_half;
        const T* cen = b == 0 ? M.thigh_c : M.calf_c;
        const T* org = b == 0 ? K[k].r2 : K[k].r3;
        Cand& c = cand[ncand++];
        c.leg = k; c.level = 1 + b; c.foot = 0; c.gap = b == 0 ? zt : zc;
        T loc[3];
        for (int a = 0; a < 3; a++) {
          const T nza = nb[0] * R[a] + nb[1] * R[3 + a] + nb[2] * R[6 + a];
          loc[a] = cen[a] + (nza > T(0) ? -half[a] : half[a]);
        }
        T w3[3];
        m3_v(R, loc, w3);
        for (int a = 0; a < 3; a++) c.pc[a] = org[a] + w3[a];
        invalid++;
      }
    }
    const T gf = st.pos[2] + dot3(nb, K[k].r4) - M.foot_radius;
    if (gf < M.foot_thresh) {
      Cand& c = cand[ncand++];
      c.leg = k; c.level = 2; c.foot = 1; c.gap = gf;
      for (int a = 0; a < 3; a++) c.pc[a] = K[k].r4[a] - M.foot_radius * nb[a];
      active |= 1 << k;
    }
  }
  T Ld[6];
  base_factor(tot, S6, Ld);
  T ab[6];
  {
    T y[6];
    for (int i = 0; i < 6; i++) y[i] = -fb[i];
    chol_fwd(S6, Ld, y);
    chol_bwd(S6, Ld, y, ab);
  }
  ab[3] += X.wxv[0]; ab[4] += X.wxv[1]; ab[5] += X.wxv[2];
  T wb1[3], vb1[3];
  base_velocity_update(st, X, ab, dt, mcv, wb1, vb1);
  for (int k = 0; k < 4; k++)
    for (int j = 0; j < 3; j++) {
      T acc = ev[k][j];
      for (int c = 0; c < 6; c++) acc -= Bm[k][6 * j + c] * ab[c];
      st.qd[3 * k + j] = clamp_vel(st.qd[3 * k + j] + dt * acc, mcv);
    }

  // ---- rows
  GenRow<T> lim[QS_MAX_LIMITS];
  GenRow<T> nrm[QS_MAX_CONTACTS];
  GenRow<T> fr[2 * QS_MAX_CONTACTS];
  int nlim = 0, nn = 0;
  if (SC.enable_limits) {
    for (int k = 0; k < 4; k++)
      for (int j = 0; j < 3; j++)
        for (int side = 0; side < 2; side++) {
          const T qv = st.q[3 * k + j];
          const T pen = side ? M.joint_hi[j] - qv : qv - M.joint_lo[j];
          if (pen > T(0)) continue;
          T Jk[3] = {T(0), T(0), T(0)};
          Jk[j] = side ? T(-1) : T(1);
          T rel;
          gen_build_row(lim[nlim], k, (const T*)nullptr, Jk, Mi[k], Bm[k], S6, Ld, wb1, vb1, st.qd + 3 * k, &rel);
          lim[nlim].rhs = -pen * T(SC.limit_erp) / dt - rel;
          nlim++;
        }
  }
  int foot_of_row[QS_MAX_CONTACTS];
  for (int c = 0; c < ncand; c++) {
    const Cand& cd = cand[c];
    if (!cd.foot && !SC.body_response) continue;
    foot_of_row[nn] = cd.foot ? cd.leg : -1;
    for (int dd = 0; dd < 3; dd++) {
      T Jb[6], Jk[3] = {T(0), T(0), T(0)};
      if (cd.leg >= 0) body_point_jac(K[cd.leg], cd.level, cd.pc, X.tdir[dd], Jb, Jk);
      else { cross3(cd.pc, X.tdir[dd], Jb); Jb[3] = X.tdir[dd][0]; Jb[4] = X.tdir[dd][1]; Jb[5] = X.tdir[dd][2]; }
      GenRow<T>& r = dd == 0 ? nrm[nn] : fr[2 * nn + dd - 1];
      T rel;
      const int lg = cd.leg;
      gen_build_row(r, lg, Jb, Jk, lg >= 0 ? Mi[lg] : (const T*)nullptr, lg >= 0 ? Bm[lg] : (const T*)nullptr, S6, Ld,
                    wb1, vb1, lg >= 0 ? st.qd + 3 * lg : (const T*)nullptr, &rel);
      if (dd == 0) {
        const T dist = cd.gap + T(SC.linear_slop);
        T pos_err = T(0), vel_err = -rel;
        if (dist > T(0)) vel_err -= dist / dt; else pos_err = -dist * T(SC.contact_erp) / dt;
        r.rhs = pos_err + vel_err;
      } else {
        r.rhs = -rel;
      }
    }
    nn++;
  }
  T u[6];   // z; the leg parts (delta) are in dl
#pragma unroll
  for (int c = 0; c < 6; c++) u[c] = T(0);
  for (int c = 0; c < 12; c++) dl[c * dl_stride] = T(0);
  for (int r = 0; r < nn; r++) {  // warm start, feet only
    const int f = foot_of_row[r];
    if (f >= 0 && (cs.mask & (1 << f))) {
      const T imp = cs.lam_n[f] * T(SC.warmstart);
      nrm[r].lam = imp;
      gen_row_apply(nrm[r], imp, u, dl, dl_stride);
    }
  }
  if (nlim + nn > 0) {
    const T thr = T(SC.residual_threshold);
    for (int it = 0; it < SC.num_iterations; it++) {
      T res = T(0);
      for (int j = 0; j < nlim; j++) {
        GenRow<T>& r = lim[(it & 1) ? j : nlim - 1 - j];
        T dI = (r.rhs - gen_row_w(r, u, dl, dl_stride)) * r.dinv;
        const T sum = r.lam + dI;
        if (sum < T(0)) { dI = -r.lam; r.lam = T(0); }
        else if (sum > T(100)) { dI = T(100) - r.lam; r.lam = T(100); }
        else r.lam = sum;
        gen_row_apply(r, dI, u, dl, dl_stride);
        const T dv = div_t(dI, r.dinv);
        res = tmax(res, dv * dv);
      }
      for (int j = 0; j < nn; j++) {
        GenRow<T>& r = nrm[j];
        T dI = (r.rhs - gen_row_w(r, u, dl, dl_stride)) * r.dinv;
        const T sum = r.lam + dI;
        if (sum < T(0)) { dI = -r.lam; r.lam = T(0); } else r.lam = sum;
        gen_row_apply(r, dI, u, dl, dl_stride);
        const T dv = div_t(dI, r.dinv);
        res = tmax(res, dv * dv);
      }
      for (int j = 0; j < nn; j++) {
        GenRow<T>& ra = fr[2 * j];
        GenRow<T>& rb = fr[2 * j + 1];
        T sa = ra.lam + (ra.rhs - gen_row_w(ra, u, dl, dl_stride)) * ra.dinv;
        T sb = rb.lam + (rb.rhs - gen_row_w(rb, u, dl, dl_stride)) * rb.dinv;
        const T limf = mu * T(SC.mu_link) * nrm[j].lam;
        const T r2 = sa * sa + sb * sb;
        if (r2 >= limf * limf) {
          const T sc = r2 > T(0) ? limf * rsqrt_t(r2) : T(0);
          sa *= sc; sb *= sc;
        }
        const T dIa = sa - ra.lam, dIb = sb - rb.lam;
        ra.lam = sa; rb.lam = sb;
        gen_row_apply(ra, dIa, u, dl, dl_stride);
        gen_row_apply(rb, dIb, u, dl, dl_stride);
        const T qa = div_t(dIa, ra.dinv), qb = div_t(dIb, rb.dinv);
        res = tmax(res, qa * qa + qb * qb);
      }
      if (res <= thr) break;
    }
    T dnu[6];
    chol_bwd(S6, Ld, u, dnu);
    T dw[3], dv[3];
    m3_v(X.Rb, dnu, dw);
    m3_v(X.Rb, dnu + 3, dv);
    for (int i = 0; i < 3; i++) {
      st.vang[i] = clamp_vel(st.vang[i] + dw[i], mcv);
      st.vlin[i] = clamp_vel(st.vlin[i] + dv[i], mcv);
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
#pragma unroll
      for (int j = 0; j < 3; j++) {
        T acc = dl[(3 * k + j) * dl_stride];
        for (int c = 0; c < 6; c++) acc -= Bm[k][6 * j + c] * dnu[c];
        st.qd[3 * k + j] = clamp_vel(st.qd[3 * k + j] + acc, mcv);
      }
  }
  cs.mask = active;
  cs.invalid = invalid;
  for (int k = 0; k < 4; k++) cs.lam_n[k] = T(0);
  for (int r = 0; r < nn; r++)
    if (foot_of_row[r] >= 0) cs.lam_n[foot_of_row[r]] = nrm[r].lam;
  integrate_positions(st, dt);
}

}  // namespace qs
