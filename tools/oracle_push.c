/* oracle_push.c -- Bullet's applyExternalForce(robot, -1, F, x, WORLD_FRAME) on the base (Quadruped.apply_external_force,
 * quadruped.py:338-343) for the CPU oracle, as test infrastructure beside it: the oracle's sources are compiled in
 * unchanged, and a push acts through the oracle's own qso_world_step.
 *
 * In Bullet the force enters the unconstrained dynamics of the step: v2 = v + dt (a(v) + M^-1 J^T F), after which the
 * contact and limit solver and the integration run on v2.  qso_world_step computes v2 = v + dt a(v) from the stored
 * velocities (its step 2, ABA + RNEA) and uses the stored velocities nowhere else.  qsp_push_before_step therefore
 * replaces them by the v' whose unconstrained update is the pushed one, v' + dt a(v') = v + dt (a(v) + M^-1 J^T F),
 * solved by fixed-point iteration (the map contracts by dt |da/dv|, about 1e-3 per round: fp64 rounding after a few
 * rounds); the step that follows is then the pushed step to rounding.  The contact history (warm start) is kept.
 * A zero force leaves every velocity bit-identical; calls before one step add up.
 *
 *   gcc -O2 -fPIC -std=c11 -D_GNU_SOURCE -shared -o liboracle_push.so tools/oracle_push.c -lm
 *
 * Usage on a World of the oracle library (same sources, same struct layout): add the tick's joint torques
 * (qso_world_add_torque), call qsp_push_before_step(w, F, x), then qso_world_step(w). */
#include "../oracle/qso_physics.c"

/* the stored velocities (world base omega, world base velocity, joint rates) after step 2 of qso_world_step, before its
 * clamp: the same operations as that step */
static void unconstrained_velocity(QsoWorld* w, double* out) {
  double nu[ND], h[ND], f[ND], acc[ND], t[3], dw[3], dv[3];
  const double dt = w->P.dt;
  kinematics(w);
  aba_factor(w);
  gen_vel(w, nu);
  rnea(w, nu, NULL, 1, h);
  for (int k = 0; k < 6; k++) f[k] = -h[k];
  for (int k = 0; k < 12; k++) f[6 + k] = w->tau[k] - h[6 + k];
  aba_solve(w, f, acc);
  cross(nu, nu + 3, t);
  for (int k = 0; k < 3; k++) acc[3 + k] += t[k];
  m3_v(w->Rw[0], acc, dw);
  m3_v(w->Rw[0], acc + 3, dv);
  for (int k = 0; k < 3; k++) { out[k] = w->vang[k] + dt * dw[k]; out[3 + k] = w->vlin[k] + dt * dv[k]; }
  for (int k = 0; k < 12; k++) out[6 + k] = w->qd[k] + dt * acc[6 + k];
}

void qsp_push_before_step(QsoWorld* w, const double* force, const double* pos) {
  const double dt = w->P.dt;
  double target[ND], cur[ND], fe[ND], d[ND], r[3], n[3], dw[3], dv[3];
  unconstrained_velocity(w, target);   /* (runs the kinematics and the ABA factor of the current pose) */
  /* the generalized force of the push: [n_b, f_b] in base coordinates about the base origin, no joint part */
  for (int k = 0; k < 3; k++) r[k] = pos[k] - w->pos[k];
  cross(r, force, n);
  memset(fe, 0, sizeof fe);
  m3t_v(w->Rw[0], n, fe);
  m3t_v(w->Rw[0], force, fe + 3);
  aba_solve(w, fe, d);
  m3_v(w->Rw[0], d, dw);
  m3_v(w->Rw[0], d + 3, dv);
  for (int k = 0; k < 3; k++) { target[k] += dt * dw[k]; target[3 + k] += dt * dv[k]; }
  for (int k = 0; k < 12; k++) target[6 + k] += dt * d[6 + k];
  for (int it = 0; it < 12; it++) {
    unconstrained_velocity(w, cur);
    int changed = 0;
    for (int k = 0; k < 3; k++) {
      const double ew = target[k] - cur[k], ev = target[3 + k] - cur[3 + k];
      changed |= (ew != 0) | (ev != 0);
      w->vang[k] += ew;
      w->vlin[k] += ev;
    }
    for (int k = 0; k < 12; k++) {
      const double e = target[6 + k] - cur[6 + k];
      changed |= e != 0;
      w->qd[k] += e;
    }
    if (!changed) break;
  }
}
