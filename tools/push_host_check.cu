// push_host_check.cu -- the pushed tick (kExt instantiation of physics_tick / physics_tick_general, csrc/qs_physics.cuh)
// on the HOST in fp64.  Reads cases from a text file, one per line:
//   n_ticks mu state[37] tau[12] force[3] (world, N) point[3] (base frame, from the base position, m)
// and runs each case three times for n_ticks ticks, the fast tick handing a tick to the general solver when it asks
// (as k_debug_ticks does):
//   P  kExt, pushed on every tick
//   Z  kExt, with no push (ext == nullptr)
//   D  the default instantiation
// Every tick prints "<run> <case> <tick> <rc> <state[37]>" with %.17g (exact round trip of a double).
// tests/test_external_force.py builds it twice (default and -DQS_PACK_LEGS=0) and checks P and D against the oracle
// World given the same force, and Z against D bit for bit.  No GPU needed.
//   nvcc -std=c++17 -w [-DQS_PACK_LEGS=0] -o /tmp/push_host_check tools/push_host_check.cu && /tmp/push_host_check in.txt out.txt
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../quadruped_springs_b200/csrc/qs_physics.cuh"
#include "../quadruped_springs_b200/csrc/qs_model_host.h"
using namespace qs;
using T = double;

static void dump(FILE* f, char run, int c, int t, int rc, const EnvState<T>& st) {
  std::fprintf(f, "%c %d %d %d", run, c, t, rc);
  for (int i = 0; i < 3; i++) std::fprintf(f, " %.17g", st.pos[i]);
  for (int i = 0; i < 4; i++) std::fprintf(f, " %.17g", st.quat[i]);
  for (int i = 0; i < 3; i++) std::fprintf(f, " %.17g", st.vlin[i]);
  for (int i = 0; i < 3; i++) std::fprintf(f, " %.17g", st.vang[i]);
  for (int i = 0; i < 12; i++) std::fprintf(f, " %.17g", st.q[i]);
  for (int i = 0; i < 12; i++) std::fprintf(f, " %.17g", st.qd[i]);
  std::fprintf(f, "\n");
}

int main(int argc, char** argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: %s in.txt out.txt\n", argv[0]); return 2; }
  ModelConstT<T> M;
  host::build_model<T>(M, 0.02);
  ModelLegPairsT<T> M2;
  make_leg_pairs(M, M2);
  SolverConst SC;   // the oracle's default World parameters (oracle/qso_physics.c qso_default_params)
  std::memset(&SC, 0, sizeof SC);
  SC.dt = 1e-3f; SC.gravity_z = -9.8f; SC.contact_erp = 0.08f; SC.limit_erp = 0.2f; SC.linear_slop = 1e-5f;
  SC.warmstart = 0.1f; SC.residual_threshold = 1e-7f; SC.max_coord_vel = 30.1f; SC.mu_link = 1.f;
  SC.num_iterations = 30; SC.enable_limits = 1; SC.body_response = 1;
  FILE* in = std::fopen(argv[1], "r");
  FILE* out = std::fopen(argv[2], "w");
  if (!in || !out) { std::perror("push_host_check"); return 1; }
  static T scratch[QS_TICK_SCRATCH];
  const Scratch<T> scr{scratch, 1};
  const EnvModelRef em{nullptr, 0, 0};
  int n_ticks, cases = 0;
  while (std::fscanf(in, "%d", &n_ticks) == 1) {
    double mu, s[37], tau[12], w6[6];
    if (std::fscanf(in, "%lf", &mu) != 1) return 3;
    for (double& v : s) if (std::fscanf(in, "%lf", &v) != 1) return 3;
    for (double& v : tau) if (std::fscanf(in, "%lf", &v) != 1) return 3;
    for (double& v : w6) if (std::fscanf(in, "%lf", &v) != 1) return 3;
    ExtWrench<T> w;
    for (int i = 0; i < 3; i++) { w.f[i] = w6[i]; w.p[i] = w6[3 + i]; }
    for (const char run : {'P', 'Z', 'D'}) {
      EnvState<T> st;
      ContactState<T> cs;
      std::memset(&st, 0, sizeof st);
      std::memset(&cs, 0, sizeof cs);
      for (int i = 0; i < 3; i++) { st.pos[i] = s[i]; st.vlin[i] = s[7 + i]; st.vang[i] = s[10 + i]; }
      for (int i = 0; i < 4; i++) st.quat[i] = s[3 + i];
      for (int i = 0; i < 12; i++) { st.q[i] = s[13 + i]; st.qd[i] = s[25 + i]; }
      for (int t = 0; t < n_ticks; t++) {
        int rc;
        T dl[12];
        if (run == 'D') {
          rc = physics_tick<T>(st, tau, T(mu), cs, M, SC, true, scr, em, &M2);
          if (rc) physics_tick_general<T>(st, tau, T(mu), cs, M, SC, em, dl, 1);
        } else {
          const ExtWrench<T>* ext = run == 'P' ? &w : nullptr;
          rc = physics_tick<T, true, 0, false, true>(st, tau, T(mu), cs, M, SC, true, scr, em, &M2, ext);
          if (rc) physics_tick_general<T, false, true>(st, tau, T(mu), cs, M, SC, em, dl, 1, ext);
        }
        dump(out, run, cases, t, rc, st);
      }
    }
    cases++;
  }
  std::fclose(in);
  std::fclose(out);
  std::printf("push_host_check ok: %d cases (QS_PACK_LEGS=%d)\n", cases, int(QS_PACK_LEGS));
  return 0;
}
