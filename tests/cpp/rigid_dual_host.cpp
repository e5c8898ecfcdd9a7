// TEST INFRASTRUCTURE - NOT PRODUCT CODE, never loaded by the package.
// The dual-number instance of the rigid-body world kernel (tiny-differentiable-simulator_b200/csrc/tds_rigid.cu) compiled FOR THE HOST
// like tests/cpp/rigid_host.cpp does, driven through its DualIO parameter: the products behind tds_b200_rigid_{jvp,vjp}_device.
//   g++ -std=c++17 -O1 -shared -fPIC -I<csrc> -I<include> -I/usr/local/cuda/include tests/cpp/rigid_dual_host.cpp -o tests/cpp/_rigid_dual_host.so
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>
#include <vector>

#define TDS_B200_EXACT_RCP 1
#define TDS_RIGID_KERNEL_ONLY 1
namespace emu { struct Dim { unsigned x, y, z; }; static Dim tIdx, bIdx, bDim; }
#define threadIdx emu::tIdx
#define blockIdx emu::bIdx
#define blockDim emu::bDim
#undef __global__
#define __global__
#undef __grid_constant__
#define __grid_constant__
#undef __launch_bounds__
#define __launch_bounds__(...)

#include "../../tiny-differentiable-simulator_b200/csrc/tds_rigid.cu"

extern "C" {
// Jacobian-vector / vector-Jacobian products through the dual instance's DualIO path, launched the way
// tds_b200_rigid_{jvp,vjp}_device (tds_rigid.cu) launches it.  Arrays [n][13 nb] (state) / [n][3 nb] (force).  JVP when t_out is
// set: t_state, t_force (null = zero) -> t_out.  VJP when g_out is set: -> g_state, g_force (null = not wanted, not launched).
int tdsemu_rigid_dual(const double* desc, int nb, const double* params, int n, const double* state, const double* force, int steps,
                      const double* t_state, const double* t_force, double* t_out, const double* g_out, double* g_state, double* g_force) {
  RigidWorld W;
  { const int rcw = tds_rigid_world_from_desc(desc, nb, &W); if (rcw) return rcw; }
  W.dt = params[0]; for (int k = 0; k < 3; ++k) W.gravity[k] = params[1 + k];
  W.friction = params[4]; W.restitution = params[5]; W.erp = params[6]; W.num_solver_iterations = (int)params[7];
  const int ns = (n + 31) & ~31, rows = 13 * nb;
  auto soa = [&](const double* a, int d) {
    std::vector<double> v((size_t)d * ns, 0.0);
    if (a) for (int e = 0; e < n; ++e) for (int k = 0; k < d; ++k) v[(size_t)k * ns + e] = a[(size_t)e * d + k];
    return v;
  };
  auto aos = [&](const std::vector<double>& v, int d, double* a) {
    for (int e = 0; e < n; ++e) for (int k = 0; k < d; ++k) a[(size_t)e * d + k] = v[(size_t)k * ns + e];
  };
  std::vector<double> s = soa(state, rows), f = soa(force, 3 * nb), ts = soa(t_state, rows), tf = soa(t_force, 3 * nb),
                      to = soa(nullptr, rows), cot = soa(g_out, rows), gs = soa(nullptr, rows), gf = soa(nullptr, 3 * nb);
  const bool force_used = force || t_force || g_force;   // a null force is zero force
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  emu::bDim = {1, 1, 1};
  emu::tIdx = {0, 0, 0};
  auto run = [&](int n_dirs, int dir0) {
    for (int e = 0; e < n; ++e)
      for (int d = 0; d < n_dirs; ++d) {
        emu::bIdx = {(unsigned)e, (unsigned)d, 0};
        tdsrb::tds_rigid_step_kernel<tds::Dual<double>, double>(W, s.data(), nullptr, force_used ? f.data() : nullptr, steps, n, ns,
                                                                nullptr, dir0, dio);
      }
  };
  if (t_out) {
    dio.jvp_tan[0] = t_state ? ts.data() : nullptr; dio.jvp_tan[1] = t_force ? tf.data() : nullptr; dio.jvp_out = to.data();
    run(1, 0);
    aos(to, rows, t_out);
    memset(&dio, 0, sizeof(dio));
  }
  if (g_out) {
    dio.vjp_cot = cot.data(); dio.vjp_out[0] = g_state ? gs.data() : nullptr; dio.vjp_out[1] = g_force ? gf.data() : nullptr;
    if (g_state) { run(rows, 0); aos(gs, rows, g_state); }
    if (g_force) { run(3 * nb, rows); aos(gf, 3 * nb, g_force); }
  }
  return 0;
}
}  // extern "C"
