// TEST INFRASTRUCTURE - NOT PRODUCT CODE, never loaded by the package.
// The dual-number instance of the generic step kernel (tiny-differentiable-simulator_b200/csrc/tds_stepw.cu) compiled FOR THE HOST,
// with the same single-lane meanings of the CUDA built-ins as tests/cpp/stepw_host.cpp, driven through its DualIO parameter:
// the Jacobian-vector and vector-Jacobian products behind tds_b200_step_{jvp,vjp}_device.
//   g++ -std=c++17 -O1 -shared -fPIC -I<csrc> -I<include> -I/usr/local/cuda/include tests/cpp/stepw_dual_host.cpp -o tests/cpp/_stepw_dual_host.so
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#define TDS_B200_EXACT_RCP 1
#define TDS_STEPW_KERNEL_ONLY 1
struct EmuDim { unsigned x, y, z; };
static thread_local EmuDim emu_threadIdx, emu_blockIdx, emu_blockDim, emu_gridDim;
#define threadIdx emu_threadIdx
#define blockIdx emu_blockIdx
#define blockDim emu_blockDim
#define gridDim emu_gridDim
#define __any_sync(mask, pred) ((pred) ? 1 : 0)
#define __reduce_max_sync(mask, v) (v)
static inline float __int_as_float(int i) { float f; memcpy(&f, &i, 4); return f; }
#define __syncwarp() ((void)0)
#define clock64() (0LL)
#undef __shared__
#define __shared__
#undef __grid_constant__
#define __grid_constant__
#undef __global__
#define __global__
#undef __launch_bounds__
#define __launch_bounds__(...)
alignas(16) char smem_raw[16];

#include "tds_model.h"
#include "../../tiny-differentiable-simulator_b200/csrc/tds_stepw.cu"

extern "C" {

// Jacobian-vector / vector-Jacobian products through the dual instance's DualIO path, launched the way
// tds_b200_step_{jvp,vjp}_device (tds_capi.cu) launches it.  Arguments as tdsemu_stepw; every tangent / gradient array is
// [n][dim] (blocks q | qd | tau or action).  JVP when t_out is set: t_q, t_qd, t_tau (null = zero) -> t_out [n][rows].
// VJP when g_out [n][rows] is set: -> g_q, g_qd, g_tau (null = not wanted, not launched).  Returns rows * 1000 + columns.
int tdsemu_stepw_dual(const double* model, int n_model, const double* params, const double* env, int mode, int use_pd, int n,
                      const double* q, const double* qd, const double* tau, const double* t_q, const double* t_qd,
                      const double* t_tau, double* t_out, const double* g_out, double* g_q, double* g_qd, double* g_tau) {
  DevModel* D = new DevModel;
  int rc = tds_build_dev_model(model, n_model, D);
  if (rc) { delete D; return rc; }
  tds_build_layout_w(D, 16, 16, 16, -1, 16);
  SimParams P;
  memset(&P, 0, sizeof(P));
  P.dt = params[0]; P.inv_dt = 1.0 / params[0];
  for (int k = 0; k < 3; ++k) P.gravity[k] = params[1 + k];
  P.friction = params[4]; P.restitution = params[5]; P.erp = params[6]; P.cfm = params[7];
  P.pgs_iterations = (int)params[8]; P.keep_all_points = (int)params[9];
  P.contact_model = (int)params[10]; P.spring_k = params[11]; P.damper_d = params[12]; P.exponent_n = params[13];
  P.v_transition = params[14]; P.hard_contact_condition = (int)params[15];
  EnvParams E;
  memset(&E, 0, sizeof(E));
  if (env) {
    E.n_act = (int)env[0]; E.start_link = (int)env[1];
    E.kp = (float)env[2]; E.kd = (float)env[3]; E.max_force = (float)env[4]; E.action_limit = (float)env[5];
    int k = 0;
    for (int i = D->floating ? 0 : E.start_link; i < D->n_links && k < E.n_act; ++i) {
      if (D->flags[i] & TDS_LF_FIXED) continue;
      E.act_link[k] = i; E.initial_poses[k] = (float)env[6 + k]; ++k;
    }
  }
  const int ns = (n + 31) & ~31, n_q = D->n_q, n_qd = D->n_qd;
  const int n_tau = n_qd - (D->floating ? 6 : 0), n_in = use_pd ? E.n_act : n_tau;
  const int rows = mode == 0 ? n_qd : n_q + n_qd;
  const int dim[3] = {n_q, n_qd, n_in}, first[3] = {0, n_q, n_q + n_qd};
  auto soa_f = [&](const double* a, int d) {
    std::vector<float> v((size_t)(d > 0 ? d : 1) * ns, 0.f);
    if (a) for (int e = 0; e < n; ++e) for (int k = 0; k < d; ++k) v[(size_t)k * ns + e] = (float)a[(size_t)e * d + k];
    return v;
  };
  auto soa_d = [&](const double* a, int d) {
    std::vector<double> v((size_t)(d > 0 ? d : 1) * ns, 0.0);
    if (a) for (int e = 0; e < n; ++e) for (int k = 0; k < d; ++k) v[(size_t)k * ns + e] = a[(size_t)e * d + k];
    return v;
  };
  auto aos_d = [&](const std::vector<double>& v, int d, double* a) {
    for (int e = 0; e < n; ++e) for (int k = 0; k < d; ++k) a[(size_t)e * d + k] = v[(size_t)k * ns + e];
  };
  std::vector<float> sq = soa_f(q, n_q), sqd = soa_f(qd, n_qd), st = soa_f(tau, n_in);
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.q_in = sq.data(); io.qd_in = sqd.data(); io.tau_in = (tau || use_pd) ? st.data() : nullptr;
  io.n = n; io.n_stride = ns;
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  const double* tan_in[3] = {t_q, t_qd, t_tau};
  double* grad[3] = {g_q, g_qd, g_tau};
  std::vector<double> tan[3], gout[3], tout = soa_d(nullptr, rows), cot = soa_d(g_out, rows);
  for (int b = 0; b < 3; ++b) {
    if (tan_in[b]) { tan[b] = soa_d(tan_in[b], dim[b]); dio.jvp_tan[b] = tan[b].data(); }
    if (grad[b]) { gout[b] = soa_d(nullptr, dim[b]); dio.vjp_out[b] = gout[b].data(); }
  }
  auto run = [&](int n_dirs) {
    std::vector<char> scratch((size_t)n_dirs * ((n + 31) / 32) * D->x_total * 32 * 4 + 64);
    const int warps = (n + 31) / 32;
    emu_blockDim = {32, 1, 1};
    emu_gridDim = {(unsigned)warps, (unsigned)n_dirs, 1};
    for (unsigned by = 0; by < (unsigned)n_dirs; ++by)
      for (unsigned bx = 0; bx < (unsigned)warps; ++bx)
        for (unsigned t = 0; t < 32; ++t) {
          if ((int)(bx * 32 + t) >= n) continue;
          emu_blockIdx = {bx, by, 0};
          emu_threadIdx = {t, 0, 0};
          typedef tds::Dual<double> DD;
          tdsw::tds_stepw_kernel<DD, DD, DD, DD, false>(*D, P, E, io, mode, use_pd, scratch.data(), dio);
        }
  };
  if (t_out) {
    dio.jvp_out = tout.data();
    run(1);
    aos_d(tout, rows, t_out);
    dio.jvp_out = nullptr;
  }
  if (g_out) {
    dio.vjp_cot = cot.data();
    for (int b = 0; b < 3; ++b) {
      if (!grad[b] || dim[b] == 0) continue;
      io.jac_dir0 = first[b];
      run(dim[b]);
      aos_d(gout[b], dim[b], grad[b]);
    }
  }
  const int cols = n_q + n_qd + n_in;
  delete D;
  return rows * 1000 + cols;
}

}  // extern "C"
