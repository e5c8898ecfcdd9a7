// C-ABI of libtds_b200.so (include/tds_b200.h): simulator lifecycle, device fast path, host-buffer
// paths and the reference's "C-ABI v1" drop-in symbols for the Laikago model.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "tds_b200.h"
#include "tds_b200_model.h"
#include "tds_model.h"
#include "tds_types.h"
#include "tds_team.h"

extern "C" int tds_launch_stept(const TeamModel* TM, const TeamLink* tl_dev, const DevModel* M, const SimParams* P,
                                const EnvParams* E, const StepIO* io, int mode, int use_pd, int precision,
                                char* gscratch, int use_smem, cudaStream_t stream);
extern "C" unsigned long long tds_stepr_table_owner(int dev);
extern "C" int tds_launch_stepr(const TeamModel* TM, const TeamLink* tl_host, unsigned long long token, const DevModel* M,
                                const SimParams* P, const EnvParams* E, const StepIO* io, int mode, int use_pd,
                                int precision, char* gscratch, int use_smem, cudaStream_t stream);
extern "C" size_t tds_stepr_tile_bytes(const TeamModel* TM);
extern "C" int tds_spec_find(const double* model, int n_model, const DevModel* D, const EnvParams* E);
extern "C" size_t tds_spec_smem_bytes(int spec, int precision);
extern "C" const char* tds_spec_name(int spec);
extern "C" int tds_launch_step_spec(int spec, const SimParams* P, const EnvParams* E, const StepIO* io, int mode, int use_pd,
                                    int precision, cudaStream_t stream);
extern "C" int tds_launch_stepw_dual(const DevModel* M, const SimParams* P, const EnvParams* E, const StepIO* io, const DualIO* dio,
                                     int mode, int use_pd, int n_dirs, char* gscratch, cudaStream_t stream);
extern "C" int tds_launch_stepw(const DevModel* M, const SimParams* P, const EnvParams* E, const StepIO* io,
                                int mode, int use_pd, int precision, char* gscratch, int use_smem,
                                int warps_per_block, cudaStream_t stream);

// candidate contact points of a model, reference enumeration order: (link_a, link_b) per point
// (plane candidates first, then - worlds of several multibodies - the candidates between multibodies, list after list)
struct ContactCandTable {
  int n_points;
  signed char link_a[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS], link_b[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS];   // link index inside its multibody
  signed char body_a[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS], body_b[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS];   // multibody of the world (0 = the plane)
  signed char geom_a[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS], geom_b[TDS_MAX_POINTS + TDS_MAX_PAIR_POINTS];   // index in collision_geometries(link)
};

// Candidate points of a model in the reference's enumeration order (World::compute_contacts_multi_body_internal,
// src/world.hpp:212-281).  The plane is multibody 0 of the world, created first (body A of its contacts, base link -1); the
// multibodies of the model follow as 1, 2, ...; link indices are the reference's: inside their multibody.
static ContactCandTable make_cand_table(const DevModel& D) {
  ContactCandTable T;
  memset(&T, 0, sizeof(T));
  int first[TDS_MAX_LINKS + 1];   // first link of every multibody
  for (int i = 0, b = -1; i < D.n_links; ++i) if (D.body_of[i] != b) { b = D.body_of[i]; first[b] = i; }
  auto local = [&](int link) { return link < 0 ? -1 : link - first[D.body_of[link]]; };
  auto geom_in_link = [&](int g) { return g - D.geom_begin[D.g_link[g] + 1]; };   // iii / jjj of the reference's loops
  int c = 0;
  if (D.has_plane)
    for (int g = 0; g < D.n_geoms; ++g) {
      const int pts = D.g_type[g] == TDSG_SPHERE ? 1 : (D.g_type[g] == TDSG_CAPSULE ? 2 : (D.g_type[g] == TDSG_BOX ? 8 : 0));
      for (int j = 0; j < pts; ++j, ++c) {
        T.body_a[c] = 0; T.link_a[c] = -1; T.geom_a[c] = 0; T.geom_b[c] = (signed char)geom_in_link(g);
        T.body_b[c] = (signed char)(1 + (D.g_link[g] < 0 ? 0 : D.body_of[D.g_link[g]])); T.link_b[c] = (signed char)local(D.g_link[g]);
      }
    }
  for (int p = 0; p < D.n_pair_points; ++p, ++c) {
    const int la = D.g_link[D.pp_ga[p]], lb = D.g_link[D.pp_gb[p]];
    T.body_a[c] = (signed char)(1 + D.body_of[la]); T.link_a[c] = (signed char)local(la);
    T.body_b[c] = (signed char)(1 + D.body_of[lb]); T.link_b[c] = (signed char)local(lb);
    T.geom_a[c] = (signed char)geom_in_link(D.pp_ga[p]); T.geom_b[c] = (signed char)geom_in_link(D.pp_gb[p]);
  }
  T.n_points = c;
  return T;
}

namespace {

std::string g_err;  // mirror of the last error (the public accessor lives in urdf_model.cpp)
extern "C" void tds_b200_set_error(const char* msg);
void set_err(const std::string& s) { g_err = s; tds_b200_set_error(s.c_str()); }

#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_err(std::string(#expr) + ": " + cudaGetErrorString(_e));                      \
      return (int)_e;                                                                   \
    }                                                                                   \
  } while (0)

// ---- layout conversion kernels (host AoS fp64/fp32 <-> device SoA fp32) --------------------------
template <typename TI>
__global__ void aos_to_soa_kernel(const TI* __restrict__ in, int in_stride, int in_off, float* __restrict__ out,
                                  int dim, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  for (int k = 0; k < dim; ++k) out[(size_t)k * ns + e] = (float)in[(size_t)e * in_stride + in_off + k];
}
template <typename TO>
__global__ void soa_to_aos_kernel(const float* __restrict__ in, TO* __restrict__ out, int out_stride, int out_off,
                                  int dim, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  for (int k = 0; k < dim; ++k) out[(size_t)e * out_stride + out_off + k] = (TO)in[(size_t)k * ns + e];
}

// obs[e] = q | qd (AoS), and optionally reward / done appended behind the n observation rows (one contiguous
// block -> one device->host copy when the caller's three output buffers are adjacent)
__global__ void pack_env_out_kernel(const float* __restrict__ q, const float* __restrict__ qd, const float* __restrict__ reward,
                                    const float* __restrict__ done, float* __restrict__ out, int n_q, int n_qd, int n, int ns,
                                    int with_tail) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float* o = out + (size_t)e * (n_q + n_qd);
  for (int k = 0; k < n_q; ++k) o[k] = q[(size_t)k * ns + e];
  for (int k = 0; k < n_qd; ++k) o[n_q + k] = qd[(size_t)k * ns + e];
  if (with_tail) {
    float* tail = out + (size_t)n * (n_q + n_qd);
    tail[e] = reward[e];
    tail[n + e] = done[e];
  }
}

// TinyMatrix3x3::getRotation, src/math/tiny/tiny_matrix3x3.h:434-466 (used for the visual outputs)
__device__ void matrix_to_quat_dev(const float* m, float* q) {
  float trace = m[0] + m[4] + m[8];
  float temp[4];
  if (trace < 0.f) {
    int i = m[0] < m[4] ? (m[4] < m[8] ? 2 : 1) : (m[0] < m[8] ? 2 : 0);
    int j = (i + 1) % 3, k = (i + 2) % 3;
    float tmp = ((m[i * 3 + i] - m[j * 3 + j]) - m[k * 3 + k]) + 1.f;
    float s = sqrtf(tmp);
    temp[i] = s * 0.5f;
    s = 0.5f / s;
    temp[3] = (m[j * 3 + k] - m[k * 3 + j]) * s;
    temp[j] = (m[i * 3 + j] + m[j * 3 + i]) * s;
    temp[k] = (m[i * 3 + k] + m[k * 3 + i]) * s;
  } else {
    float s = sqrtf(trace + 1.f);
    temp[3] = s * 0.5f;
    s = 0.5f / s;
    temp[0] = (m[5] - m[7]) * s;
    temp[1] = (m[6] - m[2]) * s;
    temp[2] = (m[1] - m[3]) * s;
  }
  q[0] = temp[0]; q[1] = temp[1]; q[2] = temp[2]; q[3] = -temp[3];
}

// Output packing of LocomotionContactSimulation::step_forward_original,
// examples/environments/locomotion_contact_simulation.h:273-303: q | qd | visuals (pos3, quat4) | up.z
__global__ void pack_v1_output_kernel(const __grid_constant__ DevVisuals V, const float* __restrict__ q,
                                      const float* __restrict__ qd, const float* __restrict__ link_xf,
                                      double* __restrict__ out, int out_dim, int n, int ns, int floating) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double* o = out + (size_t)e * out_dim;
  int j = 0;
  for (int k = 0; k < V.n_q; ++k) o[j++] = (double)q[(size_t)k * ns + e];
  for (int k = 0; k < V.n_qd; ++k) o[j++] = (double)qd[(size_t)k * ns + e];
  for (int v = 0; v < V.n_vis; ++v) {
    const float* x = link_xf + (size_t)V.v_link[v] * 12 * ns + e;
    float R[9], t[3], Rv[9], q4[4];
    for (int k = 0; k < 9; ++k) R[k] = x[(size_t)k * ns];
    for (int k = 0; k < 3; ++k) t[k] = x[(size_t)(9 + k) * ns];
    for (int r = 0; r < 3; ++r) {
      o[j++] = (double)(t[r] + R[r * 3] * V.v_t[v][0] + R[r * 3 + 1] * V.v_t[v][1] + R[r * 3 + 2] * V.v_t[v][2]);
      for (int c = 0; c < 3; ++c)
        Rv[r * 3 + c] = R[r * 3] * V.v_R[v][c] + R[r * 3 + 1] * V.v_R[v][3 + c] + R[r * 3 + 2] * V.v_R[v][6 + c];
    }
    matrix_to_quat_dev(Rv, q4);
    o[j++] = q4[0]; o[j++] = q4[1]; o[j++] = q4[2]; o[j++] = q4[3];
  }
  double upz = 1.0;  // base_X_world.rotation(2,2): identity for fixed base (:131), else from the new base quat
  if (floating) {
    const double x = q[e], y = q[(size_t)ns + e], z = q[(size_t)2 * ns + e], w = q[(size_t)3 * ns + e];
    upz = 1.0 - 2.0 * (x * x + y * y) / (x * x + y * y + z * z + w * w);
  }
  o[j++] = upz;
}

// Visual-transform stream in the instancing renderer's layout (SURVEY 8f.2): instance i = env * n_vis + v;
// positions[4 i + {0,1,2,3}] = x, y, z, 1 and orientations[4 i + {0..3}] = quaternion xyzw, the two arrays
// TinyGLInstancingRenderer keeps (src/visualizer/opengl/tiny_gl_instancing_renderer.cpp:366-367, 440-457).  Same
// per-visual transform as the v1 output records (locomotion_contact_simulation.h:281-299).
__global__ void pack_visual_instances_kernel(const __grid_constant__ DevVisuals V, const float* __restrict__ link_xf,
                                             float4* __restrict__ positions, float4* __restrict__ orientations, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int v = blockIdx.y;
  if (e >= n) return;
  const float* x = link_xf + (size_t)V.v_link[v] * 12 * ns + e;
  float R[9], t[3], Rv[9], q4[4], p[3];
  for (int k = 0; k < 9; ++k) R[k] = x[(size_t)k * ns];
  for (int k = 0; k < 3; ++k) t[k] = x[(size_t)(9 + k) * ns];
  for (int r = 0; r < 3; ++r) {
    p[r] = t[r] + R[r * 3] * V.v_t[v][0] + R[r * 3 + 1] * V.v_t[v][1] + R[r * 3 + 2] * V.v_t[v][2];
    for (int c = 0; c < 3; ++c)
      Rv[r * 3 + c] = R[r * 3] * V.v_R[v][c] + R[r * 3 + 1] * V.v_R[v][3 + c] + R[r * 3 + 2] * V.v_R[v][6 + c];
  }
  matrix_to_quat_dev(Rv, q4);
  const size_t i = (size_t)e * V.n_vis + v;
  positions[i] = make_float4(p[0], p[1], p[2], 1.f);
  orientations[i] = make_float4(q4[0], q4[1], q4[2], q4[3]);
}

// ---- environment layer on the device (SURVEY 8f.1) ---------------------------------------------------------------
// counter-based uniform in [0, 1): splitmix64 of (seed, environment, joint)
__device__ inline float unit_uniform(unsigned long long seed, unsigned e, unsigned a) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (((unsigned long long)e << 8) + a + 1ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}
// LaikagoContactSimulation::reset, laikago_environment2.h:63-89: reset pose, joint noise on the actuated joints, qd = 0
__global__ void env_reset_fill_kernel(float* __restrict__ q, float* __restrict__ qd, const float* __restrict__ noise, float amp,
                                      unsigned long long seed, EnvParams E, int n_q, int n_qd, const int* __restrict__ act_qidx,
                                      int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  for (int k = 0; k < n_q; ++k) q[(size_t)k * ns + e] = E.reset_q[k];
  for (int k = 0; k < n_qd; ++k) qd[(size_t)k * ns + e] = 0.f;
  for (int a = 0; a < E.n_act; ++a) {
    const float d = noise ? noise[(size_t)a * ns + e] : amp * (2.f * unit_uniform(seed, (unsigned)e, (unsigned)a) - 1.f);
    q[(size_t)act_qidx[a] * ns + e] += d;
  }
}
__global__ void env_select_kernel(const float* __restrict__ mask, const float* __restrict__ q_src, const float* __restrict__ qd_src,
                                  float* __restrict__ q, float* __restrict__ qd, int n_q, int n_qd, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n || (mask && mask[e] == 0.f)) return;
  for (int k = 0; k < n_q; ++k) q[(size_t)k * ns + e] = q_src[(size_t)k * ns + e];
  for (int k = 0; k < n_qd; ++k) qd[(size_t)k * ns + e] = qd_src[(size_t)k * ns + e];
}
// VectorizedEnvironment::policy (ars_vectorized_environment.h:293-300): one linear layer with bias per environment
// (neural_network.hpp:223-265, parameters = weights [n_act][n_obs] row-major | biases [n_act]); the observation is
// q | qd with x and y zeroed (ars_vectorized_environment.h:285-287).  params: [n_params][ns] on the device.
// One thread per (environment, action): blockIdx.y = action; consecutive threads = consecutive environments, so every
// parameter / state row is read coalesced.
__global__ void policy_linear_kernel(const float* __restrict__ q, const float* __restrict__ qd, const float* __restrict__ params,
                                     float* __restrict__ act, int n_q, int n_qd, int n_act, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = blockIdx.y;
  if (e >= n) return;
  const int n_obs = n_q + n_qd;
  float s = params[(size_t)(n_act * n_obs + a) * ns + e];
  const float* w = params + (size_t)a * n_obs * ns + e;
#pragma unroll 4
  for (int k = 2; k < n_q; ++k) s += q[(size_t)k * ns + e] * w[(size_t)k * ns];
#pragma unroll 4
  for (int k = 0; k < n_qd; ++k) s += qd[(size_t)k * ns + e] * w[(size_t)(n_q + k) * ns];
  act[(size_t)a * ns + e] = s;
}
// ARSVectorizedWorker::rollouts bookkeeping (ars_vectorized_worker.h:117-139): done is sticky, rewards and step counts
// accumulate only while the environment is alive
__global__ void rollout_accum_kernel(const float* __restrict__ reward, const float* __restrict__ done, float shift,
                                     float* __restrict__ sticky, float* __restrict__ total, int* __restrict__ steps, int n) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  if (sticky[e] != 0.f) return;
  if (done[e] != 0.f) { sticky[e] = 1.f; return; }
  total[e] += reward[e] - shift;
  steps[e] += 1;
}
// Contact-pair index list of one step, in the reference's enumeration order (World::compute_contacts_multi_body_internal,
// src/world.hpp:212-281: bodies i < j, links of A, geoms of A, links of B, geoms of B, points in emission order).  The
// candidate points of a model are static (every sphere / capsule end emits one point, contact_point.hpp:112-124,149-158);
// what varies per environment is which of them the constraint solver keeps: all with keep_all_points_, else those with
// distance < 0 (MultiBodyConstraintSolver::resolve_collision, src/mb_constraint_solver.hpp:169-180).
// links: [2 * n_points][ns] = (link_a, link_b) of the k-th kept point (MultiBodyContactPoint::link_a/b, :29-40), -9 beyond count.
// cand (optional): [n_points][ns] index of the k-th kept point in the candidate list (tds_b200_contact_pairs), -9 beyond count.
// A distance of +inf marks a candidate between multibodies whose contact function emitted nothing (contact_point.hpp:80).
__global__ void contact_list_kernel(const float* __restrict__ dist, ContactCandTable T, int keep_all, int* __restrict__ count,
                                    int* __restrict__ links, int* __restrict__ cand, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int k = 0;
  for (int c = 0; c < T.n_points; ++c) {
    const float d = dist[(size_t)c * ns + e];
    if (d < 3.0e38f && (keep_all || d < 0.f)) {
      links[(size_t)(2 * k) * ns + e] = T.link_a[c];
      links[(size_t)(2 * k + 1) * ns + e] = T.link_b[c];
      if (cand) cand[(size_t)k * ns + e] = c;
      ++k;
    }
  }
  count[e] = k;
  for (; k < T.n_points; ++k) {
    links[(size_t)(2 * k) * ns + e] = -9; links[(size_t)(2 * k + 1) * ns + e] = -9;
    if (cand) cand[(size_t)k * ns + e] = -9;
  }
}
// integrate_euler (src/dynamics/integrator.hpp:10-133) and integrate_euler_qdd (:141-195) as stand-alone stages of the
// fine-grained pytinydiffsim surface (forward_dynamics -> integrate_euler_qdd -> World::step -> integrate_euler): the fused
// step kernels do the same arithmetic in their epilogues.  qdd may be null (= the zero vector integrate_euler_qdd leaves).
struct IntegrateTable { int n_links, floating, n_q, n_qd; signed char q_idx[TDS_MAX_LINKS], qd_idx[TDS_MAX_LINKS], fixed[TDS_MAX_LINKS]; };
__global__ void integrate_euler_kernel(float* __restrict__ q, float* __restrict__ qd, const float* __restrict__ qdd, double dt,
                                       IntegrateTable T, int update_q, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  auto Q = [&](int k) -> float& { return q[(size_t)k * ns + e]; };
  auto QD = [&](int k) -> float& { return qd[(size_t)k * ns + e]; };
  if (qdd) for (int k = 0; k < T.n_qd; ++k) QD(k) = (float)((double)QD(k) + (double)qdd[(size_t)k * ns + e] * dt);
  if (!update_q) return;
  if (T.floating) {   // quat_velocity + quat_increment + normalize (tiny_algebra.hpp:604-614)
    const double h = 0.5 * dt;
    double qx = Q(0), qy = Q(1), qz = Q(2), qw = Q(3);
    const double w0 = QD(0), w1 = QD(1), w2 = QD(2);
    const double dw = (-qx * w0 - qy * w1 - qz * w2) * h, dx = (qw * w0 + qz * w1 - qy * w2) * h;
    const double dy = (qw * w1 + qx * w2 - qz * w0) * h, dz = (qw * w2 + qy * w0 - qx * w1) * h;
    qx += dx; qy += dy; qz += dz; qw += dw;
    const double len = sqrt(qx * qx + qy * qy + qz * qz + qw * qw);
    Q(0) = (float)(qx / len); Q(1) = (float)(qy / len); Q(2) = (float)(qz / len); Q(3) = (float)(qw / len);
    for (int k = 0; k < 3; ++k) Q(4 + k) = (float)((double)Q(4 + k) + (double)QD(3 + k) * dt);
  }
  for (int i = 0; i < T.n_links; ++i)
    if (!T.fixed[i]) Q(T.q_idx[i]) = (float)((double)Q(T.q_idx[i]) + (double)QD(T.qd_idx[i]) * dt);
}
// ---- ARS on the device (examples/ars/ars_vectorized_worker.h, ars_learner.h) --------------------------------------
// Observation filter statistics, ars_vectorized_worker.h:93-110: every rollout step pushes the observation the policy saw
// (q | qd with x, y zeroed) into a per-(environment, component) RunningStat (running_stat.h:17-37, Welford).
// stats: [3 * n_obs][ns] = count | mean | S per component; sticky (may be null): finished environments stop pushing -
// the reference keeps pushing the frozen observation of a done environment, which only inflates its count; documented.
__global__ void obs_stat_push_kernel(const float* __restrict__ q, const float* __restrict__ qd, float* __restrict__ stats,
                                     int n_q, int n_qd, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int o = blockIdx.y;
  if (e >= n) return;
  const int n_obs = n_q + n_qd;
  float x = o < n_q ? q[(size_t)o * ns + e] : qd[(size_t)(o - n_q) * ns + e];
  if (o < 2) x = 0.f;                                   // ars_vectorized_environment.h:285-287
  float* cnt = stats + (size_t)o * ns + e;
  float* mean = stats + (size_t)(n_obs + o) * ns + e;
  float* S = stats + (size_t)(2 * n_obs + o) * ns + e;
  const float c = *cnt + 1.f;
  if (c == 1.f) { *mean = x; *S = 0.f; }
  else { const float m0 = *mean, m1 = m0 + (x - m0) / c; *S += (x - m0) * (x - m1); *mean = m1; }
  *cnt = c;
}
// per-environment policy parameters of a perturbed rollout: params[p][e] = w[p] + sign * delta_std * delta[p][e]
// (ARSVectorizedWorker::do_rollouts, ars_vectorized_worker.h:205-262)
__global__ void ars_perturb_kernel(const float* __restrict__ w, const float* __restrict__ deltas, float scale,
                                   float* __restrict__ params, int n, int ns) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int p = blockIdx.y;
  if (e >= n) return;
  params[(size_t)p * ns + e] = w[p] + scale * deltas[(size_t)p * ns + e];
}
// ARSLearner::weighted_sum_custom + train_step (ars_learner.h:67-91,185-189): g_hat[p] = (1 / N) sum_e (r+ - r-)[e]
// delta[p][e] delta_std ; w[p] += step_size g_hat[p].  One block per parameter, tree reduction over the environments.
__global__ void ars_update_kernel(float* __restrict__ w, const float* __restrict__ deltas, const float* __restrict__ r_pos,
                                  const float* __restrict__ r_neg, float delta_std, float step_size, int n, int ns) {
  __shared__ float red[256];
  const int p = blockIdx.x;
  float acc = 0.f;
  for (int e = threadIdx.x; e < n; e += blockDim.x) acc += (r_pos[e] - r_neg[e]) * deltas[(size_t)p * ns + e];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) w[p] += step_size * (red[0] * delta_std / (float)n);
}
__global__ void rollout_init_kernel(float* sticky, float* total, int* steps, int n) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) { sticky[e] = 0.f; total[e] = 0.f; steps[e] = 0; }
}

}  // namespace

struct tds_b200_sim {
  int device = 0;
  int n = 0, ns = 0;
  DevModel dm[3];         // one layout per precision mode
  DevModel dm_ad;         // layout of the differentiable instance (dual numbers, 16-byte scalars)
  char* jac_scratch = nullptr; size_t jac_scratch_bytes = 0;
  double* jac_dev = nullptr; size_t jac_dev_bytes = 0;
  bool smem_ok[3] = {false, false, false};
  bool smem_ok_w[3] = {false, false, false};
  // 3: role-warp kernel (tds_stepr.cu), 2: lane-team kernel (tds_stept.cu), 1: one-lane world-frame kernel
  // (tds_stepw.cu).  Requests fall back 3 -> 2 -> 1 when the model has no
  // tree decomposition (chains) or a tile does not fit in shared memory.
  // 4: ahead-of-time specialised kernel (tds_steps.cu) when the model is one it was generated for, else 3.
  int kernel = 4;
  int kernel_req = 4;
  bool spec_ok = false;
  int spec_idx = -1;       // which compiled model (tds_steps.cu) equals this simulator's, -1: none
  std::vector<double> model;   // flat model (identity check of the specialised kernel)
  bool smem_ok_r[3] = {false, false, false};
  unsigned long long table_token = 0;
  bool team_ok = false;
  bool smem_ok_t[3] = {false, false, false};
  TeamModel tm[3];
  std::vector<TeamLink> team_table;
  TeamLink* team_dev = nullptr;
  int warps_per_block[3] = {1, 1, 1};
  DevVisuals vis;
  SimParams P;
  EnvParams E;
  int precision_req = TDS_B200_PREC_AUTO;   // what the caller asked for
  int precision = TDS_B200_PREC_F64;        // what runs: AUTO resolves to MIXED for a model with a compiled (validated)
                                            // instance, else to the strict F64 (rebuild_team)
  int n_tau = 0, n_points = 0;
  ContactCandTable cand;              // static candidate table (reference enumeration order)
  int *c_count = nullptr, *c_links = nullptr, *c_cand = nullptr;   // device: per-environment contact list of the last tds_b200_contact_list_* call
  // resident state + staging
  float *q = nullptr, *qd = nullptr, *act = nullptr, *qdd = nullptr, *reward = nullptr, *done = nullptr;
  float *cdist = nullptr, *link_xf = nullptr;
  char* scratch = nullptr;
  size_t scratch_bytes = 0;
  void* stage_dev = nullptr;   // device staging for AoS host buffers
  size_t stage_dev_bytes = 0;
  void* stage_host = nullptr;  // pinned host staging
  size_t stage_host_bytes = 0;
  cudaStream_t stream = nullptr;
  int max_smem_optin = 0;
  long long* phase_clk = nullptr;  // profiling only (tds_b200_debug_phase_clocks)
  // tds_b200_env_step_host with pinned caller buffers: the copy / transpose / step / copy sequence is captured once
  // per buffer set and replayed (one graph launch instead of nine stream operations)
  // environment layer scratch: reset staging, zero actions, actuated coordinate map, rollout bookkeeping
  float *rq = nullptr, *rqd = nullptr, *zero_act = nullptr, *pol_act = nullptr, *sticky = nullptr, *r_total = nullptr, *pol_params = nullptr;
  int *act_qidx = nullptr, *r_steps = nullptr;
  float* obs_stats = nullptr;      // caller-owned [3 * n_obs][ns] running statistics of the observation filter, or null
  bool act_qidx_valid = false;
  size_t pol_params_rows = 0;
  // set around the step launch of tds_b200_env_step_host when the specialised kernel serves the host layouts itself
  const float* io_act_aos = nullptr; float* io_obs_aos = nullptr; float* io_obs_tail = nullptr;
  const void* zc_key[4] = {nullptr, nullptr, nullptr, nullptr};   // zero-copy path: last buffer set and its device aliases
  void* zc_dev[4] = {nullptr, nullptr, nullptr, nullptr};
  bool zc_ok = false;
  unsigned zc_calls = 0;          // the cached classification is re-validated every 64 calls
  const void* g_key[4] = {nullptr, nullptr, nullptr, nullptr};
  int g_seen = 0;
  cudaGraphExec_t g_exec = nullptr;
};

static void drop_host_graph(tds_b200_sim* s) {
  if (s->g_exec) { cudaGraphExecDestroy(s->g_exec); s->g_exec = nullptr; }
  s->g_seen = 0;
  s->g_key[0] = s->g_key[1] = s->g_key[2] = s->g_key[3] = nullptr;
}

static bool is_pinned(const void* p) {
  if (!p) return true;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

static int ensure_stage(tds_b200_sim* s, size_t dev_bytes, size_t host_bytes) {
  if (dev_bytes > s->stage_dev_bytes) {
    // the graph of tds_b200_env_step_host holds addresses inside the staging buffer: it dies with the buffer
    drop_host_graph(s);
    if (s->stage_dev) cudaFree(s->stage_dev);
    s->stage_dev = nullptr; s->stage_dev_bytes = 0;
    CUDA_TRY(cudaMalloc(&s->stage_dev, dev_bytes));
    s->stage_dev_bytes = dev_bytes;
  }
  if (host_bytes > s->stage_host_bytes) {
    if (s->stage_host) cudaFreeHost(s->stage_host);
    s->stage_host = nullptr; s->stage_host_bytes = 0;
    CUDA_TRY(cudaMallocHost(&s->stage_host, host_bytes));
    s->stage_host_bytes = host_bytes;
  }
  return 0;
}

static int ensure_scratch(tds_b200_sim* s, int prec) {
  const int words = s->dm[prec].w_total > s->dm[prec].x_total ? s->dm[prec].w_total : s->dm[prec].x_total;
  size_t need = (size_t)words * 4 * s->ns;
  if (need > s->scratch_bytes) {
    if (s->scratch) cudaFree(s->scratch);
    s->scratch = nullptr; s->scratch_bytes = 0;
    CUDA_TRY(cudaMalloc((void**)&s->scratch, need));
    s->scratch_bytes = need;
  }
  return 0;
}

// (Re)build the team decomposition: depends on the model and on the action -> link map of the environment.
static int rebuild_team(tds_b200_sim* s) {
  s->team_ok = false;
  s->spec_ok = false; s->spec_idx = -1;
  TeamModel base;
  if (s->precision_req == TDS_B200_PREC_AUTO) s->precision = TDS_B200_PREC_F64;
  if (s->dm[0].world_only) return 0;   // box shapes / spherical joints: the generic world-frame kernel serves the model
  int rc = tds_build_team(&s->dm[0], &s->E, &base, &s->team_table);
  if (rc != 0) return 0;   // chains etc.: the one-lane kernel is used
  const int sizes[3][3] = {{4, 8, 4}, {8, 8, 8}, {4, 4, 4}};
  for (int p = 0; p < 3; ++p) {
    s->tm[p] = base;
    tds_build_team_layout(&s->tm[p], sizes[p][0], sizes[p][1], sizes[p][2]);
    const size_t warp_bytes = ((size_t)s->tm[p].t_total * (32 / TDS_TEAM_T) + (size_t)s->tm[p].l_total * 32) * 4;
    s->smem_ok_t[p] = warp_bytes <= (size_t)s->max_smem_optin;
    s->smem_ok_r[p] = tds_stepr_tile_bytes(&s->tm[p]) <= (size_t)s->max_smem_optin;
  }
  static unsigned long long next_token = 1;
  s->table_token = next_token++;
  s->spec_idx = tds_spec_find(s->model.data(), (int)s->model.size(), &s->dm[0], &s->E);
  s->spec_ok = s->spec_idx >= 0;
  if (s->precision_req == TDS_B200_PREC_AUTO) s->precision = s->spec_ok ? TDS_B200_PREC_MIXED : TDS_B200_PREC_F64;
  if (!s->team_dev) CUDA_TRY(cudaMalloc((void**)&s->team_dev, sizeof(TeamLink) * TDS_TEAM_T * TDS_TEAM_MAXK));
  CUDA_TRY(cudaMemcpy(s->team_dev, s->team_table.data(), sizeof(TeamLink) * TDS_TEAM_T * TDS_TEAM_MAXK, cudaMemcpyHostToDevice));
  s->team_ok = true;
  return 0;
}

extern "C" {

static const char* tds_model_error(int rc) {
  switch (rc) {
    case -1: return "not a flat model of this layout version (magic / size mismatch)";
    case -2: return "too many links, collision geoms or candidate contact points (TDS_MAX_LINKS / TDS_MAX_GEOMS / TDS_MAX_POINTS)";
    case -3: return "unknown joint type";
    case -4: return "links are not ordered parent before child";
    case -5: return "collision geoms are not grouped by link";
    case -6: return "mesh collision shape against the ground plane: the contact stage implements sphere, capsule and box";
    case -7: return "world of several multibodies (TDSM_H_NBODIES): fixed base only, links of a multibody contiguous, as many root links as multibodies";
    default: return "unknown error";
  }
}

// Host-only check (no GPU needed): 0 when tds_b200_create would accept the model, else the negative code; the reason
// is left in tds_b200_last_error().
int tds_b200_validate_model(const double* model, int n_model) {
  if (!model) { set_err("null model"); return -1; }
  DevModel* D = new DevModel;
  const int rc = tds_build_dev_model(model, n_model, D);
  delete D;
  if (rc) set_err(std::string("unsupported model: ") + tds_model_error(rc));
  return rc;
}

tds_b200_sim* tds_b200_create(const double* model, int n_model, int n_envs, int device) {
  if (!model || n_envs <= 0) { set_err("bad arguments"); return nullptr; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_err("no CUDA device available: libtds_b200 has no CPU fallback");
    return nullptr;
  }
  if (cudaSetDevice(device) != cudaSuccess) { set_err("cudaSetDevice failed"); return nullptr; }
  tds_b200_sim* s = new tds_b200_sim;
  s->device = device;
  s->n = n_envs;
  s->ns = (n_envs + 31) & ~31;
  DevModel base;
  int rc = tds_build_dev_model(model, n_model, &base);
  if (rc) {
    set_err(std::string("unsupported model: ") + tds_model_error(rc));
    delete s;
    return nullptr;
  }
  cudaDeviceGetAttribute(&s->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  const int sizes[3][3] = {{4, 8, 4}, {8, 8, 8}, {4, 4, 4}};  // sizeof(RA, RC, RS) per precision mode
  for (int p = 0; p < 3; ++p) {
    s->dm[p] = base;
    tds_build_layout(&s->dm[p], sizes[p][0], sizes[p][1], sizes[p][2], -1);
    tds_build_layout_w(&s->dm[p], sizes[p][0], sizes[p][1], sizes[p][2], -1);
    size_t per_warp = (size_t)s->dm[p].w_total * 32 * 4;
    s->smem_ok[p] = per_warp <= (size_t)s->max_smem_optin;
    s->smem_ok_w[p] = (size_t)s->dm[p].x_total * 32 * 4 <= (size_t)s->max_smem_optin;
    // several warps per block only help when many blocks would otherwise be needed per SM
    s->warps_per_block[p] = 1;
  }
  s->dm_ad = base;
  tds_build_layout_w(&s->dm_ad, 16, 16, 16, -1, 16);
  s->model.assign(model, model + n_model);
  if (const char* kv = getenv("TDS_B200_KERNEL"))
    s->kernel_req = strcmp(kv, "world") == 0 ? 1 : (strcmp(kv, "team") == 0 ? 2 : (strcmp(kv, "role") == 0 ? 3 : 4));
  s->kernel = s->kernel_req;
  s->n_tau = base.n_qd - (base.floating ? 6 : 0);
  s->n_points = base.max_contacts + base.n_pair_points;
  s->cand = make_cand_table(base);
  // visuals for the v1 output packing
  memset(&s->vis, 0, sizeof(s->vis));
  {
    const double* vis = model + TDSM_HEADER + TDSM_BASE + (size_t)base.n_links * TDSM_LINK + (size_t)base.n_geoms * TDSM_GEOM;
    int nv = base.n_vis < TDS_MAX_VIS ? base.n_vis : TDS_MAX_VIS;
    s->vis.n_vis = nv; s->vis.n_links = base.n_links; s->vis.n_q = base.n_q; s->vis.n_qd = base.n_qd;
    for (int v = 0; v < nv; ++v) {
      const double* r = vis + (size_t)v * TDSM_VIS;
      s->vis.v_link[v] = (int)r[TDSM_V_LINK];
      for (int k = 0; k < 9; ++k) s->vis.v_R[v][k] = (float)r[TDSM_V_R + k];
      for (int k = 0; k < 3; ++k) s->vis.v_t[v][k] = (float)r[TDSM_V_T + k];
    }
  }
  // defaults = the reference's (world.hpp:65-72, mb_constraint_solver.hpp:59-70)
  s->P.dt = 1e-3; s->P.inv_dt = 1.0 / s->P.dt;
  s->P.gravity[0] = 0; s->P.gravity[1] = 0; s->P.gravity[2] = -9.81;
  s->P.friction = 0.5; s->P.restitution = 0.0; s->P.erp = 0.2; s->P.cfm = 1e-5;
  s->P.pgs_iterations = 1; s->P.keep_all_points = 0;
  s->P.contact_model = 0; s->P.hard_contact_condition = 1;
  s->P.spring_k = 50000.0; s->P.damper_d = 5000.0; s->P.exponent_n = 1.5; s->P.v_transition = 0.01;
  memset(&s->E, 0, sizeof(s->E));
  const size_t ns = s->ns;
  auto alloc = [&](float** p, size_t rows) { return cudaMalloc((void**)p, sizeof(float) * rows * ns) == cudaSuccess && cudaMemset(*p, 0, sizeof(float) * rows * ns) == cudaSuccess; };
  bool ok = alloc(&s->q, base.n_q > 0 ? base.n_q : 1) && alloc(&s->qd, base.n_qd > 0 ? base.n_qd : 1) &&
            alloc(&s->act, (base.n_qd > TDS_MAX_ACT ? base.n_qd : TDS_MAX_ACT)) && alloc(&s->qdd, base.n_qd > 0 ? base.n_qd : 1) &&
            alloc(&s->reward, 1) && alloc(&s->done, 1) && alloc(&s->cdist, s->n_points > 0 ? s->n_points : 1) &&
            alloc(&s->link_xf, (size_t)(base.n_links > 0 ? base.n_links : 1) * 12);
  if (!ok || cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess || rebuild_team(s) != 0) {
    set_err("device allocation failed");
    tds_b200_destroy(s);
    return nullptr;
  }
  return s;
}

void tds_b200_destroy(tds_b200_sim* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  cudaFree(s->q); cudaFree(s->qd); cudaFree(s->act); cudaFree(s->qdd); cudaFree(s->reward); cudaFree(s->done);
  drop_host_graph(s);
  cudaFree(s->rq); cudaFree(s->rqd); cudaFree(s->zero_act); cudaFree(s->pol_act); cudaFree(s->sticky); cudaFree(s->r_total);
  cudaFree(s->pol_params); cudaFree(s->act_qidx); cudaFree(s->r_steps);
  cudaFree(s->c_count); cudaFree(s->c_links); cudaFree(s->c_cand); cudaFree(s->jac_scratch); cudaFree(s->jac_dev);
  cudaFree(s->cdist); cudaFree(s->link_xf); cudaFree(s->scratch); cudaFree(s->stage_dev); cudaFree(s->phase_clk); cudaFree(s->team_dev);
  if (s->stage_host) cudaFreeHost(s->stage_host);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int tds_b200_set_params(tds_b200_sim* s, double dt, const double gravity[3], double friction, double restitution,
                        double erp, double cfm, int pgs_iterations, int keep_all_points) {
  if (!s) return -1;
  drop_host_graph(s);
  s->P.dt = dt; s->P.inv_dt = 1.0 / dt;
  for (int k = 0; k < 3; ++k) s->P.gravity[k] = gravity[k];
  s->P.friction = friction; s->P.restitution = restitution; s->P.erp = erp; s->P.cfm = cfm;
  s->P.pgs_iterations = pgs_iterations; s->P.keep_all_points = keep_all_points;
  return 0;
}

int tds_b200_set_contact_model(tds_b200_sim* s, int contact_model, double spring_k, double damper_d, double exponent_n,
                               double v_transition, int hard_contact_condition) {
  if (!s || contact_model < 0 || contact_model > 1) { set_err("contact_model must be 0 (LCP) or 1 (spring-damper)"); return -1; }
  if (contact_model == 1 && !(spring_k >= 0.0 && damper_d >= 0.0 && exponent_n > 0.0 && v_transition > 0.0)) {
    set_err("spring-damper parameters out of range"); return -2;
  }
  drop_host_graph(s);
  s->P.contact_model = contact_model; s->P.hard_contact_condition = hard_contact_condition ? 1 : 0;
  s->P.spring_k = spring_k; s->P.damper_d = damper_d; s->P.exponent_n = exponent_n; s->P.v_transition = v_transition;
  return 0;
}

int tds_b200_set_env(tds_b200_sim* s, int n_act, const double* initial_poses, int start_link, double kp, double kd,
                     double max_force, double action_limit, int reward_kind) {
  if (!s || n_act < 0 || n_act > TDS_MAX_ACT) { set_err("bad n_act"); return -1; }
  drop_host_graph(s);
  const DevModel& M = s->dm[0];
  EnvParams E;
  memset(&E, 0, sizeof(E));
  E.n_act = n_act; E.start_link = start_link;
  E.kp = (float)kp; E.kd = (float)kd; E.max_force = (float)max_force; E.action_limit = (float)action_limit;
  E.reward_kind = reward_kind;
  int k = 0;
  const int first = M.floating ? 0 : start_link;  // locomotion_contact_simulation.h:181
  for (int i = first; i < M.n_links && k < n_act; ++i) {
    if (M.flags[i] & TDS_LF_FIXED) continue;
    E.act_link[k] = i;
    E.initial_poses[k] = (float)initial_poses[k];
    ++k;
  }
  if (k != n_act) { set_err("model has fewer actuated links than n_act"); return -2; }
  E.auto_reset = s->E.auto_reset;
  memcpy(E.reset_q, s->E.reset_q, sizeof(E.reset_q));
  s->E = E;
  s->act_qidx_valid = false;
  return rebuild_team(s);
}

int tds_b200_set_auto_reset(tds_b200_sim* s, int enable, const double* reset_q) {
  if (!s) return -1;
  const DevModel& M = s->dm[0];
  if (enable && !reset_q) { set_err("auto-reset needs a reset pose"); return -1; }
  drop_host_graph(s);
  s->E.auto_reset = enable ? 1 : 0;
  if (reset_q)
    for (int k = 0; k < M.n_q; ++k) s->E.reset_q[k] = (float)reset_q[k];
  return 0;
}

int tds_b200_set_precision(tds_b200_sim* s, int precision) {
  if (!s || precision < TDS_B200_PREC_AUTO || precision > 2) return -1;
  drop_host_graph(s);
  s->precision_req = precision;
  s->precision = precision != TDS_B200_PREC_AUTO ? precision : (s->spec_ok ? TDS_B200_PREC_MIXED : TDS_B200_PREC_F64);
  return 0;
}

int tds_b200_get_dims(const tds_b200_sim* s, int dims[8]) {
  if (!s) return -1;
  const DevModel& M = s->dm[0];
  dims[0] = s->n; dims[1] = s->ns; dims[2] = M.n_q; dims[3] = M.n_qd; dims[4] = s->n_tau; dims[5] = M.n_links;
  dims[6] = s->n_points; dims[7] = s->E.n_act;
  return 0;
}

int tds_b200_step_device(tds_b200_sim* s, int mode, int use_pd, const float* q_in, const float* qd_in,
                         const float* tau_or_action, float* q_out, float* qd_out, float* qdd_out, float* reward,
                         float* done, float* contact_dist, float* link_xf, void* stream) {
  if (!s) return -1;
  const int p = s->precision;
  StepIO io;
  io.q_in = q_in; io.qd_in = qd_in; io.tau_in = tau_or_action;
  io.q_out = q_out; io.qd_out = qd_out; io.qdd_out = qdd_out;
  io.reward = reward; io.done = done; io.contact_dist = contact_dist; io.link_xf = link_xf;
  io.phase_clk = s->phase_clk;
  io.act_aos = s->io_act_aos; io.obs_aos = s->io_obs_aos; io.obs_tail = s->io_obs_tail;
  io.jac = nullptr; io.jac_n_in = 0; io.jac_dir0 = 0;
  io.n = s->n; io.n_stride = s->ns;
  if (use_pd && s->E.n_act == 0) { set_err("use_pd without tds_b200_set_env"); return -3; }
  int kern = s->kernel_req;
  if (s->dm[0].world_only || mode == 3 || s->P.contact_model != 0) kern = 1;   // (mode 3 = TDS_B200_MODE_WORLD)   // box shapes / spherical joints: served by the generic world-frame kernel only
  if (kern == 4 && !(s->spec_ok && tds_spec_smem_bytes(s->spec_idx, p) <= (size_t)s->max_smem_optin)) kern = 3;
  if (kern == 4) {
    s->kernel = kern;
    static const int solo = getenv("TDS_B200_DEBUG_SOLO") ? 256 : 0;   // profiling aid, see tds_steps.cu
    int rcs = tds_launch_step_spec(s->spec_idx, &s->P, &s->E, &io, mode | solo, use_pd, p, (cudaStream_t)stream);
    if (rcs) set_err(std::string("specialised step launch: ") + cudaGetErrorString((cudaError_t)rcs));
    return rcs;
  }
  if (kern == 3 && !(s->team_ok && s->smem_ok_r[p])) kern = 2;
  if (kern == 2 && !s->team_ok) kern = 1;
  s->kernel = kern;
  if (kern == 3) {
    int rcr = tds_launch_stepr(&s->tm[p], s->team_table.data(), s->table_token, &s->dm[p], &s->P, &s->E, &io, mode, use_pd, p,
                               nullptr, 1, (cudaStream_t)stream);
    if (rcr) set_err(std::string("role-warp step launch: ") + cudaGetErrorString((cudaError_t)rcr));
    return rcr;
  }
  if (kern == 2) {
    const int use_smem_t = s->smem_ok_t[p] ? 1 : 0;
    if (!use_smem_t) {
      const size_t warp_bytes = ((size_t)s->tm[p].t_total * (32 / TDS_TEAM_T) + (size_t)s->tm[p].l_total * 32) * 4;
      const size_t need = warp_bytes * ((s->n + (32 / TDS_TEAM_T) - 1) / (32 / TDS_TEAM_T));
      if (need > s->scratch_bytes) {
        if (s->scratch) cudaFree(s->scratch);
        s->scratch = nullptr; s->scratch_bytes = 0;
        CUDA_TRY(cudaMalloc((void**)&s->scratch, need));
        s->scratch_bytes = need;
      }
    }
    int rct = tds_launch_stept(&s->tm[p], s->team_dev, &s->dm[p], &s->P, &s->E, &io, mode, use_pd, p, s->scratch, use_smem_t,
                               (cudaStream_t)stream);
    if (rct) set_err(std::string("team step launch: ") + cudaGetErrorString((cudaError_t)rct));
    return rct;
  }
  const int use_smem = s->smem_ok_w[p] ? 1 : 0;
  if (!use_smem) { int rc = ensure_scratch(s, p); if (rc) return rc; }
  int rc = tds_launch_stepw(&s->dm[p], &s->P, &s->E, &io, mode, use_pd, p, s->scratch, use_smem,
                            s->warps_per_block[p], (cudaStream_t)stream);
  if (rc) set_err(std::string("step launch: ") + cudaGetErrorString((cudaError_t)rc));
  return rc;
}

// ---- differentiable step (SURVEY 8f.4): d(q', qd') / d(q, qd, tau | action, kp, kd, max_force), or d qdd / d(...) in
// forward-dynamics mode, by forward-mode dual numbers through the world-frame step kernel (tds_stepw.cu, tds_dual.cuh).
int tds_b200_jacobian_dims(const tds_b200_sim* s, int mode, int use_pd, int dims[2]) {
  if (!s || !dims) return -1;
  const DevModel& M = s->dm[0];
  dims[0] = mode == TDS_B200_MODE_FD ? M.n_qd : M.n_q + M.n_qd;
  dims[1] = M.n_q + M.n_qd + (use_pd ? s->E.n_act + 3 : s->n_tau);
  return 0;
}

// Scratch of the dual-number instance for launches of up to `dirs` directions, bounded by 2 GB (more directions: several
// launches of *chunk).  Grows only when a call needs more than the arena holds.
static int ensure_dual_scratch(tds_b200_sim* s, int dirs, int* chunk) {
  const size_t warps = (size_t)(s->n + 31) / 32;
  const size_t per_dir = warps * (size_t)s->dm_ad.x_total * 32 * 4;
  const size_t cap = (size_t)2 << 30;
  int c = (int)(cap / per_dir);
  if (c < 1) c = 1;
  if (c > dirs) c = dirs;
  if (per_dir * c > s->jac_scratch_bytes) {
    if (s->jac_scratch) cudaFree(s->jac_scratch);
    s->jac_scratch = nullptr; s->jac_scratch_bytes = 0;
    CUDA_TRY(cudaMalloc((void**)&s->jac_scratch, per_dir * c));
    s->jac_scratch_bytes = per_dir * c;
  }
  *chunk = c;
  return 0;
}

int tds_b200_step_jacobian_device(tds_b200_sim* s, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                                  double* jac, void* stream) {
  if (!s || !q || !qd || !jac) return -1;
  if (mode == 3) { set_err("jacobian: modes FD, NOCONTACT, FULL"); return -2; }
  if (use_pd && s->E.n_act == 0) { set_err("use_pd without tds_b200_set_env"); return -3; }
  int dims[2];
  tds_b200_jacobian_dims(s, mode, use_pd, dims);
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.q_in = q; io.qd_in = qd; io.tau_in = tau_or_action;
  io.jac = jac; io.jac_n_in = dims[1];
  io.n = s->n; io.n_stride = s->ns;
  DualIO none;
  memset(&none, 0, sizeof(none));
  int chunk;
  int rc = ensure_dual_scratch(s, dims[1], &chunk);
  if (rc) return rc;
  for (int d0 = 0; d0 < dims[1]; d0 += chunk) {
    io.jac_dir0 = d0;
    const int nd = dims[1] - d0 < chunk ? dims[1] - d0 : chunk;
    rc = tds_launch_stepw_dual(&s->dm_ad, &s->P, &s->E, &io, &none, mode, use_pd, nd, s->jac_scratch, (cudaStream_t)stream);
    if (rc) { set_err(std::string("jacobian launch: ") + cudaGetErrorString((cudaError_t)rc)); return rc; }
  }
  return 0;
}

// ---- Jacobian-vector and vector-Jacobian products of one step (same instance, same rows and columns as the dense Jacobian,
// without the PD-gain columns).  Blocks: q [n_q], qd [n_qd], tau [n_tau] or action [n_act]; every array fp64 [dim][n_stride].
static int dual_check(tds_b200_sim* s, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                      const char* what) {
  if (!s || !q || !qd || mode < 0 || mode > 3) { set_err(std::string(what) + ": bad argument"); return -1; }
  if (mode == 3) { set_err(std::string(what) + ": modes FD, NOCONTACT, FULL"); return -2; }
  if (use_pd && s->E.n_act == 0) { set_err("use_pd without tds_b200_set_env"); return -3; }
  if (use_pd && !tau_or_action) { set_err(std::string(what) + ": use_pd needs the actions"); return -1; }
  return 0;
}

int tds_b200_step_jvp_device(tds_b200_sim* s, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                             const double* t_q, const double* t_qd, const double* t_tau, double* t_out, void* stream) {
  int rc = dual_check(s, mode, use_pd, q, qd, tau_or_action, "step_jvp");
  if (rc) return rc;
  if (!t_out || (t_tau && !tau_or_action)) { set_err("step_jvp: bad argument"); return -1; }
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.q_in = q; io.qd_in = qd; io.tau_in = tau_or_action;
  io.n = s->n; io.n_stride = s->ns;
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  dio.jvp_tan[0] = t_q; dio.jvp_tan[1] = t_qd; dio.jvp_tan[2] = t_tau; dio.jvp_out = t_out;
  int chunk;
  if ((rc = ensure_dual_scratch(s, 1, &chunk))) return rc;
  rc = tds_launch_stepw_dual(&s->dm_ad, &s->P, &s->E, &io, &dio, mode, use_pd, 1, s->jac_scratch, (cudaStream_t)stream);
  if (rc) { set_err(std::string("jvp launch: ") + cudaGetErrorString((cudaError_t)rc)); return rc; }
  return 0;
}

int tds_b200_step_vjp_device(tds_b200_sim* s, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                             const double* g_out, double* g_q, double* g_qd, double* g_tau, void* stream) {
  int rc = dual_check(s, mode, use_pd, q, qd, tau_or_action, "step_vjp");
  if (rc) return rc;
  if (!g_out || (g_tau && !tau_or_action)) { set_err("step_vjp: bad argument"); return -1; }
  const DevModel& M = s->dm[0];
  const int n_in = use_pd ? s->E.n_act : s->n_tau;
  const int first[3] = {0, M.n_q, M.n_q + M.n_qd}, count[3] = {M.n_q, M.n_qd, n_in};
  double* const grad[3] = {g_q, g_qd, g_tau};
  int dirs = 0;   // only the requested blocks are launched
  for (int b = 0; b < 3; ++b) if (grad[b] && count[b] > dirs) dirs = count[b];
  if (dirs == 0) return 0;
  StepIO io;
  memset(&io, 0, sizeof(io));
  io.q_in = q; io.qd_in = qd; io.tau_in = tau_or_action;
  io.n = s->n; io.n_stride = s->ns;
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  dio.vjp_cot = g_out;
  for (int b = 0; b < 3; ++b) dio.vjp_out[b] = grad[b];
  int chunk;
  if ((rc = ensure_dual_scratch(s, dirs, &chunk))) return rc;
  for (int b = 0; b < 3; ++b) {
    if (!grad[b]) continue;
    for (int d0 = 0; d0 < count[b]; d0 += chunk) {
      io.jac_dir0 = first[b] + d0;
      const int nd = count[b] - d0 < chunk ? count[b] - d0 : chunk;
      rc = tds_launch_stepw_dual(&s->dm_ad, &s->P, &s->E, &io, &dio, mode, use_pd, nd, s->jac_scratch, (cudaStream_t)stream);
      if (rc) { set_err(std::string("vjp launch: ") + cudaGetErrorString((cudaError_t)rc)); return rc; }
    }
  }
  return 0;
}

int tds_b200_step_jacobian_host(tds_b200_sim* s, int mode, int use_pd, const double* q, const double* qd,
                                const double* tau_or_action, double* jac) {
  if (!s || !q || !qd || !jac) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const DevModel& M = s->dm[0];
  const int n = s->n, ns = s->ns;
  int dims[2];
  tds_b200_jacobian_dims(s, mode, use_pd, dims);
  const int n_in = use_pd ? s->E.n_act : s->n_tau;
  const size_t maxdim = (size_t)(M.n_q > M.n_qd ? M.n_q : M.n_qd) + 1;
  int rc = ensure_stage(s, sizeof(double) * n * maxdim, 0);
  if (rc) return rc;
  const size_t jb = sizeof(double) * (size_t)dims[0] * dims[1] * ns;
  if (jb > s->jac_dev_bytes) {
    if (s->jac_dev) cudaFree(s->jac_dev);
    s->jac_dev = nullptr; s->jac_dev_bytes = 0;
    CUDA_TRY(cudaMalloc((void**)&s->jac_dev, jb));
    s->jac_dev_bytes = jb;
  }
  double* st = (double*)s->stage_dev;
  const int T = 128, B = (n + T - 1) / T;
  cudaStream_t sm = s->stream;
  auto up = [&](const double* src, int dim, float* dst) -> int {
    if (dim == 0) return 0;
    CUDA_TRY(cudaMemcpyAsync(st, src, sizeof(double) * n * dim, cudaMemcpyHostToDevice, sm));
    aos_to_soa_kernel<double><<<B, T, 0, sm>>>(st, dim, 0, dst, dim, n, ns);
    return 0;
  };
  if ((rc = up(q, M.n_q, s->q))) return rc;
  if ((rc = up(qd, M.n_qd, s->qd))) return rc;
  if (tau_or_action) { if ((rc = up(tau_or_action, n_in, s->act))) return rc; }
  else CUDA_TRY(cudaMemsetAsync(s->act, 0, sizeof(float) * ns * (n_in > 0 ? n_in : 1), sm));
  CUDA_TRY(cudaMemsetAsync(s->jac_dev, 0, jb, sm));
  rc = tds_b200_step_jacobian_device(s, mode, use_pd, s->q, s->qd, s->act, s->jac_dev, sm);
  if (rc) return rc;
  std::vector<double> tmp((size_t)dims[0] * dims[1] * ns);
  CUDA_TRY(cudaMemcpyAsync(tmp.data(), s->jac_dev, jb, cudaMemcpyDeviceToHost, sm));
  CUDA_TRY(cudaStreamSynchronize(sm));
  CUDA_TRY(cudaGetLastError());
  const size_t rc_n = (size_t)dims[0] * dims[1];
  for (int e = 0; e < n; ++e)
    for (size_t k = 0; k < rc_n; ++k) jac[(size_t)e * rc_n + k] = tmp[k * ns + e];
  return 0;
}

int tds_b200_step_host(tds_b200_sim* s, int mode, int use_pd, const double* q, const double* qd,
                       const double* tau_or_action, double* q_out, double* qd_out, double* qdd_out,
                       double* contact_dist) {
  if (!s || !q || !qd) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const DevModel& M = s->dm[0];
  const int n = s->n, ns = s->ns;
  const int n_in = use_pd ? s->E.n_act : s->n_tau;
  const size_t maxdim = (size_t)(M.n_q > M.n_qd ? M.n_q : M.n_qd) + s->n_points + 1;
  int rc = ensure_stage(s, sizeof(double) * n * maxdim, 0);
  if (rc) return rc;
  double* st = (double*)s->stage_dev;
  const int T = 128, B = (n + T - 1) / T;
  cudaStream_t sm = s->stream;
  auto up = [&](const double* src, int dim, float* dst) -> int {
    if (dim == 0) return 0;
    CUDA_TRY(cudaMemcpyAsync(st, src, sizeof(double) * n * dim, cudaMemcpyHostToDevice, sm));
    aos_to_soa_kernel<double><<<B, T, 0, sm>>>(st, dim, 0, dst, dim, n, ns);
    return 0;
  };
  if ((rc = up(q, M.n_q, s->q))) return rc;
  if ((rc = up(qd, M.n_qd, s->qd))) return rc;
  if (tau_or_action) { if ((rc = up(tau_or_action, n_in, s->act))) return rc; }
  else CUDA_TRY(cudaMemsetAsync(s->act, 0, sizeof(float) * ns * (n_in > 0 ? n_in : 1), sm));
  rc = tds_b200_step_device(s, mode, use_pd, s->q, s->qd, s->act, s->q, s->qd, s->qdd, nullptr, nullptr,
                            contact_dist ? s->cdist : nullptr, nullptr, sm);
  if (rc) return rc;
  auto down = [&](const float* src, int dim, double* dst) -> int {
    if (dim == 0 || !dst) return 0;
    soa_to_aos_kernel<double><<<B, T, 0, sm>>>(src, st, dim, 0, dim, n, ns);
    CUDA_TRY(cudaMemcpyAsync(dst, st, sizeof(double) * n * dim, cudaMemcpyDeviceToHost, sm));
    CUDA_TRY(cudaStreamSynchronize(sm));
    return 0;
  };
  if ((rc = down(s->q, M.n_q, q_out))) return rc;
  if ((rc = down(s->qd, M.n_qd, qd_out))) return rc;
  if (mode == TDS_B200_MODE_FD && (rc = down(s->qdd, M.n_qd, qdd_out))) return rc;
  if ((rc = down(s->cdist, s->n_points, contact_dist))) return rc;
  CUDA_TRY(cudaStreamSynchronize(sm));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static IntegrateTable integrate_table(const tds_b200_sim* s) {
  const DevModel& M = s->dm[0];
  IntegrateTable T;
  memset(&T, 0, sizeof(T));
  T.n_links = M.n_links; T.floating = M.floating; T.n_q = M.n_q; T.n_qd = M.n_qd;
  for (int i = 0; i < M.n_links; ++i) {
    T.fixed[i] = (M.flags[i] & TDS_LF_FIXED) ? 1 : 0;
    T.q_idx[i] = (signed char)(T.fixed[i] ? 0 : M.q_idx[i]); T.qd_idx[i] = (signed char)(T.fixed[i] ? 0 : M.qd_idx[i]);
  }
  return T;
}

int tds_b200_integrate_euler_device(tds_b200_sim* s, float* q, float* qd, const float* qdd, void* stream) {
  if (!s || !q || !qd) return -1;
  if (s->dm[0].n_sph) { set_err("stand-alone integrate_euler: spherical joints are integrated by the step kernel only"); return -3; }
  const int T = 128, B = (s->n + T - 1) / T;
  integrate_euler_kernel<<<B, T, 0, (cudaStream_t)stream>>>(q, qd, qdd, s->P.dt, integrate_table(s), 1, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_integrate_euler_qdd_device(tds_b200_sim* s, float* qd, const float* qdd, void* stream) {
  if (!s || !qd || !qdd) return -1;
  const int T = 128, B = (s->n + T - 1) / T;
  integrate_euler_kernel<<<B, T, 0, (cudaStream_t)stream>>>(qd, qd, qdd, s->P.dt, integrate_table(s), 0, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static int write_tuples(const ContactCandTable& T, int* tuples, int cap) {
  for (int c = 0; c < T.n_points && c < cap && tuples; ++c) {
    tuples[4 * c + 0] = T.body_a[c]; tuples[4 * c + 1] = T.link_a[c];
    tuples[4 * c + 2] = T.body_b[c]; tuples[4 * c + 3] = T.link_b[c];
  }
  return T.n_points;
}

static int write_tuples6(const ContactCandTable& T, int* tuples, int cap) {
  for (int c = 0; c < T.n_points && c < cap && tuples; ++c) {
    tuples[6 * c + 0] = T.body_a[c]; tuples[6 * c + 1] = T.link_a[c]; tuples[6 * c + 2] = T.geom_a[c];
    tuples[6 * c + 3] = T.body_b[c]; tuples[6 * c + 4] = T.link_b[c]; tuples[6 * c + 5] = T.geom_b[c];
  }
  return T.n_points;
}

// (mb_a, link_a, geom_a, mb_b, link_b, geom_b) per candidate: the loop indices i, ii, iii, j, jj, jjj of
// World::compute_contacts_multi_body_internal (src/world.hpp:212-240) at which the point is emitted.
int tds_b200_model_contact_tuples(const double* model, int n_model, int* tuples, int cap) {
  if (!model) { set_err("null model"); return -1; }
  DevModel* D = new DevModel;
  const int rc = tds_build_dev_model(model, n_model, D);
  ContactCandTable T;
  if (rc == 0) T = make_cand_table(*D);
  delete D;
  if (rc) { set_err(std::string("unsupported model: ") + tds_model_error(rc)); return rc; }
  return write_tuples6(T, tuples, cap);
}

int tds_b200_contact_tuples(const tds_b200_sim* s, int* tuples, int cap) {
  if (!s) return -1;
  return write_tuples6(s->cand, tuples, cap);
}

// Host-only variant (no GPU needed): the candidate list of a flat model.
int tds_b200_model_contact_pairs(const double* model, int n_model, int* tuples, int cap) {
  if (!model) { set_err("null model"); return -1; }
  DevModel* D = new DevModel;
  const int rc = tds_build_dev_model(model, n_model, D);
  ContactCandTable T;
  if (rc == 0) T = make_cand_table(*D);
  delete D;
  if (rc) { set_err(std::string("unsupported model: ") + tds_model_error(rc)); return rc; }
  return write_tuples(T, tuples, cap);
}

int tds_b200_contact_pairs(const tds_b200_sim* s, int* tuples, int cap) {
  if (!s) return -1;
  return write_tuples(s->cand, tuples, cap);
}

int tds_b200_contact_list_device(tds_b200_sim* s, const float* contact_dist, int* count, int* links, void* stream) {
  if (!s || !contact_dist || !count || !links) return -1;
  if (s->cand.n_points == 0) return 0;
  const int T = 128, B = (s->n + T - 1) / T;
  contact_list_kernel<<<B, T, 0, (cudaStream_t)stream>>>(contact_dist, s->cand, s->P.keep_all_points, count, links, nullptr, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_contact_list_host(tds_b200_sim* s, int* count, int* links) {
  if (!s || !count) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const int n = s->n, ns = s->ns, np = s->cand.n_points;
  if (np == 0) { for (int e = 0; e < n; ++e) count[e] = 0; return 0; }
  if (!s->c_count) {
    CUDA_TRY(cudaMalloc((void**)&s->c_count, sizeof(int) * ns));
    CUDA_TRY(cudaMalloc((void**)&s->c_links, sizeof(int) * (size_t)ns * 2 * np));
  }
  int rc = tds_b200_contact_list_device(s, s->cdist, s->c_count, s->c_links, s->stream);
  if (rc) return rc;
  std::vector<int> tmp((size_t)ns * 2 * np);
  CUDA_TRY(cudaMemcpyAsync(count, s->c_count, sizeof(int) * n, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(tmp.data(), s->c_links, sizeof(int) * tmp.size(), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (links)
    for (int e = 0; e < n; ++e)
      for (int k = 0; k < 2 * np; ++k) links[(size_t)e * 2 * np + k] = tmp[(size_t)k * ns + e];
  return 0;
}

int tds_b200_contact_list_candidates_host(tds_b200_sim* s, int* count, int* cand) {
  if (!s || !count || !cand) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const int n = s->n, ns = s->ns, np = s->cand.n_points;
  if (np == 0) { for (int e = 0; e < n; ++e) count[e] = 0; return 0; }
  if (!s->c_count) {
    CUDA_TRY(cudaMalloc((void**)&s->c_count, sizeof(int) * ns));
    CUDA_TRY(cudaMalloc((void**)&s->c_links, sizeof(int) * (size_t)ns * 2 * np));
  }
  if (!s->c_cand) CUDA_TRY(cudaMalloc((void**)&s->c_cand, sizeof(int) * (size_t)ns * np));
  const int T = 128, B = (n + T - 1) / T;
  contact_list_kernel<<<B, T, 0, s->stream>>>(s->cdist, s->cand, s->P.keep_all_points, s->c_count, s->c_links, s->c_cand, n, ns);
  CUDA_TRY(cudaGetLastError());
  std::vector<int> tmp((size_t)ns * np);
  CUDA_TRY(cudaMemcpyAsync(count, s->c_count, sizeof(int) * n, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(tmp.data(), s->c_cand, sizeof(int) * tmp.size(), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  for (int e = 0; e < n; ++e)
    for (int k = 0; k < np; ++k) cand[(size_t)e * np + k] = tmp[(size_t)k * ns + e];
  return 0;
}

int tds_b200_env_set_state_host(tds_b200_sim* s, const double* q, const double* qd) {
  if (!s) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const DevModel& M = s->dm[0];
  const int n = s->n, ns = s->ns;
  int rc = ensure_stage(s, sizeof(double) * n * (size_t)(M.n_q + M.n_qd), 0);
  if (rc) return rc;
  double* st = (double*)s->stage_dev;
  const int T = 128, B = (n + T - 1) / T;
  CUDA_TRY(cudaMemcpyAsync(st, q, sizeof(double) * n * M.n_q, cudaMemcpyHostToDevice, s->stream));
  aos_to_soa_kernel<double><<<B, T, 0, s->stream>>>(st, M.n_q, 0, s->q, M.n_q, n, ns);
  double* st2 = st + (size_t)n * M.n_q;
  CUDA_TRY(cudaMemcpyAsync(st2, qd, sizeof(double) * n * M.n_qd, cudaMemcpyHostToDevice, s->stream));
  aos_to_soa_kernel<double><<<B, T, 0, s->stream>>>(st2, M.n_qd, 0, s->qd, M.n_qd, n, ns);
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

int tds_b200_env_get_state_host(tds_b200_sim* s, double* q, double* qd) {
  if (!s) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const DevModel& M = s->dm[0];
  const int n = s->n, ns = s->ns;
  int rc = ensure_stage(s, sizeof(double) * n * (size_t)(M.n_q + M.n_qd), 0);
  if (rc) return rc;
  double* st = (double*)s->stage_dev;
  const int T = 128, B = (n + T - 1) / T;
  soa_to_aos_kernel<double><<<B, T, 0, s->stream>>>(s->q, st, M.n_q, 0, M.n_q, n, ns);
  soa_to_aos_kernel<double><<<B, T, 0, s->stream>>>(s->qd, st + (size_t)n * M.n_q, M.n_qd, 0, M.n_qd, n, ns);
  if (q) CUDA_TRY(cudaMemcpyAsync(q, st, sizeof(double) * n * M.n_q, cudaMemcpyDeviceToHost, s->stream));
  if (qd) CUDA_TRY(cudaMemcpyAsync(qd, st + (size_t)n * M.n_q, sizeof(double) * n * M.n_qd, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

int tds_b200_env_step_device(tds_b200_sim* s, const float* actions, float* reward, float* done, void* stream) {
  if (!s) return -1;
  return tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, actions, s->q, s->qd, nullptr, reward, done,
                              nullptr, nullptr, stream);
}

int tds_b200_num_visuals(const tds_b200_sim* s) { return s ? s->vis.n_vis : -1; }

int tds_b200_env_step_visual_device(tds_b200_sim* s, const float* actions, float* reward, float* done, float* positions,
                                    float* orientations, void* stream) {
  if (!s || !positions || !orientations) return -1;
  if (s->vis.n_vis <= 0) { set_err("model has no link visuals"); return -2; }
  int rc = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, actions, s->q, s->qd, nullptr, reward, done, nullptr,
                                s->link_xf, stream);
  if (rc) return rc;
  const int T = 128, B = (s->n + T - 1) / T;
  pack_visual_instances_kernel<<<dim3(B, s->vis.n_vis), T, 0, (cudaStream_t)stream>>>(s->vis, s->link_xf, (float4*)positions,
                                                                                     (float4*)orientations, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static int ensure_env_layer(tds_b200_sim* s) {
  if (s->rq) return 0;
  const DevModel& M = s->dm[0];
  const size_t ns = s->ns;
  CUDA_TRY(cudaMalloc((void**)&s->rq, sizeof(float) * ns * (M.n_q > 0 ? M.n_q : 1)));
  CUDA_TRY(cudaMalloc((void**)&s->rqd, sizeof(float) * ns * (M.n_qd > 0 ? M.n_qd : 1)));
  CUDA_TRY(cudaMalloc((void**)&s->zero_act, sizeof(float) * ns * TDS_MAX_ACT));
  CUDA_TRY(cudaMemset(s->zero_act, 0, sizeof(float) * ns * TDS_MAX_ACT));
  CUDA_TRY(cudaMalloc((void**)&s->pol_act, sizeof(float) * ns * TDS_MAX_ACT));
  CUDA_TRY(cudaMalloc((void**)&s->sticky, sizeof(float) * ns));
  CUDA_TRY(cudaMalloc((void**)&s->r_total, sizeof(float) * ns));
  CUDA_TRY(cudaMalloc((void**)&s->r_steps, sizeof(int) * ns));
  CUDA_TRY(cudaMalloc((void**)&s->act_qidx, sizeof(int) * TDS_MAX_ACT));
  return 0;
}

int tds_b200_env_reset_device(tds_b200_sim* s, const float* mask, const float* noise, float noise_amp, unsigned long long seed,
                              int settle_steps, void* stream) {
  if (!s) return -1;
  if (s->E.n_act == 0) { set_err("env reset without tds_b200_set_env"); return -3; }
  CUDA_TRY(cudaSetDevice(s->device));
  int rc = ensure_env_layer(s);
  if (rc) return rc;
  const DevModel& M = s->dm[0];
  cudaStream_t sm = stream ? (cudaStream_t)stream : s->stream;   // NULL: the simulator's own stream (as the host paths)
  if (!s->act_qidx_valid) {   // once per actuator map (synchronous: keeps the reset itself capturable into a CUDA graph)
    int qidx[TDS_MAX_ACT];
    for (int a = 0; a < s->E.n_act; ++a) qidx[a] = M.q_idx[s->E.act_link[a]];
    CUDA_TRY(cudaMemcpy(s->act_qidx, qidx, sizeof(int) * s->E.n_act, cudaMemcpyHostToDevice));
    s->act_qidx_valid = true;
  }
  const int T = 128, B = (s->n + T - 1) / T;
  env_reset_fill_kernel<<<B, T, 0, sm>>>(s->rq, s->rqd, noise, noise_amp, seed, s->E, M.n_q, M.n_qd, s->act_qidx, s->n, s->ns);
  // settle with zero actions on the staging copy (laikago_environment2.h:92-110); no auto-reset inside
  const int saved_auto = s->E.auto_reset;
  s->E.auto_reset = 0;
  for (int i = 0; i < settle_steps && rc == 0; ++i)
    rc = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->rq, s->rqd, s->zero_act, s->rq, s->rqd, nullptr, nullptr, nullptr,
                              nullptr, nullptr, sm);
  s->E.auto_reset = saved_auto;
  if (rc) return rc;
  env_select_kernel<<<B, T, 0, sm>>>(mask, s->rq, s->rqd, s->q, s->qd, M.n_q, M.n_qd, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_ars_perturb_device(tds_b200_sim* s, const float* w, const float* deltas, float scale, float* params, int n_params,
                                void* stream) {
  if (!s || !w || !deltas || !params || n_params <= 0) return -1;
  const int T = 128, B = (s->n + T - 1) / T;
  ars_perturb_kernel<<<dim3(B, n_params), T, 0, (cudaStream_t)stream>>>(w, deltas, scale, params, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_ars_update_device(tds_b200_sim* s, float* w, const float* deltas, const float* r_pos, const float* r_neg,
                               float delta_std, float step_size, int n_params, void* stream) {
  if (!s || !w || !deltas || !r_pos || !r_neg || n_params <= 0) return -1;
  ars_update_kernel<<<n_params, 256, 0, (cudaStream_t)stream>>>(w, deltas, r_pos, r_neg, delta_std, step_size, s->n, s->ns);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_env_set_obs_stats(tds_b200_sim* s, float* stats) {
  if (!s) return -1;
  s->obs_stats = stats;
  return 0;
}

int tds_b200_env_rollout_device(tds_b200_sim* s, const float* policy, int n_params, int rollout_length, float shift,
                                float* total_rewards, int* steps, void* stream) {
  if (!s || !policy || !total_rewards || !steps) return -1;
  if (s->E.n_act == 0) { set_err("rollout without tds_b200_set_env"); return -3; }
  const DevModel& M = s->dm[0];
  if (n_params != s->E.n_act * (M.n_q + M.n_qd) + s->E.n_act) { set_err("policy size must be n_act * (n_q + n_qd) + n_act"); return -2; }
  CUDA_TRY(cudaSetDevice(s->device));
  int rc = ensure_env_layer(s);
  if (rc) return rc;
  cudaStream_t sm = stream ? (cudaStream_t)stream : s->stream;
  const int T = 128, B = (s->n + T - 1) / T;
  rollout_init_kernel<<<B, T, 0, sm>>>(s->sticky, total_rewards, steps, s->n);
  const int saved_auto = s->E.auto_reset;
  s->E.auto_reset = 0;   // an episode ends at done (ars_vectorized_worker.h:121-133)
  for (int r = 0; r < rollout_length && rc == 0; ++r) {
    policy_linear_kernel<<<dim3(B, s->E.n_act), T, 0, sm>>>(s->q, s->qd, policy, s->pol_act, M.n_q, M.n_qd, s->E.n_act, s->n, s->ns);
    if (s->obs_stats) obs_stat_push_kernel<<<dim3(B, M.n_q + M.n_qd), T, 0, sm>>>(s->q, s->qd, s->obs_stats, M.n_q, M.n_qd, s->n, s->ns);
    rc = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, s->pol_act, s->q, s->qd, nullptr, s->reward, s->done, nullptr,
                              nullptr, sm);
    rollout_accum_kernel<<<B, T, 0, sm>>>(s->reward, s->done, shift, s->sticky, total_rewards, steps, s->n);
  }
  s->E.auto_reset = saved_auto;
  if (rc) return rc;
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_env_rollout_host(tds_b200_sim* s, const double* policy, int n_params, int rollout_length, double shift,
                              const double* noise, double noise_amp, unsigned long long seed, int settle_steps,
                              double* total_rewards, int* steps) {
  if (!s || !policy) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  int rc = ensure_env_layer(s);
  if (rc) return rc;
  const int n = s->n, ns = s->ns, na = s->E.n_act;
  cudaStream_t sm = s->stream;
  const int T = 128, B = (n + T - 1) / T;
  const size_t rows = (size_t)n_params > (size_t)na ? (size_t)n_params : (size_t)na;
  if (rows > s->pol_params_rows) {
    cudaFree(s->pol_params); s->pol_params = nullptr; s->pol_params_rows = 0;
    CUDA_TRY(cudaMalloc((void**)&s->pol_params, sizeof(float) * rows * ns));
    s->pol_params_rows = rows;
  }
  rc = ensure_stage(s, sizeof(double) * (size_t)n * rows, 0);
  if (rc) return rc;
  double* st = (double*)s->stage_dev;
  const float* d_noise = nullptr;
  if (noise) {   // [n][n_act] -> [n_act][ns]
    CUDA_TRY(cudaMemcpyAsync(st, noise, sizeof(double) * n * na, cudaMemcpyHostToDevice, sm));
    aos_to_soa_kernel<double><<<B, T, 0, sm>>>(st, na, 0, s->pol_params, na, n, ns);
    d_noise = s->pol_params;
  }
  rc = tds_b200_env_reset_device(s, nullptr, d_noise, (float)noise_amp, seed, settle_steps, sm);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(st, policy, sizeof(double) * n * n_params, cudaMemcpyHostToDevice, sm));
  aos_to_soa_kernel<double><<<B, T, 0, sm>>>(st, n_params, 0, s->pol_params, n_params, n, ns);
  rc = tds_b200_env_rollout_device(s, s->pol_params, n_params, rollout_length, (float)shift, s->r_total, s->r_steps, sm);
  if (rc) return rc;
  std::vector<float> tot(n);
  CUDA_TRY(cudaMemcpyAsync(tot.data(), s->r_total, sizeof(float) * n, cudaMemcpyDeviceToHost, sm));
  if (steps) CUDA_TRY(cudaMemcpyAsync(steps, s->r_steps, sizeof(int) * n, cudaMemcpyDeviceToHost, sm));
  CUDA_TRY(cudaStreamSynchronize(sm));
  if (total_rewards) for (int i = 0; i < n; ++i) total_rewards[i] = (double)tot[i];
  return 0;
}

// Profiling aid (not part of the drop-in surface): enable per-warp clock64() stamps at the phase
// boundaries of the step kernel; out (host) receives [n_warps][16] stamps of the last step.
int tds_b200_get_precision(const tds_b200_sim* s) { return s ? s->precision : -1; }

const char* tds_b200_kernel_name(const tds_b200_sim* s) {
  static const char* names[5] = {"", "tds_stepw_kernel (common frame, lane per environment)",
                                 "tds_stept_kernel (lane team per environment)", "tds_stepr_kernel (warp per tree role)",
                                 "tds_step_spec_kernel (warp per tree role, model-specialised)"};
  return (s && s->kernel >= 0 && s->kernel <= 4) ? names[s->kernel] : "";
}

int tds_b200_debug_phase_clocks(tds_b200_sim* s, int enable, long long* out_host, int cap_warps) {
  if (!s) return -1;
  const int nw = s->ns / (32 / TDS_TEAM_T);   // team kernel: 8 environments per warp
  if (enable && !s->phase_clk) {
    CUDA_TRY(cudaMalloc((void**)&s->phase_clk, sizeof(long long) * 16 * nw));
    CUDA_TRY(cudaMemset(s->phase_clk, 0, sizeof(long long) * 16 * nw));
  }
  if (out_host && s->phase_clk) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out_host, s->phase_clk, sizeof(long long) * 16 * (nw < cap_warps ? nw : cap_warps), cudaMemcpyDeviceToHost));
  }
  if (!enable && s->phase_clk) { cudaFree(s->phase_clk); s->phase_clk = nullptr; }
  return nw;
}

void* tds_b200_stream(tds_b200_sim* s) { return s ? (void*)s->stream : nullptr; }
float* tds_b200_env_q(tds_b200_sim* s) { return s ? s->q : nullptr; }
float* tds_b200_env_qd(tds_b200_sim* s) { return s ? s->qd : nullptr; }

int tds_b200_env_step_host(tds_b200_sim* s, const float* actions, float* obs, float* rewards, float* dones) {
  if (!s || !actions) return -1;
  CUDA_TRY(cudaSetDevice(s->device));
  const DevModel& M = s->dm[0];
  const int n = s->n, ns = s->ns, na = s->E.n_act, nobs = M.n_q + M.n_qd;
  // device staging: actions AoS in | obs AoS out | reward | done
  const size_t in_b = sizeof(float) * (size_t)n * na, obs_b = sizeof(float) * (size_t)n * nobs;
  // obs | rewards | dones adjacent in the caller's memory: pack them on the device and copy once
  const bool packed = obs && rewards == obs + (size_t)n * nobs && dones == rewards + n;
  int rc = ensure_stage(s, in_b + obs_b + sizeof(float) * 2 * (size_t)n, 0);
  if (rc) return rc;
  float* d_in = (float*)s->stage_dev;
  float* d_obs = (float*)((char*)s->stage_dev + in_b);
  cudaStream_t sm = s->stream;
  const int T = 128, B = (n + T - 1) / T;
  // the specialised kernel reads environment-major actions and writes the observation block itself
  const bool direct = s->kernel_req == 4 && s->spec_ok && s->P.contact_model == 0 && tds_spec_smem_bytes(s->spec_idx, s->precision) <= (size_t)s->max_smem_optin;
  auto enqueue = [&]() -> int {
    CUDA_TRY(cudaMemcpyAsync(d_in, actions, in_b, cudaMemcpyHostToDevice, sm));
    if (direct) {
      s->io_act_aos = d_in; s->io_obs_aos = obs ? d_obs : nullptr; s->io_obs_tail = (obs && packed) ? d_obs + (size_t)n * nobs : nullptr;
    } else aos_to_soa_kernel<float><<<B, T, 0, sm>>>(d_in, na, 0, s->act, na, n, ns);
    int r = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, s->act, s->q, s->qd, nullptr, s->reward, s->done,
                                 nullptr, nullptr, sm);
    s->io_act_aos = nullptr; s->io_obs_aos = nullptr; s->io_obs_tail = nullptr;
    if (r) return r;
    if (obs && direct) {
      CUDA_TRY(cudaMemcpyAsync(obs, d_obs, obs_b + (packed ? sizeof(float) * 2 * (size_t)n : 0), cudaMemcpyDeviceToHost, sm));
    } else if (obs) {
      pack_env_out_kernel<<<B, T, 0, sm>>>(s->q, s->qd, s->reward, s->done, d_obs, M.n_q, M.n_qd, n, ns, packed ? 1 : 0);
      CUDA_TRY(cudaMemcpyAsync(obs, d_obs, obs_b + (packed ? sizeof(float) * 2 * (size_t)n : 0), cudaMemcpyDeviceToHost, sm));
    }
    if (!packed) {
      if (rewards) CUDA_TRY(cudaMemcpyAsync(rewards, s->reward, sizeof(float) * n, cudaMemcpyDeviceToHost, sm));
      if (dones) CUDA_TRY(cudaMemcpyAsync(dones, s->done, sizeof(float) * n, cudaMemcpyDeviceToHost, sm));
    }
    return 0;
  };
  // Zero-copy: pinned (mapped) caller buffers and the specialised kernel -> the step kernel itself reads the actions
  // from host memory and writes observations / rewards / dones there (coalesced, staged through shared memory): one
  // launch, no staging copies.
  static const bool no_zero_copy = getenv("TDS_B200_NO_ZEROCOPY") != nullptr;
  if (direct && !s->phase_clk && !no_zero_copy) {
    void *da = nullptr, *dob = nullptr, *dr = nullptr, *dd = nullptr;
    bool ok;
    if ((++s->zc_calls & 63u) != 0 && s->zc_key[0] == actions && s->zc_key[1] == obs && s->zc_key[2] == rewards && s->zc_key[3] == dones) {
      ok = s->zc_ok;   // same buffers as the last call: the pointer queries (a microsecond each) are cached
      da = s->zc_dev[0]; dob = s->zc_dev[1]; dr = s->zc_dev[2]; dd = s->zc_dev[3];
    } else {
      ok = is_pinned(actions) && is_pinned(obs) && is_pinned(rewards) && is_pinned(dones);
      ok = ok && cudaHostGetDevicePointer(&da, (void*)actions, 0) == cudaSuccess;
      if (ok && obs) ok = cudaHostGetDevicePointer(&dob, obs, 0) == cudaSuccess;
      if (ok && rewards) ok = cudaHostGetDevicePointer(&dr, rewards, 0) == cudaSuccess;
      if (ok && dones) ok = cudaHostGetDevicePointer(&dd, dones, 0) == cudaSuccess;
      if (!ok) cudaGetLastError();
      s->zc_key[0] = actions; s->zc_key[1] = obs; s->zc_key[2] = rewards; s->zc_key[3] = dones;
      s->zc_dev[0] = da; s->zc_dev[1] = dob; s->zc_dev[2] = dr; s->zc_dev[3] = dd;
      s->zc_ok = ok;
    }
    if (ok) {
      s->io_act_aos = (const float*)da; s->io_obs_aos = (float*)dob; s->io_obs_tail = nullptr;
      rc = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, s->act, s->q, s->qd, nullptr, dr ? (float*)dr : s->reward,
                                dd ? (float*)dd : s->done, nullptr, nullptr, sm);
      s->io_act_aos = nullptr; s->io_obs_aos = nullptr;
      if (rc) return rc;
      CUDA_TRY(cudaStreamSynchronize(sm));
      CUDA_TRY(cudaGetLastError());
      return 0;
    }
  }
  const void* key[4] = {actions, obs, rewards, dones};
  const bool same = s->g_key[0] == key[0] && s->g_key[1] == key[1] && s->g_key[2] == key[2] && s->g_key[3] == key[3];
  // the role-warp kernel reads its link table from ONE constant symbol per device: if another simulator took the symbol over
  // since the capture, the captured launch would run on that simulator's table - drop the graph, the eager path re-uploads
  if (s->g_exec && s->kernel == 3 && tds_stepr_table_owner(s->device) != s->table_token) drop_host_graph(s);
  if (same && s->g_exec) {
    CUDA_TRY(cudaGraphLaunch(s->g_exec, sm));
  } else if (same && s->g_seen >= 2 && !s->phase_clk && is_pinned(actions) && is_pinned(obs) && is_pinned(rewards) && is_pinned(dones)) {
    // third call with the same pinned buffers (the first two ran eagerly: lazy kernel attributes are set): capture
    cudaGraph_t g = nullptr;
    CUDA_TRY(cudaStreamBeginCapture(sm, cudaStreamCaptureModeThreadLocal));
    rc = enqueue();
    cudaError_t ce = cudaStreamEndCapture(sm, &g);
    if (rc || ce != cudaSuccess) {
      if (g) cudaGraphDestroy(g);
      cudaGetLastError();
      s->g_seen = -1000000;   // do not try again for this buffer set
      rc = enqueue();
      if (rc) return rc;
    } else {
      ce = cudaGraphInstantiate(&s->g_exec, g, 0);
      cudaGraphDestroy(g);
      if (ce != cudaSuccess) { s->g_exec = nullptr; set_err(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce)); return (int)ce; }
      CUDA_TRY(cudaGraphLaunch(s->g_exec, sm));
    }
  } else {
    if (!same) { drop_host_graph(s); for (int k = 0; k < 4; ++k) s->g_key[k] = key[k]; }
    ++s->g_seen;
    rc = enqueue();
    if (rc) return rc;
  }
  CUDA_TRY(cudaStreamSynchronize(sm));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- C-ABI v1 drop-in (src/utils/cuda_codegen.hpp:156-266) for the models ars_train_policy_cuda loads by name
// "cuda_model_" + env_name() (examples/ars/ars_train_policy_cuda.cpp:507): cuda_model_laikago and cuda_model_ant -------
static const double k_laikago_model[] = {
#include "generated/laikago_model.inc"
};
static const double k_ant_model[] = {
#include "generated/ant_model.inc"
};
struct V1Spec {
  const char* name;
  const double* model; int n_model;
  int in_dim, out_dim, written;       // written = n_q + n_qd + 7 * n_visuals + 1 (the rest of output_dim is never written)
  int n_q, n_act;
  double dt, init[TDS_MAX_ACT], kp, kd, max_force;
  int reward_kind;
};
// LaikagoContactSimulation: laikago_environment2.h:36-61, locomotion_contact_simulation.h:131-135 (51 -> 411)
static const V1Spec k_v1_laikago = {"cuda_model_laikago", k_laikago_model, (int)(sizeof(k_laikago_model) / sizeof(double)), 51, 411, 156, 18, 12,
                                    1e-3, {0.2, 0, -0.7, 0.2, 0, -0.7, 0.2, 0, -0.7, 0.2, 0, -0.7}, 100.0, 2.0, 50.0, 1};
// AntContactSimulation2: ant_environment2.h:28-70 (39 = q14|qd14|action8|kp,kd,max_force -> 155 = 28 + 14 links x 9 visuals + 1)
static const V1Spec k_v1_ant = {"cuda_model_ant", k_ant_model, (int)(sizeof(k_ant_model) / sizeof(double)), 39, 155, 92, 14, 8,
                                0.01, {0.0, -0.5, 0.0, -0.5, 0.0, -0.5, 0.0, -0.5}, 15.0, 0.3, 3.0, 3};
struct V1Instance {
  tds_b200_sim* sim = nullptr;
  double *dev_in = nullptr, *dev_out = nullptr;
  int n = 0;
  std::mutex mu;
};
static V1Instance g_v1_laikago, g_v1_ant;

static void v1_fail(const V1Spec& S, const char* what) {
  // the reference prints and exits on allocation failure (cuda_codegen.hpp:201-208)
  fprintf(stderr, "%s (tds_b200): %s: %s\n", S.name, what, g_err.c_str());
  exit(1);
}

static void v1_release(V1Instance& I) {
  if (I.sim) tds_b200_destroy(I.sim);
  I.sim = nullptr;
  cudaFree(I.dev_in); cudaFree(I.dev_out);
  I.dev_in = I.dev_out = nullptr;
  I.n = 0;
}

static void v1_allocate(V1Instance& I, const V1Spec& S, int num_total_threads) {
  std::lock_guard<std::mutex> lk(I.mu);
  v1_release(I);
  int dev = 0;
  cudaGetDevice(&dev);
  I.sim = tds_b200_create(S.model, S.n_model, num_total_threads, dev);
  if (!I.sim) v1_fail(S, "allocate");
  const double g[3] = {0, 0, -9.81};
  tds_b200_set_params(I.sim, S.dt, g, 1.0, 0.0, 0.2, 1e-5, 1, 1);
  tds_b200_set_env(I.sim, S.n_act, S.init, 6, S.kp, S.kd, S.max_force, 0.4, S.reward_kind);
  I.n = num_total_threads;
  if (cudaMalloc((void**)&I.dev_in, sizeof(double) * (size_t)num_total_threads * S.in_dim) != cudaSuccess ||
      cudaMalloc((void**)&I.dev_out, sizeof(double) * (size_t)num_total_threads * S.written) != cudaSuccess) {
    set_err("cudaMalloc failed");
    v1_fail(S, "allocate");
  }
}

static void v1_forward_zero(V1Instance& I, const V1Spec& S, int num_total_threads, double* output, const double* input) {
  std::lock_guard<std::mutex> lk(I.mu);
  if (!I.sim || num_total_threads > I.n) { set_err("forward_zero called before allocate (or with more threads)"); v1_fail(S, "forward_zero"); }
  tds_b200_sim* s = I.sim;
  const int n = num_total_threads, ns = s->ns;
  cudaStream_t sm = s->stream;
  const int T = 128, B = (n + T - 1) / T;
  const int saved_n = s->n;
  s->n = n;
  cudaMemcpyAsync(I.dev_in, input, sizeof(double) * (size_t)n * S.in_dim, cudaMemcpyHostToDevice, sm);
  aos_to_soa_kernel<double><<<B, T, 0, sm>>>(I.dev_in, S.in_dim, 0, s->q, S.n_q, n, ns);
  aos_to_soa_kernel<double><<<B, T, 0, sm>>>(I.dev_in, S.in_dim, S.n_q, s->qd, S.n_q, n, ns);
  aos_to_soa_kernel<double><<<B, T, 0, sm>>>(I.dev_in, S.in_dim, 2 * S.n_q, s->act, S.n_act, n, ns);
  // kp, kd, max_force travel in the input vector (locomotion_contact_simulation.h:164-166); the v1 ABI is
  // called with one value for the whole batch (ars_vectorized_environment.h:223-236): read env 0's.
  const int v0 = 2 * S.n_q + S.n_act;
  s->E.kp = (float)input[v0]; s->E.kd = (float)input[v0 + 1]; s->E.max_force = (float)input[v0 + 2];
  int rc = tds_b200_step_device(s, TDS_B200_MODE_FULL, 1, s->q, s->qd, s->act, s->q, s->qd, nullptr, nullptr, nullptr,
                                nullptr, s->link_xf, sm);
  if (rc) v1_fail(S, "step");
  pack_v1_output_kernel<<<B, T, 0, sm>>>(s->vis, s->q, s->qd, s->link_xf, I.dev_out, S.written, n, ns, s->dm[0].floating);
  // entries >= written are never written by the reference either (they keep the caller's values)
  cudaMemcpy2DAsync(output, sizeof(double) * S.out_dim, I.dev_out, sizeof(double) * S.written, sizeof(double) * S.written, n,
                    cudaMemcpyDeviceToHost, sm);
  cudaError_t e = cudaStreamSynchronize(sm);
  s->n = saved_n;
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); v1_fail(S, "forward_zero"); }
}

#define TDS_V1_SYMBOLS(model, inst, spec)                                                                              \
  CudaFunctionMetaData model##_forward_zero_meta(void) {                                                               \
    CudaFunctionMetaData d; d.output_dim = spec.out_dim; d.input_dim = spec.in_dim; d.global_dim = 0; return d;        \
  }                                                                                                                    \
  void model##_forward_zero_allocate(int num_total_threads) { v1_allocate(inst, spec, num_total_threads); }            \
  void model##_forward_zero_deallocate(void) { std::lock_guard<std::mutex> lk(inst.mu); v1_release(inst); }            \
  void model##_forward_zero(int num_total_threads, int num_blocks, int num_threads_per_block, double* output,          \
                            const double* input) {                                                                     \
    (void)num_blocks; (void)num_threads_per_block;                                                                     \
    v1_forward_zero(inst, spec, num_total_threads, output, input);                                                     \
  }
TDS_V1_SYMBOLS(cuda_model_laikago, g_v1_laikago, k_v1_laikago)
TDS_V1_SYMBOLS(cuda_model_ant, g_v1_ant, k_v1_ant)
static const int k_laikago_in = 51, k_laikago_out = 411;

// ---- C-ABI v2 (src/utils/cuda/cuda_codegen.hpp:32-231, loaded by tds::CudaLibrary / CudaModel / CudaFunction,
// src/utils/cuda/cuda_{library,model,function}.hpp): model_info + <model>_forward_zero{,_meta,_allocate,_deallocate,
// _send_local,_send_global}.  The model is exported as "b200_laikago" (the v1 symbols keep the name cuda_model_laikago:
// the two generations use the same symbol names with different meta structs, so they cannot share a model name).
// <model>_jacobian: b200_laikago_jacobian below (forward-mode dual numbers through the step kernel).
static std::vector<double> g_v2_local;   // thread-local inputs as last sent ([n][51], host)
static int g_v2_sent = 0;

void model_info(char const* const** names, int* count) {
  static const char* k_names[1] = {"b200_laikago"};
  *names = k_names;
  *count = 1;
}

CudaFunctionMetaDataV2 b200_laikago_forward_zero_meta(void) {
  CudaFunctionMetaDataV2 d;
  d.output_dim = k_laikago_out; d.local_input_dim = k_laikago_in; d.global_input_dim = 0; d.accumulated_output = false;
  return d;
}

void b200_laikago_forward_zero_allocate(int num_total_threads) {
  cuda_model_laikago_forward_zero_allocate(num_total_threads);
  g_v2_local.assign((size_t)num_total_threads * k_laikago_in, 0.0);
  g_v2_sent = 0;
}

void b200_laikago_forward_zero_deallocate(void) {
  cuda_model_laikago_forward_zero_deallocate();
  g_v2_local.clear(); g_v2_local.shrink_to_fit();
  g_v2_sent = 0;
}

bool b200_laikago_forward_zero_send_local(int num_total_threads, const double* input) {
  if (!input || (size_t)num_total_threads * k_laikago_in > g_v2_local.size()) {
    fprintf(stderr, "Error while sending thread-local input data to GPU: %d threads exceed the allocation.\n", num_total_threads);
    return false;
  }
  memcpy(g_v2_local.data(), input, sizeof(double) * (size_t)num_total_threads * k_laikago_in);
  g_v2_sent = num_total_threads;
  return true;
}

bool b200_laikago_forward_zero_send_global(const double* input) { (void)input; return true; }   // global_input_dim = 0

void b200_laikago_forward_zero(int num_total_threads, int num_blocks, int num_threads_per_block, double* output) {
  if (num_total_threads > g_v2_sent) { fprintf(stderr, "b200_laikago_forward_zero: launch before send_local\n"); exit(1); }
  cuda_model_laikago_forward_zero(num_total_threads, num_blocks, num_threads_per_block, output, g_v2_local.data());
}

// <model>_jacobian of the v2 generation (CudaModelSourceGen::jacobian_source, src/utils/cuda/cuda_codegen.hpp:303-426;
// loaded by tds::CudaModel as the function named "<model>_jacobian", src/utils/cuda/cuda_model.hpp:14-25): dense rows
// (output_i, input_i) in row-major order per thread.  Output sparsity (set_jac_output_sparsity, :283-288): the 36 state
// rows q' | qd' of the 411 outputs; all 51 local inputs (q | qd | action | kp, kd, max_force) as columns; no accumulation.
static V1Instance g_v2_jac;
static std::vector<double> g_v2_jac_local;
static int g_v2_jac_sent = 0;
static const int k_jac_rows = 36, k_jac_cols = 51;

CudaFunctionMetaDataV2 b200_laikago_jacobian_meta(void) {
  CudaFunctionMetaDataV2 d;
  d.output_dim = k_jac_rows * k_jac_cols; d.local_input_dim = k_laikago_in; d.global_input_dim = 0; d.accumulated_output = false;
  return d;
}
void b200_laikago_jacobian_allocate(int num_total_threads) {
  v1_allocate(g_v2_jac, k_v1_laikago, num_total_threads);
  g_v2_jac_local.assign((size_t)num_total_threads * k_laikago_in, 0.0);
  g_v2_jac_sent = 0;
}
void b200_laikago_jacobian_deallocate(void) {
  { std::lock_guard<std::mutex> lk(g_v2_jac.mu); v1_release(g_v2_jac); }
  g_v2_jac_local.clear(); g_v2_jac_local.shrink_to_fit();
  g_v2_jac_sent = 0;
}
bool b200_laikago_jacobian_send_local(int num_total_threads, const double* input) {
  if (!input || (size_t)num_total_threads * k_laikago_in > g_v2_jac_local.size()) {
    fprintf(stderr, "Error while sending thread-local input data to GPU: %d threads exceed the allocation.\n", num_total_threads);
    return false;
  }
  memcpy(g_v2_jac_local.data(), input, sizeof(double) * (size_t)num_total_threads * k_laikago_in);
  g_v2_jac_sent = num_total_threads;
  return true;
}
bool b200_laikago_jacobian_send_global(const double* input) { (void)input; return true; }
void b200_laikago_jacobian(int num_total_threads, int num_blocks, int num_threads_per_block, double* output) {
  (void)num_blocks; (void)num_threads_per_block;
  std::lock_guard<std::mutex> lk(g_v2_jac.mu);
  if (!g_v2_jac.sim || num_total_threads > g_v2_jac_sent) { fprintf(stderr, "b200_laikago_jacobian: launch before allocate / send_local\n"); exit(1); }
  tds_b200_sim* s = g_v2_jac.sim;
  const int n = num_total_threads;
  std::vector<double> q((size_t)n * 18), qd((size_t)n * 18), act((size_t)n * 12);
  for (int e = 0; e < n; ++e) {
    const double* x = g_v2_jac_local.data() + (size_t)e * k_laikago_in;
    memcpy(&q[(size_t)e * 18], x, 18 * sizeof(double)); memcpy(&qd[(size_t)e * 18], x + 18, 18 * sizeof(double));
    memcpy(&act[(size_t)e * 12], x + 36, 12 * sizeof(double));
  }
  s->E.kp = (float)g_v2_jac_local[48]; s->E.kd = (float)g_v2_jac_local[49]; s->E.max_force = (float)g_v2_jac_local[50];
  const int saved_n = s->n;
  s->n = n;
  const int rc = tds_b200_step_jacobian_host(s, TDS_B200_MODE_FULL, 1, q.data(), qd.data(), act.data(), output);
  s->n = saved_n;
  if (rc) { fprintf(stderr, "b200_laikago_jacobian: %s\n", g_err.c_str()); exit(1); }
}

}  // extern "C"
