/* C-ABI of libtds_b200.so: the B200-native batched rigid-body env-step.
 *
 * Plain pointers and sizes only (no torch / C++ types).  Each entry point cites the reference
 * interface it replaces (paths relative to erwincoumans/tiny-differentiable-simulator @ 8381b8c).
 * INTEGRATION.md shows the reference-side bindings (dlopen of the v1 symbols, a
 * CustomForwardDynamicsStepper subclass, a pybind shim).
 *
 * Device-side state is SoA fp32: array[dim][n_stride], environment index fastest
 * (n_stride = n_envs rounded up to 32), so a warp of 32 environments reads 128 contiguous bytes
 * per coordinate.
 */
#ifndef TDS_B200_H
#define TDS_B200_H
#ifndef __cplusplus
#include <stdbool.h>
#endif
#ifdef __cplusplus
extern "C" {
#endif

typedef struct tds_b200_sim tds_b200_sim;

/* pipeline selector of tds_b200_step_* */
#define TDS_B200_MODE_FD 0        /* tds::forward_dynamics only, src/dynamics/forward_dynamics.hpp:11 (qdd out) */
#define TDS_B200_MODE_NOCONTACT 1 /* FD -> integrate_euler, examples/environments/cartpole_environment2.h:86-93 */
#define TDS_B200_MODE_FULL 2      /* FD -> integrate_euler_qdd -> World::step -> integrate_euler,
                                     examples/environments/locomotion_contact_simulation.h:261-269 */

#define TDS_B200_MODE_WORLD 3     /* World::step(dt) alone, src/world.hpp:302-363: contact detection + constraint solve on the
                                     given (q, qd); qd out, q unchanged.  Stage of the fine-grained pytinydiffsim sequence
                                     forward_dynamics -> integrate_euler_qdd -> world.step -> integrate_euler
                                     (python/pytinydiffsim.inl:659-663,857-876) */

/* arithmetic selector */
#define TDS_B200_PREC_MIXED 0 /* default: fp32 ABA / factorisation / PGS; fp64 kinematics, contact geometry,
                                 composite inertias, CRBA products, Jacobians and LCP right-hand side */
#define TDS_B200_PREC_F64 1   /* strict: every stage fp64; meets 1e-5 on every model of the parity suite */
#define TDS_B200_PREC_F32 2   /* comparison only (the reference's own fp32 build misses the tolerance) */
#define TDS_B200_PREC_AUTO (-1) /* default: MIXED for a model the library holds a compiled, parity-validated instance of
                                   (Laikago, Ant), F64 otherwise */

const char* tds_b200_last_error(void);

/* ---- model compiler (setup time) -------------------------------------------------------------
 * Replaces UrdfCache::construct -> UrdfParser::load_urdf + UrdfToMultiBody::convert_to_multi_body
 * (src/urdf/urdf_cache.hpp:74-84, src/urdf/urdf_parser.hpp:707-925, src/urdf/urdf_to_multi_body.hpp:41).
 * urdf / plane_urdf: file path or URDF text (text if the first non-blank char is '<'); plane_urdf may
 * be NULL/"" for a world without ground plane.  Writes the flat model (include/tds_b200_model.h);
 * returns its length in doubles (call with out=NULL to size), <0 on error. */
int tds_b200_urdf_to_model(const char* urdf, const char* plane_urdf, int floating, double* out, int cap);

/* ---- simulator lifecycle ----------------------------------------------------------------------
 * One sim = n_envs independent copies of World{plane, MultiBody} (src/world.hpp:41, multi_body.hpp:13)
 * resident on CUDA device `device`.  Returns NULL on error (see tds_b200_last_error). */
tds_b200_sim* tds_b200_create(const double* model, int n_model_doubles, int n_envs, int device);
/* Host-only acceptance check of a flat model (no GPU needed): 0, or the negative code tds_b200_create would fail with
 * (mesh shapes against the plane, spherical joints with a stiffness, capacity); the reason is in tds_b200_last_error(). */
int tds_b200_validate_model(const double* model, int n_model);
void tds_b200_destroy(tds_b200_sim* sim);

/* World / solver parameters: World::{default_friction,default_restitution} (src/world.hpp:68-69),
 * gravity (world.hpp:50), MultiBodyConstraintSolver::{erp_,cfm_,pgs_iterations_,keep_all_points_}
 * (src/mb_constraint_solver.hpp:59-70).  Defaults equal the reference's. */
int tds_b200_set_params(tds_b200_sim* sim, double dt, const double gravity[3], double friction, double restitution,
                        double erp, double cfm, int pgs_iterations, int keep_all_points);

/* Contact law.  0 (default): the reference's impulse-level LCP solved by projected Gauss-Seidel
 * (MultiBodyConstraintSolver, src/mb_constraint_solver.hpp).  1: spring-damper contacts - the reference's
 * MultiBodyConstraintSolverSpring, whose SOURCE IS ABSENT from the snapshot (only the parameter names survive,
 * python/pytinydiffsim.inl:825-856: spring_k, damper_d, exponent_n, hard_contact_condition, v_transition, ...), so the law
 * is the one written down in DESIGN.md "Spring-damper contacts" (Hunt-Crossley normal force k x^n + d x^n xdot, clamped at
 * 0 with hard_contact_condition; friction mu f_n tanh(|v_t| / v_transition) against the tangential velocity; applied as
 * impulses f dt through M^-1 Jc^T): PARITY UNPINNED, self-consistent with oracle/tds_oracle.c. */
int tds_b200_set_contact_model(tds_b200_sim* sim, int contact_model, double spring_k, double damper_d, double exponent_n,
                               double v_transition, int hard_contact_condition);

/* PD / environment parameters of LocomotionContactSimulation
 * (examples/environments/locomotion_contact_simulation.h:28-48,168-258): action k drives the k-th
 * non-fixed link at or after `start_link` (base_dof_) towards initial_poses[k] + clamp(action, +-limit).
 * reward_kind: 0 none, 1 Laikago fixed-base emulation, 2 floating, 3 Ant fixed-base emulation (ant_environment2.h:75-105)
 * (examples/environments/laikago_environment2.h:130-171). */
int tds_b200_set_env(tds_b200_sim* sim, int n_act, const double* initial_poses, int start_link, double kp,
                     double kd, double max_force, double action_limit, int reward_kind);

/* VectorizedEnvironment's auto_reset_when_done (examples/ars/ars_vectorized_environment.h:262-283) on the
 * device: an environment that reports done is put back to reset_q[n_q] with zero velocity at the end of
 * that step (the reward/done outputs of the step are kept).  The host-side reset() of the Python mirror adds
 * the reference's joint noise and settle steps (laikago_environment2.h:63-116). */
int tds_b200_set_auto_reset(tds_b200_sim* sim, int enable, const double* reset_q);

int tds_b200_set_precision(tds_b200_sim* sim, int precision);
int tds_b200_get_precision(const tds_b200_sim* sim);   /* the resolved selector (never AUTO) */
/* Name of the step kernel the last tds_b200_step_* call launched (selection: DESIGN.md "Kernel selection"). */
const char* tds_b200_kernel_name(const tds_b200_sim* sim);

/* dims[0..7] = n_envs, n_stride, n_q (MultiBody::dof), n_qd (dof_qd), n_tau (dof_actuated), n_links,
 *              n_contact_points, n_act */
int tds_b200_get_dims(const tds_b200_sim* sim, int dims[8]);

/* ---- device-resident fast path -------------------------------------------------------------------
 * One launch = one step of all environments.  Pointers are DEVICE pointers to SoA fp32 arrays
 * [dim][n_stride]; q_in/qd_in may alias q_out/qd_out.  `tau_or_action`: [n_tau][n_stride] joint torques
 * (MultiBody::tau_, multi_body.hpp:86) when use_pd == 0, else [n_act][n_stride] policy actions.
 * Optional outputs may be NULL: qdd_out [n_qd][ns] (MODE_FD), reward/done [n_stride],
 * contact_dist [n_contact_points][ns] (ContactPoint::distance of every candidate point in the
 * reference's enumeration order, src/world.hpp:212-281), link_xf [n_links*12][ns].
 * stream: a cudaStream_t (NULL = default stream).  Asynchronous.  Returns a cudaError_t value. */
int tds_b200_step_device(tds_b200_sim* sim, int mode, int use_pd, const float* q_in, const float* qd_in,
                         const float* tau_or_action, float* q_out, float* qd_out, float* qdd_out, float* reward,
                         float* done, float* contact_dist, float* link_xf, void* stream);

/* ---- differentiable step (SURVEY 8f.4; the role of <model>_jacobian in the reference's generated libraries,
 * src/utils/cuda/cuda_codegen.hpp:303-426, there produced by CppAD from the recorded tape) -----------------------------
 * Dense Jacobian of one step per environment by forward-mode dual numbers (fp64) through the step kernel: rows = q' | qd'
 * (modes NOCONTACT / FULL) or qdd (mode FD); columns = q | qd | tau (use_pd == 0) or q | qd | action | kp, kd, max_force
 * (use_pd == 1: the input vector of LocomotionContactSimulation, locomotion_contact_simulation.h:160-166).  Derivatives
 * are those of the branch taken (contact set, clamps).  dims[0..1] = rows, columns.
 *   device: q, qd, tau_or_action as in tds_b200_step_device; jac [rows * cols][n_stride] fp64 (row-major per environment)
 *   host:   q [n][n_q], qd [n][n_qd], tau_or_action [n][..] fp64; jac [n][rows][cols] fp64 */
int tds_b200_jacobian_dims(const tds_b200_sim* sim, int mode, int use_pd, int dims[2]);
int tds_b200_step_jacobian_device(tds_b200_sim* sim, int mode, int use_pd, const float* q, const float* qd,
                                  const float* tau_or_action, double* jac, void* stream);
int tds_b200_step_jacobian_host(tds_b200_sim* sim, int mode, int use_pd, const double* q, const double* qd,
                                const double* tau_or_action, double* jac);

/* Jacobian-vector (forward mode) and vector-Jacobian (reverse mode: what a gradient needs) products of one step, without the
 * dense Jacobian.  Same instance, rows (q' | qd', or qdd in mode FD) and input blocks (q | qd | tau, or action with use_pd;
 * the PD-gain columns only through the dense Jacobian) as tds_b200_step_jacobian_device; q, qd, tau_or_action as in
 * tds_b200_step_device (tau_or_action required with use_pd and whenever its tangent / gradient is).  Every tangent and
 * gradient is fp64 [dim][n_stride]; padding columns (environment >= n) are not written.
 *   jvp: t_q, t_qd, t_tau tangents of the input blocks (NULL = zero) -> t_out [rows][n_stride].  One dual lane per environment.
 *   vjp: g_out cotangent [rows][n_stride] -> g_q, g_qd, g_tau (gradient of each block; NULL = not wanted, its directions are not
 *        launched).  One dual lane per environment and wanted input direction; each writes one double.
 * Return 0, -1 on a bad argument, -2 for TDS_B200_MODE_WORLD, -3 for use_pd without tds_b200_set_env, else a CUDA error.
 * The scratch arena of the dual instance is shared with the dense Jacobian and only grows. */
int tds_b200_step_jvp_device(tds_b200_sim* sim, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                             const double* t_q, const double* t_qd, const double* t_tau, double* t_out, void* stream);
int tds_b200_step_vjp_device(tds_b200_sim* sim, int mode, int use_pd, const float* q, const float* qd, const float* tau_or_action,
                             const double* g_out, double* g_q, double* g_qd, double* g_tau, void* stream);

/* Stand-alone integration stages of the fine-grained surface (device SoA arrays as above):
 * integrate_euler (src/dynamics/integrator.hpp:10-133): qd += qdd dt (qdd may be NULL = zero), q += qd dt, floating base
 * quaternion increment + normalisation; integrate_euler_qdd (:141-195): qd += qdd dt only. */
int tds_b200_integrate_euler_device(tds_b200_sim* sim, float* q, float* qd, const float* qdd, void* stream);
int tds_b200_integrate_euler_qdd_device(tds_b200_sim* sim, float* qd, const float* qdd, void* stream);

/* ---- host-buffer path (what VectorizedEnvironment-style callers use) --------------------------------
 * Replaces the per-call loop of SerialForwardStepper / OpenMPForwardStepper::step
 * (examples/ars/ars_vectorized_environment.h:88-137) with MultiBody-style host arrays:
 * q [n_envs][n_q], qd [n_envs][n_qd], tau_or_action [n_envs][n_tau | n_act], AoS fp64 host memory.
 * Copies in, steps once, copies out (synchronous).  Outputs may be NULL. */
int tds_b200_step_host(tds_b200_sim* sim, int mode, int use_pd, const double* q, const double* qd,
                       const double* tau_or_action, double* q_out, double* qd_out, double* qdd_out,
                       double* contact_dist);

/* Environment-level step on the sim's own resident state: VectorizedEnvironment::step
 * (examples/ars/ars_vectorized_environment.h:214-291) minus the policy: actions [n_envs][n_act] fp32
 * host (pinned for speed) -> obs [n_envs][n_q+n_qd], rewards [n_envs], dones [n_envs] fp32 host.
 * State stays on the device between calls.  Synchronous.
 * Fast paths (same results): with pinned (mapped) buffers and a model the library holds a specialised kernel for, the
 * step kernel itself reads the actions from and writes obs / rewards / dones to host memory (one launch, no copies);
 * otherwise pinned buffers -> the copy/transpose/step/pack/copy sequence is replayed from a CUDA graph captured on the
 * third call with the same pointers, and obs, rewards, dones adjacent in memory (rewards == obs + n_envs*(n_q+n_qd),
 * dones == rewards + n_envs) -> one device->host copy instead of three. */
/* ---- contact-pair index lists (World::compute_contacts_multi_body_internal, src/world.hpp:212-281;
 * MultiBodyContactPoint::{multi_body_a, link_a, multi_body_b, link_b}, src/mb_constraint_solver.hpp:29-40) -------------
 * The candidate points of a model are static: plane (body 0, base link -1) x every sphere / capsule end of the robot
 * (body 1) in the reference's enumeration order.  tds_b200_contact_pairs writes one tuple (body_a, link_a, body_b, link_b)
 * per candidate (the list World::mb_contacts_ holds after every step) and returns their number.
 * tds_b200_contact_list_*: the list the constraint solver keeps in a step (all candidates with keep_all_points, else
 * those with distance < 0: resolve_collision, mb_constraint_solver.hpp:169-180), computed on the device from the
 * contact distances of that step: count[e] and (link_a, link_b) of the k-th kept point, -9 beyond count.
 *   device: contact_dist [n_points][ns] (output of tds_b200_step_device), count [ns], links [2 * n_points][ns]
 *   host:   uses the distances of the last tds_b200_step_host(..., contact_dist != NULL); count [n], links [n][n_points][2]
 * Worlds of several multibodies (TDSM_H_NBODIES > 1, include/tds_b200_model.h): the multibodies of the model are bodies
 * 1, 2, ... of the world (the plane, if any, is body 0), link indices are those inside their multibody, and the candidates
 * BETWEEN multibodies (sphere-sphere, capsule-sphere; one list of World::mb_contacts_ per pair a < b, src/world.hpp:212-281)
 * follow the plane candidates; contact_dist carries their distances in the same order (+inf: the contact function emitted no
 * point).  tds_b200_contact_list_candidates_host: cand [n][n_points] = index into the candidate list of the k-th kept point. */
int tds_b200_contact_pairs(const tds_b200_sim* sim, int* tuples, int cap);
int tds_b200_model_contact_pairs(const double* model, int n_model, int* tuples, int cap);   /* host-only, from a flat model */
/* (mb_a, link_a, geom_a, mb_b, link_b, geom_b) per candidate = the loop indices of world.hpp:212-240 at which the point is emitted
 * (geom: index in collision_geometries(link)); 6 ints per candidate, same order as tds_b200_contact_pairs */
int tds_b200_contact_tuples(const tds_b200_sim* sim, int* tuples, int cap);
int tds_b200_model_contact_tuples(const double* model, int n_model, int* tuples, int cap);   /* host-only */
int tds_b200_contact_list_device(tds_b200_sim* sim, const float* contact_dist, int* count, int* links, void* stream);
int tds_b200_contact_list_host(tds_b200_sim* sim, int* count, int* links);
int tds_b200_contact_list_candidates_host(tds_b200_sim* sim, int* count, int* cand);

int tds_b200_env_set_state_host(tds_b200_sim* sim, const double* q, const double* qd);
int tds_b200_env_get_state_host(tds_b200_sim* sim, double* q, double* qd);
int tds_b200_env_step_host(tds_b200_sim* sim, const float* actions, float* obs, float* rewards, float* dones);
/* Same, device-resident: actions/reward/done are device SoA arrays; advances the resident state. */
int tds_b200_env_step_device(tds_b200_sim* sim, const float* actions, float* reward, float* done, void* stream);
/* Device pointers of the resident state (SoA fp32 [n_q][ns], [n_qd][ns]). */
/* ---- environment layer on the device (what surrounds the step in the reference's ARS loop) ---------------------
 * Episode reset, LaikagoContactSimulation::reset (examples/environments/laikago_environment2.h:63-116): environments with
 * mask[e] != 0 (all when mask is NULL) are set to the reset pose of tds_b200_set_auto_reset plus noise on the actuated
 * joints (noise: device [n_act][n_stride], or NULL -> U(-noise_amp, noise_amp) from a counter-based generator keyed by
 * (seed, env, joint); the reference draws std::rand() * 0.05), qd = 0, then settle_steps env-steps with zero actions;
 * the other environments keep their state. */
int tds_b200_env_reset_device(tds_b200_sim* sim, const float* mask, const float* noise, float noise_amp,
                              unsigned long long seed, int settle_steps, void* stream);
/* rollout_length steps of ARSVectorizedWorker::rollouts (examples/ars/ars_vectorized_worker.h:51-141) without leaving
 * the GPU: per environment a linear policy with bias (VectorizedEnvironment::policy, ars_vectorized_environment.h:293-300;
 * parameters = weights [n_act][n_q+n_qd] row-major | biases [n_act], device layout [n_params][n_stride]) on the observation
 * (q | qd, x and y zeroed), the env-step, sticky done; total_rewards[e] = sum of (reward - shift) and steps[e] over the
 * steps the environment was alive.  Device pointers; asynchronous on `stream` (NULL: the simulator's own stream, the one
 * the host-buffer entry points use; the same holds for tds_b200_env_reset_device). */
int tds_b200_env_rollout_device(tds_b200_sim* sim, const float* policy, int n_params, int rollout_length, float shift,
                                float* total_rewards, int* steps, void* stream);
/* Observation-filter statistics of the rollouts (ars_vectorized_worker.h:93-110, running_stat.h): with a non-NULL buffer
 * (device, [3 * (n_q + n_qd)][n_stride] = count | mean | S per component, caller-owned, zero to clear) every rollout step
 * pushes the observation the policy saw into a per-environment Welford accumulator.  NULL switches it off. */
int tds_b200_env_set_obs_stats(tds_b200_sim* sim, float* stats);
/* ARS on the device (ARSVectorizedWorker::do_rollouts, ars_vectorized_worker.h:205-262; ARSLearner::weighted_sum_custom and
 * train_step, ars_learner.h:67-91,185-189).  w [n_params] device; deltas [n_params][n_stride] unit normals, one direction
 * per environment; perturb: params[p][e] = w[p] + scale * deltas[p][e] (scale = +-delta_std) in the rollout layout;
 * update: w[p] += step_size * delta_std / n * sum_e (r_pos[e] - r_neg[e]) * deltas[p][e]. */
int tds_b200_ars_perturb_device(tds_b200_sim* sim, const float* w, const float* deltas, float scale, float* params, int n_params,
                                void* stream);
int tds_b200_ars_update_device(tds_b200_sim* sim, float* w, const float* deltas, const float* r_pos, const float* r_neg,
                               float delta_std, float step_size, int n_params, void* stream);
/* reset + rollout with host buffers: policy [n_envs][n_params], noise [n_envs][n_act] or NULL, results to host. */
int tds_b200_env_rollout_host(tds_b200_sim* sim, const double* policy, int n_params, int rollout_length, double shift,
                              const double* noise, double noise_amp, unsigned long long seed, int settle_steps,
                              double* total_rewards, int* steps);

/* Env step + visual-transform stream in the instancing renderer's layout (instance = env * n_visuals + v):
 * positions[4 i] = x, y, z, 1 and orientations[4 i] = quaternion xyzw (device float arrays of 4 * n_envs * n_visuals),
 * the two arrays TinyGLInstancingRenderer holds (src/visualizer/opengl/tiny_gl_instancing_renderer.cpp:366-367,440-457);
 * same per-visual transforms as the records of the v1 output (locomotion_contact_simulation.h:281-299). */
int tds_b200_num_visuals(const tds_b200_sim* sim);
int tds_b200_env_step_visual_device(tds_b200_sim* sim, const float* actions, float* reward, float* done, float* positions,
                                    float* orientations, void* stream);

/* The simulator's own (non-blocking) cudaStream_t: what the host-buffer entry points and the env-layer calls with a NULL
 * stream run on.  Work enqueued by the caller on other streams is NOT ordered against it. */
void* tds_b200_stream(tds_b200_sim* sim);
float* tds_b200_env_q(tds_b200_sim* sim);
float* tds_b200_env_qd(tds_b200_sim* sim);

/* ---- C-ABI v1 drop-in ---------------------------------------------------------------------------------
 * Exactly the symbols the reference's CudaSourceGen emits and ars_train_policy_cuda / cuda_codegen dlsym
 * (src/utils/cuda_codegen.hpp:156-266; loaded at examples/ars/ars_train_policy_cuda.cpp:183-230):
 *   input  = num_total_threads blocks of input_dim  (51 = q18|qd18|action12|kp,kd,max_force) fp64, AoS, host
 *   output = num_total_threads blocks of output_dim (411 = q18|qd18|17x(pos3,quat4)|up.z|zeros) fp64, AoS, host
 * Synchronous: H2D, one step, D2H.  num_blocks / num_threads_per_block are accepted and ignored (the
 * launch geometry is chosen for sm_100a). */
typedef struct {
  int output_dim;
  int input_dim;
  int global_dim;
} CudaFunctionMetaData; /* src/utils/cuda_codegen.hpp:27-31 */

void cuda_model_laikago_forward_zero(int num_total_threads, int num_blocks, int num_threads_per_block,
                                     double* output, const double* input);
CudaFunctionMetaData cuda_model_laikago_forward_zero_meta(void);
void cuda_model_laikago_forward_zero_allocate(int num_total_threads);
void cuda_model_laikago_forward_zero_deallocate(void);
/* "cuda_model_" + AntContactSimulation2::env_name() (examples/ars/ars_train_policy_cuda.cpp:507, ant_environment2.h):
 * input_dim 39 = q14|qd14|action8|kp,kd,max_force, output_dim 155 = q14|qd14|9x(pos3,quat4)|up.z|zeros */
void cuda_model_ant_forward_zero(int num_total_threads, int num_blocks, int num_threads_per_block,
                                 double* output, const double* input);
CudaFunctionMetaData cuda_model_ant_forward_zero_meta(void);
void cuda_model_ant_forward_zero_allocate(int num_total_threads);
void cuda_model_ant_forward_zero_deallocate(void);

/* ---- C-ABI v2 (alt): what tds::CudaLibrary / CudaModel / CudaFunction load (src/utils/cuda/cuda_library.hpp:51-68,
 * cuda_model.hpp:14-25, cuda_function.hpp:78-100; emitted at src/utils/cuda/cuda_codegen.hpp:32-231).  One model,
 * "b200_laikago" (same 51 -> 411 function as cuda_model_laikago) with its <model>_jacobian. */
typedef struct { int output_dim; int local_input_dim; int global_input_dim; bool accumulated_output; } CudaFunctionMetaDataV2;
void model_info(char const* const** names, int* count);
CudaFunctionMetaDataV2 b200_laikago_forward_zero_meta(void);
void b200_laikago_forward_zero_allocate(int num_total_threads);
void b200_laikago_forward_zero_deallocate(void);
bool b200_laikago_forward_zero_send_local(int num_total_threads, const double* input);
bool b200_laikago_forward_zero_send_global(const double* input);
void b200_laikago_forward_zero(int num_total_threads, int num_blocks, int num_threads_per_block, double* output);
/* <model>_jacobian of the same generation (src/utils/cuda/cuda_codegen.hpp:303-426): rows = the 36 state outputs q' | qd'
 * (output sparsity, :283-288), columns = the 51 local inputs; output_dim = 36 * 51 per thread, row-major, not accumulated. */
CudaFunctionMetaDataV2 b200_laikago_jacobian_meta(void);
void b200_laikago_jacobian_allocate(int num_total_threads);
void b200_laikago_jacobian_deallocate(void);
bool b200_laikago_jacobian_send_local(int num_total_threads, const double* input);
bool b200_laikago_jacobian_send_global(const double* input);
void b200_laikago_jacobian(int num_total_threads, int num_blocks, int num_threads_per_block, double* output);

/* ---- the RigidBody path of World::step (src/world.hpp:293-363, src/rigid_body.hpp, src/rb_constraint_solver.hpp) ----------
 * A world of up to 16 rigid bodies with ONE collision shape each (sphere, plane, capsule, box), a batch of such worlds per
 * simulator, one GPU lane per world: apply_gravity / apply_force_impulse / clear_forces, contacts of every pair through the
 * reference's dispatcher (sphere-sphere, plane-sphere / capsule / box, capsule-sphere, and the swapped calls), the
 * sequential-impulse solver (num_solver_iterations sweeps over the contact list), integrate.
 *   desc   [n_bodies][6]  = mass (0: static), shape (TDSG_*, tds_b200_model.h), p0..p3: sphere radius | capsule radius, length |
 *                           box extents | plane normal [3], constant
 *   state  per body 13 doubles: position [3], orientation xyzw [4], linear velocity [3], angular velocity [3]
 *          device layout [13 * n_bodies][n_stride] fp64 (n_stride = n_worlds rounded up to 32), host layout [n_worlds][n_bodies][13]
 *   force  RigidBody::apply_central_force before the FIRST step ([3 * n_bodies][n_stride] / [n_worlds][n_bodies][3]) or NULL
 * Defaults are the reference's (dt 1/60 is ours): gravity (0, 0, -9.81), friction 0.5, restitution 0, erp 0.1, 1 solver iteration.
 * tds_b200_rigid_jacobian_host: d state_out / d (state | force) [n_worlds][13 n_bodies][16 n_bodies] by forward-mode dual numbers
 * (python/examples/billiard_optimization.py differentiates exactly this path). */
typedef struct tds_b200_rigid tds_b200_rigid;
tds_b200_rigid* tds_b200_rigid_create(const double* desc, int n_bodies, int n_worlds, int device);
void tds_b200_rigid_destroy(tds_b200_rigid* h);
int tds_b200_rigid_set_params(tds_b200_rigid* h, double dt, const double* gravity, double friction, double restitution, double erp,
                              int num_solver_iterations);
int tds_b200_rigid_step_device(tds_b200_rigid* h, const double* state_in, double* state_out, const double* force, int steps, void* stream);
int tds_b200_rigid_step_host(tds_b200_rigid* h, const double* state, const double* force, int steps, double* state_out);
int tds_b200_rigid_jacobian_host(tds_b200_rigid* h, const double* state, const double* force, int steps, double* state_out, double* jac);
/* Jacobian-vector / vector-Jacobian products of `steps` steps with respect to (state | force), device layouts as
 * tds_b200_rigid_step_device, tangents and gradients fp64 [13 * n_bodies][n_stride] (state) / [3 * n_bodies][n_stride] (force).
 * One dual lane carries its derivative through all the steps, so memory does not grow with `steps`.  NULL force: zero force.
 *   jvp: t_state, t_force (NULL = zero) -> t_out, one lane per world.
 *   vjp: g_out -> g_state, g_force (NULL = not wanted, not launched), one lane per world and wanted input direction.
 * stream NULL: the world's own stream. */
int tds_b200_rigid_jvp_device(tds_b200_rigid* h, const double* state, const double* force, int steps,
                              const double* t_state, const double* t_force, double* t_out, void* stream);
int tds_b200_rigid_vjp_device(tds_b200_rigid* h, const double* state, const double* force, int steps,
                              const double* g_out, double* g_state, double* g_force, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TDS_B200_H */
