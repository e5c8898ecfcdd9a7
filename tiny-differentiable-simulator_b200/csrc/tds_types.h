// Host/device shared POD types of the batched simulator.
#pragma once
#include <stdint.h>

#define TDS_MAX_LINKS 40
#define TDS_MAX_GEOMS 24
#define TDS_MAX_VIS 24
#define TDS_MAX_ACT 32
#define TDS_MAX_POINTS 64   // candidate contact points of a model (sphere 1, capsule 2, box 8 per geom)
#define TDS_MAX_PAIR_POINTS 64   // candidate contact points between geoms of DIFFERENT multibodies of one world
#define TDS_MAX_PAIR_GROUPS 10   // ordered multibody pairs (a < b) that have such candidates (5 multibodies: 10 pairs)

// link flags
#define TDS_LF_PARENT_ADJ 1   // parent == i-1  -> deltas are carried in registers
#define TDS_LF_CHILD_ADJ 2    // link i+1 exists and its parent is i
#define TDS_LF_REVOLUTE 4
#define TDS_LF_PRISMATIC 8
#define TDS_LF_FIXED 16
#define TDS_LF_XT_IDENT 32     // X_T rotation is the identity
#define TDS_LF_SPHERICAL 64    // JOINT_SPHERICAL: 4 coordinates (quaternion xyzw), 3 velocities; world-frame kernel only

// Device model: constant for all environments, passed as a __grid_constant__ kernel parameter
// (lives in the constant bank; every lane reads the same entry -> broadcast).
// Flattened from the reference's MultiBody/Link (src/multi_body.hpp:13, src/link.hpp:24).
struct DevModel {
  int n_links, floating, n_q, n_qd;
  int n_geoms, n_acc, has_plane, max_contacts;
  int base_acc;      // accumulator slot of the floating base (-1 if fixed base)
  int n_vis, pad1, pad2;
  // scratch arena layout, in 4-byte words per environment (see tds_step.cu)
  int w_q, w_qd, w_tau, w_link, w_acc, w_xw, w_M, w_invd, w_w, w_con, w_conS, w_Y, w_total;
  int link_words;    // words per link in the per-link region
  int acc_words, acc_ic_word;  // accumulator slot stride / offset of its Ic part (words)
  // ---- layout of the world-frame kernel (tds_stepw.cu), 4-byte words ----
  int x_q, x_qd, x_tau, x_S, x_link, x_xw, x_acc, x_M, x_dinv, x_w, x_con, x_conS, x_Y, x_total;
  int x_link_words, x_acc_words, x_acc_ic_word;
  int nb;            // number of 3x3 dof blocks (n_qd padded to a multiple of 3)
  int n_prefix;      // leading chain links with prismatic / fixed joints only: the common-frame origin is the
                     // world position of link n_prefix (computable without trigonometry); -1: floating base
  int n_xw;          // links whose world transform must be kept for non-adjacent children
  int xw_slot[TDS_MAX_LINKS];
  int geom_begin[TDS_MAX_LINKS + 2];   // geoms of link i (-1 = base) are [geom_begin[i+1], geom_begin[i+2])
  double rbic[TDS_MAX_LINKS][10];      // mass, com (link frame) [3], inertia about the com (xx,xy,xz,yy,yz,zz)
  double base_rbic[10];
  int parent[TDS_MAX_LINKS];
  int jtype[TDS_MAX_LINKS];
  int q_idx[TDS_MAX_LINKS];
  int qd_idx[TDS_MAX_LINKS];
  int flags[TDS_MAX_LINKS];
  int acc_slot[TDS_MAX_LINKS];   // accumulator slot receiving non-adjacent children (-1: none)
  double XT[TDS_MAX_LINKS][12];  // X_T: R row-major [9], t [3]
  double axis[TDS_MAX_LINKS][3];
  double rbi[TDS_MAX_LINKS][10]; // mass, h = m*com [3], I about link origin (xx,xy,xz,yy,yz,zz)
  float stiffness[TDS_MAX_LINKS];
  float damping[TDS_MAX_LINKS];
  double base_rbi[10];
  float base_inertia_com[9];     // base_rbi.inertia (about com), for the gyroscopic term
  // collision geoms of the robot in the reference's enumeration order
  int g_link[TDS_MAX_GEOMS];
  int g_type[TDS_MAX_GEOMS];
  double g_t[TDS_MAX_GEOMS][3];     // local translation
  double g_half[TDS_MAX_GEOMS][3];  // capsule: local half-axis R_local * (0,0,L/2); plane shape on a link: its unit normal
  double g_radius[TDS_MAX_GEOMS];
  double g_box[TDS_MAX_GEOMS][9];   // box: the three local half-axes R_local * diag(extent / 2 - r), columns x | y | z
  int n_sph;                        // spherical joints; S columns of the s-th one at x_S3 + s * 18 RC words
  int s3_slot[TDS_MAX_LINKS];
  int x_S3;
  int world_only;   // the model uses features only the generic world-frame kernel (tds_stepw.cu) implements
                    // (box shapes, spherical joints, several multibodies): the decomposed / specialised kernels refuse it
  // ---- several multibodies in one world (header field TDSM_H_NBODIES > 1): every root link starts a multibody ------------
  // Contacts between geoms of different multibodies (world.hpp:206-282) are solved pair of multibodies after pair of
  // multibodies, after the plane contacts (the plane is multibody 0 of the reference's world): world.hpp:351-355.
  int n_bodies;
  int body_of[TDS_MAX_LINKS];            // multibody of a link
  int n_pair_points, n_pair_groups;
  int pg_begin[TDS_MAX_PAIR_GROUPS + 1]; // candidate points of group g: [pg_begin[g], pg_begin[g + 1]), groups in (a, b) lexicographic order
  int pp_ga[TDS_MAX_PAIR_POINTS];        // geom on the lower-indexed multibody (body A of the contact)
  int pp_gb[TDS_MAX_PAIR_POINTS];        // geom on the other one (body B)
  int pp_kind[TDS_MAX_PAIR_POINTS];      // 0 sphere-sphere; +-1 capsule A (end +-L/2) x sphere B; +-2 sphere A x capsule B (dispatcher swap);
                                         // 100 + k: plane shape on A x point k of B's sphere / capsule / box; 200 + k: the plane on B (swap)
  int g_wslot[TDS_MAX_GEOMS];            // slot of the geom's world centre (+ capsule half axis) kept for the pair stage, -1: none
  int n_gw, max_pair_rows;               // slots; largest group (rows of the pair LCP)
  int x_gw, x_pcon;                      // arena: [n_gw][12] RC, [n_pair_points][9] RC
  // static ground plane (multibody 0)
  double plane_n[3];
  double plane_c;
  double fr1[3], fr2[3];  // plane_space(-n), src/mb_constraint_solver.hpp:506-520
};

struct DevVisuals {   // only used by the drop-in (v1 ABI) output packing
  int n_vis, n_links, n_q, n_qd;
  int v_link[TDS_MAX_VIS];
  float v_R[TDS_MAX_VIS][9];
  float v_t[TDS_MAX_VIS][3];
};

// World / solver / env parameters (src/world.hpp:65-69, src/mb_constraint_solver.hpp:59-70,
// examples/environments/locomotion_contact_simulation.h:168-258).
struct SimParams {
  double dt;
  double gravity[3];
  double friction, restitution, erp, cfm;
  int pgs_iterations;
  int keep_all_points;
  // contact law: 0 = the reference's impulse-level LCP / PGS; 1 = spring-damper (Hunt-Crossley normal force + smoothed
  // Coulomb friction, DESIGN.md "Spring-damper contacts"; parameter names of the reference's absent
  // MultiBodyConstraintSolverSpring, python/pytinydiffsim.inl:825-856).  World-frame kernel only.
  int contact_model;
  int hard_contact_condition;
  double spring_k, damper_d, exponent_n, v_transition;
  double inv_dt;   // 1 / dt, computed once on the host (the specialised kernel multiplies instead of dividing per contact row)
};

struct EnvParams {
  int n_act;           // action_dim
  int start_link;      // base_dof_ for fixed-base emulation (first PD-controlled link)
  float kp, kd, max_force, action_limit;
  float initial_poses[TDS_MAX_ACT];
  int act_link[TDS_MAX_ACT];   // link index driven by action k
  // reward/done (examples/environments/laikago_environment2.h:130-171)
  int reward_kind;     // 0 none, 1 laikago (fixed-base emulation), 2 laikago floating
  int auto_reset;      // reset an environment to reset_q when it reports done
  float reset_q[TDS_MAX_LINKS + 8];
};

// Pointers to SoA state in HBM: array [dim][n_stride] (environment index fastest).
struct StepIO {
  const float* q_in; const float* qd_in; const float* tau_in;  // tau_in: [n_tau][n] or action [n_act][n]
  float* q_out; float* qd_out; float* qdd_out;
  float* reward; float* done;           // may be null
  float* contact_dist;                  // [n_contact_points][n] or null
  float* link_xf;                       // [n_links*12][n] world transforms of the step's FK, or null
  long long* phase_clk;                 // [n_warps][16] clock64() stamps at phase boundaries (profiling), or null
  // host-facing layouts served directly by the specialised kernel (other kernels: staged by transposes, tds_capi.cu)
  const float* act_aos;                 // actions [n][n_act] (environment-major), or null -> tau_in
  float* obs_aos;                       // observations [n][n_q + n_qd] = q | qd after the step, or null
  float* obs_tail;                      // reward [n] then done [n] behind the observations, or null
  // differentiable step (tds_stepw.cu instantiated on dual numbers): Jacobian [n_rows * jac_n_in][n_stride], fp64;
  // rows = q' | qd' (or qdd in forward-dynamics mode), columns = q | qd | tau or action (| kp, kd, max_force with PD)
  double* jac; int jac_n_in; int jac_dir0;
  int n; int n_stride;
};

// Products with the step's Jacobian, computed by the dual-number instances instead of (or besides) the dense Jacobian.
// A trailing kernel parameter of its own, not part of StepIO: the float / double instances keep their parameter layout.
// Input blocks: q | qd | tau or action (tds_stepw.cu), state | force (tds_rigid.cu); output rows as the dense Jacobian's.
// Every array is fp64 [dim][n_stride].
struct DualIO {
  const double* jvp_tan[3];   // JVP (one lane per environment): tangent of each input block, null = zero
  double* jvp_out;            // JVP: tangent of the output rows
  const double* vjp_cot;      // VJP (one lane per environment and input direction): cotangent of the output rows
  double* vjp_out[3];         // VJP: gradient of each input block; the lane of direction d writes sum_r cot_r * d out_r / d in_d
};
