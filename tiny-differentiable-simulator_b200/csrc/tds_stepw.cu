// World-frame batched env-step kernel for sm_100a (successor of tds_step.cu's link-frame kernel).
//
// Same reference path as tds_step.cu (PD -> kinematics -> ABA -> integrate_euler_qdd -> contacts -> CRBA ->
// LCP/PGS -> integrate_euler; citations at each stage), restructured once more around the instruction count,
// because with 4096 environments one warp owns an SM and every instruction is paid at single-warp latency:
//
//   * ALL spatial quantities of an environment live in ONE common frame: world axes, origin O that moves
//     with the robot (base position, or the end of the translation-only root chain).  Then
//       - velocities / accelerations propagate by addition (v_i = v_parent + S_i qd_i),
//       - articulated and composite inertias accumulate by addition: the per-link congruence transform
//         X^T Ia X of the reference (forward_dynamics.hpp:187-189, mass_matrix.hpp:45-46; ~250 FMA per link
//         even in block form) disappears; the price is moving each link's rigid-body inertia into the common
//         frame once (~70 FMA, shared by ABA and CRBA),
//       - M_ij = S_j . (Ic_i S_i) and contact Jacobian columns = S_j.bot + S_j.top x x_c need no chain walks
//         with transforms.
//     Equivalent to the reference in exact arithmetic (spatial algebra is frame invariant); the floating-base
//     quirks that ARE frame dependent (block inverse with C = -H, gyroscopic term, un-rotated gravity) are
//     evaluated in the base frame exactly as the reference does.
//   * Only S (6 numbers), v/c/a, U, 1/D, u per link are kept; world transforms are carried in registers and
//     stored only for branch points.
//   * The contact solve works on 3x3 register blocks (dofs padded to a multiple of 3): blocked Cholesky,
//     blocked forward substitution of 3 right-hand sides per contact, matrix-free PGS on w = Y p, blocked
//     back substitution.  A block op is 18 shared loads for 27 FMA with compile-time indexing.
//   * Scalar types: RA (ABA) fp32, RC (kinematics, contact geometry, inertias in the common frame, CRBA
//     products, Jacobians, LCP right-hand side) fp64, RS (factorisation, substitutions, PGS) fp32 in the
//     default mixed mode.
#include <cuda_runtime.h>

#include "tds_wcommon.cuh"

namespace tdsw {


// per-link region, element offsets: [rigid inertia (10 RC) | later U (6 RA), invD, u] then v / c / a (6 RA)

// RQ: scalar of the state vectors (q, qd, tau): float, or the dual number type in the differentiable instance
// (RA = RC = RS = RQ = Dual<double>: blockIdx.y + io.jac_dir0 is the input direction of the lane, see tds_dual.cuh).
template <typename RA, typename RC, typename RS, typename RQ, bool SMEM>
__global__ void __launch_bounds__(128, 1)
tds_stepw_kernel(const __grid_constant__ DevModel M, const __grid_constant__ SimParams P,
                 const __grid_constant__ EnvParams E, const StepIO io, const int mode, const int use_pd,
                 char* __restrict__ gscratch, const DualIO dio = DualIO()) {
  extern __shared__ __align__(16) char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warp_in_blk = threadIdx.x >> 5;
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = env < io.n;
  const int e = live ? env : io.n - 1;
  constexpr bool AD = is_dual<RQ>::value;
  const int dir = AD ? (int)blockIdx.y + io.jac_dir0 : -1;     // differentiable instance: this lane's input direction
  Arena A;
  if (SMEM) { A.blk = smem_raw + (size_t)warp_in_blk * M.x_total * 32 * 4; A.stride = 32; A.col = lane; }
  else { A.blk = gscratch + ((size_t)blockIdx.y * ((size_t)gridDim.x * (blockDim.x >> 5)) + (size_t)(env >> 5)) * M.x_total * 32 * 4; A.stride = 32; A.col = lane; }  // per-warp block, same addressing as shared memory
  const int ST = A.stride;
  const int ns = io.n_stride;
  const int n_links = M.n_links;
  const int n = M.n_qd;
  const int nb = M.nb;
  const int n3 = 3 * nb;
  int phase_id = 0;
#define TDSW_PHASE() do { if (io.phase_clk && lane == 0) io.phase_clk[(size_t)(env >> 5) * 16 + (phase_id++)] = clock64(); } while (0)
  TDSW_PHASE();
  constexpr int RAW = (int)(sizeof(RA) / 4), RCW = (int)(sizeof(RC) / 4);
  RQ* const qv = A.ptr<RQ>(M.x_q);
  RQ* const qdv = A.ptr<RQ>(M.x_qd);
  RQ* const tauv = A.ptr<RQ>(M.x_tau);
  RC* const Sw = A.ptr<RC>(M.x_S);                 // S of link i at Sw + i*6*ST
  RC* const S3w = A.ptr<RC>(M.x_S3);               // spherical joints: three columns at S3w + s3_slot*18*ST
  // column c of link j's motion subspace (1 column, or 3 for a spherical joint)
  auto S_col = [&](int j, int c) -> Sv<RC> {
    return (M.flags[j] & TDS_LF_SPHERICAL) ? ld6<RC>(S3w + (M.s3_slot[j] * 3 + c) * 6 * ST, ST) : ld6<RC>(Sw + j * 6 * ST, ST);
  };
  auto n_cols = [&](int j) -> int { return (M.flags[j] & TDS_LF_FIXED) ? 0 : ((M.flags[j] & TDS_LF_SPHERICAL) ? 3 : 1); };
  const int LWD = M.x_link_words;
  const int VOFF = LWD - 6 * RAW;                  // word offset of v/c/a inside a link record
  RS* const Mb = A.ptr<RS>(M.x_M);
  RS* const dinv = A.ptr<RS>(M.x_dinv);
  RS* const wv = A.ptr<RS>(M.x_w);

  // ---- load state, PD torques (locomotion_contact_simulation.h:168-258) ---------------------------
  // input directions of the differentiable instance: q | qd | tau or action | kp, kd, max_force (with PD)
  const int in0 = M.n_q + n;
  // input direction idx -> its block (0 q, 1 qd, 2 tau or action) and its row there; -1: a PD gain (dense Jacobian only)
  auto blk_of = [&](int idx, int& row) -> int {
    if (idx < M.n_q) { row = idx; return 0; }
    if (idx < in0) { row = idx - M.n_q; return 1; }
    row = idx - in0;
    return row < (use_pd ? E.n_act : n - (M.floating ? 6 : 0)) ? 2 : -1;
  };
  // derivative part of input idx: the caller's tangent (JVP), else d input_idx / d direction (Jacobian column, VJP)
  auto seed = [&](RQ x, int idx) -> RQ {
    if constexpr (AD) {
      if (dio.jvp_out) { int r; const int b = blk_of(idx, r); x.d = (b >= 0 && dio.jvp_tan[b]) ? dio.jvp_tan[b][(size_t)r * ns + e] : 0.0; }
      else if (idx == dir) x.d = 1.0;
    }
    return x;
  };
  // dual instance: output row r (q' | qd', or qdd in MODE_FD) has derivative d in this lane
  double vjp_acc = 0.0;   // VJP: sum_r cot_r * d out_r / d direction
  auto emit_row = [&](int r, double d) {
    if constexpr (AD) {
      if (io.jac) io.jac[((size_t)r * io.jac_n_in + dir) * ns + e] = d;
      if (dio.jvp_out) dio.jvp_out[(size_t)r * ns + e] = d;
      if (dio.vjp_cot) vjp_acc += dio.vjp_cot[(size_t)r * ns + e] * d;
    }
  };
  auto store_vjp = [&]() {
    if constexpr (AD) {
      if (!dio.vjp_cot) return;
      int r; const int b = blk_of(dir, r);
      if (b >= 0 && dio.vjp_out[b]) dio.vjp_out[b][(size_t)r * ns + e] = vjp_acc;
    }
  };
  for (int k = 0; k < M.n_q; ++k) qv[k * ST] = seed(RQ(io.q_in[(size_t)k * ns + e]), k);
  for (int k = 0; k < n; ++k) qdv[k * ST] = seed(RQ(io.qd_in[(size_t)k * ns + e]), M.n_q + k);
  for (int k = 0; k < n; ++k) tauv[k * ST] = RQ(0.f);
  if (use_pd) {
    const RQ kp = seed(RQ(E.kp), in0 + E.n_act), kd = seed(RQ(E.kd), in0 + E.n_act + 1), fmax_ = seed(RQ(E.max_force), in0 + E.n_act + 2);
    for (int k = 0; k < E.n_act; ++k) {
      const int li = E.act_link[k];
      RQ a = seed(RQ(io.tau_in[(size_t)k * ns + e]), in0 + k);
      a = max_t(min_t(a, RQ(E.action_limit)), RQ(-E.action_limit));
      const RQ q_des = RQ(E.initial_poses[k]) + a;
      RQ f = kp * (q_des - qv[M.q_idx[li] * ST]) + kd * (RQ(0.f) - qdv[M.qd_idx[li] * ST]);
      f = min_t(max_t(f, -fmax_), fmax_);
      tauv[M.qd_idx[li] * ST] = f;
    }
  } else if (io.tau_in) {
    const int off = M.floating ? 6 : 0;
    for (int k = off; k < n; ++k) tauv[k * ST] = seed(RQ(io.tau_in[(size_t)(k - off) * ns + e]), in0 + k - off);
  }
  for (int s = 0; s < M.n_acc; ++s) {
    RA* pa = A.ptr<RA>(M.x_acc + s * M.x_acc_words);
    for (int k = 0; k < 27; ++k) pa[k * ST] = RA(0);
    RC* pc = A.ptr<RC>(M.x_acc + s * M.x_acc_words + M.x_acc_ic_word);
    for (int k = 0; k < 10; ++k) pc[k * ST] = RC(0);
  }
  const bool world_step = mode == MODE_WORLD;   // World::step(dt) on its own (src/world.hpp:302-363): q, qd in -> qd out
  const bool want_contacts = (mode == MODE_FULL || world_step) && (M.has_plane || M.n_pair_points > 0);
  TDSW_PHASE();  // 1

  // ---- common-frame origin O (world coordinates) -----------------------------------------------------
  M3<RC> Rb = m3_identity<RC>();
  V3<RC> O = v3<RC>(RC(0), RC(0), RC(0));
  if (M.floating) {
    Rb = quat_to_matrix<RC>(RC(qv[0]), RC(qv[ST]), RC(qv[2 * ST]), RC(qv[3 * ST]));
    O = v3<RC>(RC(qv[4 * ST]), RC(qv[5 * ST]), RC(qv[6 * ST]));
  } else {
    // end of the translation-only root chain: constant rotations, no trigonometry
    M3<RC> Rc = m3_identity<RC>();
    const int kp = M.n_prefix < n_links ? M.n_prefix + 1 : n_links;
    for (int i = 0; i < kp; ++i) {
      const double* xt = M.XT[i];
      O = O + mul(Rc, v3<RC>(RC(xt[9]), RC(xt[10]), RC(xt[11])));
      if (i == M.n_prefix) break;
      if (!(M.flags[i] & TDS_LF_XT_IDENT)) {
        M3<RC> r; r.xx = RC(xt[0]); r.xy = RC(xt[1]); r.xz = RC(xt[2]); r.yx = RC(xt[3]); r.yy = RC(xt[4]); r.yz = RC(xt[5]); r.zx = RC(xt[6]); r.zy = RC(xt[7]); r.zz = RC(xt[8]);
        Rc = mul(Rc, r);
      }
      if (M.flags[i] & TDS_LF_PRISMATIC) {
        const RC qi = RC(qv[M.q_idx[i] * ST]);
        O = O + mul(Rc, v3<RC>(RC(M.axis[i][0]) * qi, RC(M.axis[i][1]) * qi, RC(M.axis[i][2]) * qi));
      }
    }
  }

  // ---- pass 1: root -> leaf.  kinematics.hpp:18-148 in the common frame + contact detection ------------
  const V3<RC> pn = v3<RC>(RC(M.plane_n[0]), RC(M.plane_n[1]), RC(M.plane_n[2]));
  const RC plane_off = dot(O, pn) - RC(M.plane_c);   // n.(O + x) - c = n.x + plane_off
  int n_active = 0, pt_index = 0;
  auto emit_point = [&](int li, const V3<RC>& pos, const RC rad) {
    if (!M.has_plane) return;
    const RC dist = dot(pos, pn) + plane_off - rad;       // contact_plane_sphere, contact_point.hpp:112-116
    if (io.contact_dist && live) io.contact_dist[(size_t)pt_index * ns + e] = (float)val_of(dist);
    ++pt_index;
    if (dist < RC(0) && n_active < M.max_contacts) {
      RC* pc = A.ptr<RC>(M.x_con + n_active * 5 * RCW);
      st3<RC>(pc, ST, pos - pn * rad);                     // world_point_on_b, relative to O
      pc[3 * ST] = dist;
      pc[4 * ST] = RC(li);
      ++n_active;
    }
  };
  auto emit_geoms = [&](int li, const M3<RC>& R, const V3<RC>& pr) {
    for (int g = M.geom_begin[li + 1]; g < M.geom_begin[li + 2]; ++g) {
      const int ty = M.g_type[g];
      if (ty != TDSG_SPHERE && ty != TDSG_CAPSULE && ty != TDSG_BOX) continue;
      const V3<RC> c = pr + mul(R, v3<RC>(RC(M.g_t[g][0]), RC(M.g_t[g][1]), RC(M.g_t[g][2])));
      const RC rad = RC(M.g_radius[g]);
      if (M.g_wslot[g] >= 0) {         // kept for the contacts between multibodies (after this pass)
        RC* pw = A.ptr<RC>(M.x_gw + M.g_wslot[g] * 12 * RCW);
        st3<RC>(pw, ST, c);
        if (ty == TDSG_CAPSULE) st3<RC>(pw + 3 * ST, ST, mul(R, v3<RC>(RC(M.g_half[g][0]), RC(M.g_half[g][1]), RC(M.g_half[g][2]))));
        if (ty == TDSG_BOX) {
          const double* b = M.g_box[g];
          st3<RC>(pw + 3 * ST, ST, mul(R, v3<RC>(RC(b[0]), RC(b[1]), RC(b[2]))));
          st3<RC>(pw + 6 * ST, ST, mul(R, v3<RC>(RC(b[3]), RC(b[4]), RC(b[5]))));
          st3<RC>(pw + 9 * ST, ST, mul(R, v3<RC>(RC(b[6]), RC(b[7]), RC(b[8]))));
        }
      }
      if (ty == TDSG_SPHERE) emit_point(li, c, rad);
      else if (ty == TDSG_CAPSULE) {   // contact_plane_capsule, contact_point.hpp:128-161: end spheres at +L/2, then -L/2
        const V3<RC> half = mul(R, v3<RC>(RC(M.g_half[g][0]), RC(M.g_half[g][1]), RC(M.g_half[g][2])));
        emit_point(li, c + half, rad);
        emit_point(li, c - half, rad);
      } else {                         // contact_plane_box, contact_point.hpp:164-198: corner spheres, x outermost, z innermost
        const double* b = M.g_box[g];
        const V3<RC> ex = mul(R, v3<RC>(RC(b[0]), RC(b[1]), RC(b[2])));
        const V3<RC> ey = mul(R, v3<RC>(RC(b[3]), RC(b[4]), RC(b[5])));
        const V3<RC> ez = mul(R, v3<RC>(RC(b[6]), RC(b[7]), RC(b[8])));
        for (int k = 0; k < 8; ++k) {
          V3<RC> pos = (k & 4) ? c - ex : c + ex;
          pos = (k & 2) ? pos - ey : pos + ey;
          pos = (k & 1) ? pos - ez : pos + ez;
          emit_point(li, pos, rad);
        }
      }
    }
  };
  M3<RC> R_prev = Rb;
  V3<RC> p_prev = M.floating ? v3<RC>(RC(0), RC(0), RC(0)) : v3<RC>(-O.x, -O.y, -O.z);
  Sv<RA> v_prev;
  if (M.floating) {  // base-frame spatial velocity qd[0:6] (kinematics.hpp:45-47) expressed in the common frame
    const M3<RA> RbA = cvt<RA>(Rb);
    v_prev.top = mul(RbA, v3<RA>(RA(qdv[0]), RA(qdv[ST]), RA(qdv[2 * ST])));
    v_prev.bot = mul(RbA, v3<RA>(RA(qdv[3 * ST]), RA(qdv[4 * ST]), RA(qdv[5 * ST])));
  } else {
    v_prev.top = v3<RA>(RA(0), RA(0), RA(0)); v_prev.bot = v_prev.top;
  }
  const M3<RC> R_base = R_prev;
  const V3<RC> p_base = p_prev;
  const Sv<RA> v_base = v_prev;
  { RC* px = A.ptr<RC>(M.x_xw); st9<RC>(px, ST, R_base); st3<RC>(px + 9 * ST, ST, p_base); }
  if (want_contacts) emit_geoms(-1, R_base, p_base);
  for (int i = 0; i < n_links; ++i) {
    const int p = M.parent[i];
    const int fl = M.flags[i];
    M3<RC> Rp; V3<RC> pp; Sv<RA> vp;
    if (fl & TDS_LF_PARENT_ADJ) { Rp = R_prev; pp = p_prev; vp = v_prev; }
    else if (p >= 0) {
      const RC* px = A.ptr<RC>(M.x_xw + (M.xw_slot[p] + 1) * 12 * RCW);
      Rp = ld9<RC>(px, ST); pp = ld3<RC>(px + 9 * ST, ST);
      vp = ld6<RA>(A.ptr<RA>(M.x_link + p * LWD + VOFF), ST);
    } else { Rp = R_base; pp = p_base; vp = v_base; }
    const double* xt = M.XT[i];
    V3<RC> pi = pp + mul(Rp, v3<RC>(RC(xt[9]), RC(xt[10]), RC(xt[11])));
    M3<RC> Ri = Rp;
    if (!(fl & TDS_LF_XT_IDENT)) {
      M3<RC> r; r.xx = RC(xt[0]); r.xy = RC(xt[1]); r.xz = RC(xt[2]); r.yx = RC(xt[3]); r.yy = RC(xt[4]); r.yz = RC(xt[5]); r.zx = RC(xt[6]); r.zy = RC(xt[7]); r.zz = RC(xt[8]);
      Ri = mul(Rp, r);
    }
    Sv<RC> S; S.top = v3<RC>(RC(0), RC(0), RC(0)); S.bot = S.top;
    if (!(fl & TDS_LF_FIXED)) {   // Link::jcalc, link.hpp:229-336
      const RC qi = RC(qv[M.q_idx[i] * ST]);
      const int jt = M.jtype[i];
      const V3<RC> ax = v3<RC>(RC(M.axis[i][0]), RC(M.axis[i][1]), RC(M.axis[i][2]));
      if (fl & TDS_LF_SPHERICAL) {   // X_J = quat_to_matrix(q[0..3]) (link.hpp:268-272); S = [1 0]^T in the link frame
        const int q0 = M.q_idx[i];
        Ri = mul(Ri, quat_to_matrix<RC>(RC(qv[q0 * ST]), RC(qv[(q0 + 1) * ST]), RC(qv[(q0 + 2) * ST]), RC(qv[(q0 + 3) * ST])));
        RC* const s3 = S3w + M.s3_slot[i] * 18 * ST;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const V3<RC> w = a == 0 ? col_x(Ri) : (a == 1 ? col_y(Ri) : col_z(Ri));
          Sv<RC> Sa; Sa.top = w; Sa.bot = cross(pi, w);
          st6<RC>(s3 + a * 6 * ST, ST, Sa);
        }
      } else if (fl & TDS_LF_PRISMATIC) {
        const V3<RC> d = mul(Ri, ax);
        pi = axpy(d, qi, pi);
        S.bot = d;
      } else {
        const V3<RC> w = mul(Ri, ax);          // the joint axis is invariant under X_J
        if (jt == TDSJ_REVOLUTE_AXIS) {        // TinyQuaternion::setRotation(axis, angle), tiny_quaternion.h:178-183
          const RC dl = sqrt_t(dot(ax, ax));
          RC s, c;
          sincos_t(qi * RC(0.5), &s, &c);
          s = s / dl;
          Ri = mul(Ri, quat_to_matrix<RC>(ax.x * s, ax.y * s, ax.z * s, c));
        } else {
          RC s, c;
          sincos_t(qi, &s, &c);
          const V3<RC> cx = col_x(Ri), cy = col_y(Ri), cz = col_z(Ri);
          if (jt == TDSJ_REVOLUTE_X) set_cols(Ri, cx, axpy(cz, s, cy * c), axpy(cy, -s, cz * c));          // y' = c y + s z, z' = -s y + c z
          else if (jt == TDSJ_REVOLUTE_Y) set_cols(Ri, axpy(cz, -s, cx * c), cy, axpy(cx, s, cz * c));     // x' = c x - s z, z' = s x + c z
          else set_cols(Ri, axpy(cy, s, cx * c), axpy(cx, -s, cy * c), cz);                                 // x' = c x + s y, y' = -s x + c y
        }
        S.top = w;
        S.bot = cross(pi, w);
      }
    }
    st6<RC>(Sw + i * 6 * ST, ST, S);
    if (M.xw_slot[i] >= 0) { RC* px = A.ptr<RC>(M.x_xw + (M.xw_slot[i] + 1) * 12 * RCW); st9<RC>(px, ST, Ri); st3<RC>(px + 9 * ST, ST, pi); }
    // rigid-body inertia about O in world axes: com c = p_i + R_i com_l, I = R Icom R^T + m (|c|^2 1 - c c^T)
    {
      const double* rb = M.rbic[i];
      Rbi<RC> r;
      r.m = RC(rb[0]);
      const V3<RC> c = pi + mul(Ri, v3<RC>(RC(rb[1]), RC(rb[2]), RC(rb[3])));
      r.h = c * r.m;
      // R Icom R^T enters every product additively (no cancellation) -> RA precision is enough; the parallel-axis
      // terms m(|c|^2 1 - c c^T) and h = m c cancel against each other in M_ij and stay in RC.
      S3<RA> Icf; Icf.xx = RA(rb[4]); Icf.xy = RA(rb[5]); Icf.xz = RA(rb[6]); Icf.yy = RA(rb[7]); Icf.yz = RA(rb[8]); Icf.zz = RA(rb[9]);
      const S3<RA> Irot = rot_sym(cvt<RA>(Ri), Icf);
      r.I.xx = RC(Irot.xx); r.I.xy = RC(Irot.xy); r.I.xz = RC(Irot.xz); r.I.yy = RC(Irot.yy); r.I.yz = RC(Irot.yz); r.I.zz = RC(Irot.zz);
      const RC cc = dot(c, c);
      r.I.xx += r.m * (cc - c.x * c.x); r.I.yy += r.m * (cc - c.y * c.y); r.I.zz += r.m * (cc - c.z * c.z);
      r.I.xy -= r.m * c.x * c.y; r.I.xz -= r.m * c.x * c.z; r.I.yz -= r.m * c.y * c.z;
      st_rbi<RC>(A.ptr<RC>(M.x_link + i * LWD), ST, r);
    }
    Sv<RA> v = vp;
    if (fl & TDS_LF_SPHERICAL) {
      for (int a = 0; a < 3; ++a) {
        const RA qda = RA(qdv[(M.qd_idx[i] + a) * ST]);
        const Sv<RA> Sf = cvt_sv<RA>(S_col(i, a));
        v.top = axpy(Sf.top, qda, v.top);
        v.bot = axpy(Sf.bot, qda, v.bot);
      }
    } else if (!(fl & TDS_LF_FIXED)) {
      const RA qdi = RA(qdv[M.qd_idx[i] * ST]);
      const Sv<RA> Sf = cvt_sv<RA>(S);
      v.top = axpy(Sf.top, qdi, v.top);
      v.bot = axpy(Sf.bot, qdi, v.bot);
    }
    st6<RA>(A.ptr<RA>(M.x_link + i * LWD + VOFF), ST, v);
    if (want_contacts) emit_geoms(i, Ri, pi);
    if (io.link_xf && live) {
      float* o = io.link_xf + (size_t)i * 12 * ns + e;
      o[0] = (float)val_of(Ri.xx); o[(size_t)1 * ns] = (float)val_of(Ri.xy); o[(size_t)2 * ns] = (float)val_of(Ri.xz);
      o[(size_t)3 * ns] = (float)val_of(Ri.yx); o[(size_t)4 * ns] = (float)val_of(Ri.yy); o[(size_t)5 * ns] = (float)val_of(Ri.yz);
      o[(size_t)6 * ns] = (float)val_of(Ri.zx); o[(size_t)7 * ns] = (float)val_of(Ri.zy); o[(size_t)8 * ns] = (float)val_of(Ri.zz);
      o[(size_t)9 * ns] = (float)val_of(pi.x + O.x); o[(size_t)10 * ns] = (float)val_of(pi.y + O.y); o[(size_t)11 * ns] = (float)val_of(pi.z + O.z);
    }
    R_prev = Ri; p_prev = pi; v_prev = v;
  }
  // ---- contacts between the multibodies of the world (world.hpp:206-282), group = ordered pair of multibodies -----------------------
  // contact_sphere_sphere (contact_point.hpp:44-94) on sphere centres / capsule end spheres (contact_capsule_sphere, :406-438);
  // sphere A x capsule B goes through the dispatcher's swapped call (:478-492): points exchanged, normal negated.
  // Record: point on a [3] (relative to O), normal on b [3], distance, link a, link b; point on b = point on a - distance * normal.
  int pgc[TDS_MAX_PAIR_GROUPS];
  int n_pair_active = 0;
  if (want_contacts && M.n_pair_points > 0) {
    for (int g = 0; g < M.n_pair_groups; ++g) {
      int cnt = 0;
      for (int pt = M.pg_begin[g]; pt < M.pg_begin[g + 1]; ++pt) {
        const int ga = M.pp_ga[pt], gb = M.pp_gb[pt], kind = M.pp_kind[pt];
        const RC* wa = A.ptr<RC>(M.x_gw + M.g_wslot[ga] * 12 * RCW);
        const RC* wb = A.ptr<RC>(M.x_gw + M.g_wslot[gb] * 12 * RCW);
        if (kind >= 100) {
          // a PLANE shape on a link x point k of the other multibody's sphere / capsule / box: contact_plane_sphere
          // (contact_point.hpp:97-124) on the sphere, the capsule's end spheres (+L/2, -L/2) or the box's corner spheres (x outermost);
          // plane constant 0, world-frame normal as given - the pose of the plane's link is not used; a point is always emitted
          const bool swapped = kind >= 200;                      // the plane is on b: points exchanged, normal negated (:478-492)
          const int gp = swapped ? gb : ga, go = swapped ? ga : gb, k = kind - (swapped ? 200 : 100);
          const RC* wo = swapped ? wa : wb;
          const V3<RC> pnrm = v3<RC>(RC(M.g_half[gp][0]), RC(M.g_half[gp][1]), RC(M.g_half[gp][2]));
          V3<RC> c = ld3<RC>(wo, ST);
          const int to = M.g_type[go];
          if (to == TDSG_CAPSULE) c = k == 0 ? c + ld3<RC>(wo + 3 * ST, ST) : c - ld3<RC>(wo + 3 * ST, ST);
          else if (to == TDSG_BOX) {
            const V3<RC> ex = ld3<RC>(wo + 3 * ST, ST), ey = ld3<RC>(wo + 6 * ST, ST), ez = ld3<RC>(wo + 9 * ST, ST);
            c = (k & 4) ? c - ex : c + ex;
            c = (k & 2) ? c - ey : c + ey;
            c = (k & 1) ? c - ez : c + ez;
          }
          const RC rad = RC(M.g_radius[go]);
          const RC t = dot(c + O, pnrm);                         // -(dot(position, -normal) + constant), constant = 0
          const RC dist = t - rad;
          if (io.contact_dist && live) io.contact_dist[(size_t)(pt_index + pt) * ns + e] = (float)val_of(dist);
          if (dist < RC(0)) {
            RC* pr = A.ptr<RC>(M.x_pcon + n_pair_active * 9 * RCW);
            if (!swapped) { st3<RC>(pr, ST, c - pnrm * t); st3<RC>(pr + 3 * ST, ST, v3<RC>(-pnrm.x, -pnrm.y, -pnrm.z)); }   // point on the plane, normal on b = -n
            else { st3<RC>(pr, ST, c - pnrm * rad); st3<RC>(pr + 3 * ST, ST, pnrm); }                                        // point on the sphere, normal = +n
            pr[6 * ST] = dist;
            pr[7 * ST] = RC(M.g_link[ga]);
            pr[8 * ST] = RC(M.g_link[gb]);
            ++n_pair_active; ++cnt;
          }
          continue;
        }
        V3<RC> ca = ld3<RC>(wa, ST), cb = ld3<RC>(wb, ST);
        if (kind == 1) ca = ca + ld3<RC>(wa + 3 * ST, ST); else if (kind == -1) ca = ca - ld3<RC>(wa + 3 * ST, ST);
        if (kind == 2) cb = cb + ld3<RC>(wb + 3 * ST, ST); else if (kind == -2) cb = cb - ld3<RC>(wb + 3 * ST, ST);
        const bool swapped = kind == 2 || kind == -2;          // the contact function ran with (capsule on b, sphere on a)
        const RC r1 = RC(swapped ? M.g_radius[gb] : M.g_radius[ga]), r2 = RC(swapped ? M.g_radius[ga] : M.g_radius[gb]);
        const V3<RC> diff = swapped ? cb - ca : ca - cb;       // poseA.position - poseB.position of the call
        const RC len = sqrt_t(dot(diff, diff));
        const RC dist = len - (r1 + r2);
        // candidate distances behind the plane candidates; +inf: the contact function emitted no point (centres closer than CONTACT_EPSILON)
        if (io.contact_dist && live) io.contact_dist[(size_t)(pt_index + pt) * ns + e] = len > RC(1e-5) ? (float)val_of(dist) : __int_as_float(0x7f800000);
        if (len > RC(1e-5) && dist < RC(0)) {                  // CONTACT_EPSILON; resolve_collision keeps distance < 0 (the others are zero rows)
          const V3<RC> nrm = diff * (RC(1) / len);
          const V3<RC> p1 = (swapped ? cb : ca) - nrm * r1;    // point_a_world of the call
          RC* pr = A.ptr<RC>(M.x_pcon + n_pair_active * 9 * RCW);
          if (swapped) { st3<RC>(pr, ST, p1 - nrm * dist); st3<RC>(pr + 3 * ST, ST, v3<RC>(-nrm.x, -nrm.y, -nrm.z)); }
          else { st3<RC>(pr, ST, p1); st3<RC>(pr + 3 * ST, ST, nrm); }
          pr[6 * ST] = dist;
          pr[7 * ST] = RC(M.g_link[ga]);
          pr[8 * ST] = RC(M.g_link[gb]);
          ++n_pair_active; ++cnt;
        }
      }
      pgc[g] = cnt;
    }
  }
  const bool any_contact = __any_sync(0xffffffffu, n_active > 0 || n_pair_active > 0);
  TDSW_PHASE();  // 2

  // ---- pass 2: leaf -> root.  ABA (forward_dynamics.hpp:50-216) + CRBA (mass_matrix.hpp:39-125) ----------
  if (any_contact) {
    const int nblk = nb * (nb + 1) / 2 * 9;
    for (int k = 0; k < nblk; ++k) Mb[k * ST] = RS(0);
    for (int k = n; k < n3; ++k) Mb[(btri(k / 3, k / 3) + (k % 3) * 4) * ST] = RS(1);   // padding dofs: identity
  }
  Abi<RA> cA; Sv<RA> cP; Rbi<RC> cC;
  // M(r, c) = S_c . F for every dof column c of the ancestors of link i (and of the floating base), F = Ic S_r
  // (mass_matrix.hpp:58-111); r > c always: links are ordered parent first
  auto Mset = [&](int r, int c, RS val) { Mb[(btri(r / 3, c / 3) + (r % 3) * 3 + (c % 3)) * ST] = val; };
  auto crba_ancestors = [&](int i, int row, const Sv<RC>& F) {
    for (int j = M.parent[i]; j >= 0; j = M.parent[j]) {
      const int nc = n_cols(j);
      for (int c = 0; c < nc; ++c) Mset(row, M.qd_idx[j] + c, RS(dot(S_col(j, c), F)));
    }
    if (M.floating) {  // base columns: F in the base frame (:107-111); O is the base origin
      const V3<RC> ft = mulT(Rb, F.top), fb = mulT(Rb, F.bot);
      Mset(row, 0, RS(ft.x)); Mset(row, 1, RS(ft.y)); Mset(row, 2, RS(ft.z));
      Mset(row, 3, RS(fb.x)); Mset(row, 4, RS(fb.y)); Mset(row, 5, RS(fb.z));
    }
  };
  // Ia -= a b^T in the block form of the 1-dof update below (I: top-top, H: top-bot, M: bot-bot)
  auto abi_sub_outer = [&](Abi<RA>& Ia, const Sv<RA>& a, const Sv<RA>& b) {
    Ia.I.xx -= a.top.x * b.top.x; Ia.I.xy -= a.top.x * b.top.y; Ia.I.xz -= a.top.x * b.top.z;
    Ia.I.yy -= a.top.y * b.top.y; Ia.I.yz -= a.top.y * b.top.z; Ia.I.zz -= a.top.z * b.top.z;
    Ia.H.xx -= a.top.x * b.bot.x; Ia.H.xy -= a.top.x * b.bot.y; Ia.H.xz -= a.top.x * b.bot.z;
    Ia.H.yx -= a.top.y * b.bot.x; Ia.H.yy -= a.top.y * b.bot.y; Ia.H.yz -= a.top.y * b.bot.z;
    Ia.H.zx -= a.top.z * b.bot.x; Ia.H.zy -= a.top.z * b.bot.y; Ia.H.zz -= a.top.z * b.bot.z;
    Ia.M.xx -= a.bot.x * b.bot.x; Ia.M.xy -= a.bot.x * b.bot.y; Ia.M.xz -= a.bot.x * b.bot.z;
    Ia.M.yy -= a.bot.y * b.bot.y; Ia.M.yz -= a.bot.y * b.bot.z; Ia.M.zz -= a.bot.z * b.bot.z;
  };
  for (int i = n_links - 1; i >= 0; --i) {
    const int p = M.parent[i];
    const int fl = M.flags[i];
    RC* const rec = A.ptr<RC>(M.x_link + i * LWD);
    RA* const vrec = A.ptr<RA>(M.x_link + i * LWD + VOFF);
    Rbi<RC> Ic = ld_rbi<RC>(rec, ST);
    const Rbi<RA> rb = cvt_rbi<RA>(Ic);
    const Sv<RA> v = ld6<RA>(vrec, ST);
    Abi<RA> Ia = abi_from_rbi(rb);
    Sv<RA> pA = cross_mf(v, rbi_mul(rb, v));                 // kinematics.hpp:132
    if (fl & TDS_LF_CHILD_ADJ) { abi_add(Ia, cA); pA = pA + cP; rbi_add(Ic, cC); }
    if (M.acc_slot[i] >= 0) {
      Abi<RA> sa; Sv<RA> sp;
      acc_ld27<RA>(A.ptr<RA>(M.x_acc + M.acc_slot[i] * M.x_acc_words), ST, sa, sp);
      abi_add(Ia, sa); pA = pA + sp;
      rbi_add(Ic, ld_rbi<RC>(A.ptr<RC>(M.x_acc + M.acc_slot[i] * M.x_acc_words + M.x_acc_ic_word), ST));
    }
    Sv<RA> pa = pA;
    // U (6), invD, u overwrite the rigid-inertia record.  The RA and RC views interleave lanes differently, so
    // every lane must have finished reading its RC record before any lane writes the RA view.
    __syncwarp();
    RA* const urec = A.ptr<RA>(M.x_link + i * LWD);
    if (fl & TDS_LF_FIXED) {
      Sv<RA> z; z.top = v3<RA>(RA(0), RA(0), RA(0)); z.bot = z.top;
      st6<RA>(vrec, ST, z);
      st6<RA>(urec, ST, z);
      urec[6 * ST] = RA(0); urec[7 * ST] = RA(0);
    } else if (fl & TDS_LF_SPHERICAL) {
      // 3-dof joint (forward_dynamics.hpp:56-109): U = Ia S, D = S^T U (3 x 3), u = tau - damping qd - S^T pA,
      // Ia -= U D^-1 U^T, pa = pA + Ia c + U D^-1 u.  Record: U (18) | D^-1 (9) | u (3), then c.
      const int d0 = M.qd_idx[i];
      Sv<RC> Sd[3]; Sv<RA> S[3], U[3];
      RA qdj[3];
      Sv<RA> vJ; vJ.top = v3<RA>(RA(0), RA(0), RA(0)); vJ.bot = vJ.top;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        Sd[a] = S_col(i, a); S[a] = cvt_sv<RA>(Sd[a]);
        qdj[a] = RA(qdv[(d0 + a) * ST]);
        vJ.top = axpy(S[a].top, qdj[a], vJ.top); vJ.bot = axpy(S[a].bot, qdj[a], vJ.bot);
        U[a] = abi_mul(Ia, S[a]);
      }
      const Sv<RA> c = cross_mm(v, vJ);                      // kinematics.hpp:96-97
      RA Dm[3][3], u[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = 0; b < 3; ++b) Dm[a][b] = dot(S[a], U[b]);
        u[a] = RA(tauv[(d0 + a) * ST]) - RA(M.damping[i]) * qdj[a] - dot(S[a], pA);
      }
      if (M.stiffness[i] != 0.f) {   // tau -= stiffness * quaternion_axis_angle(q), forward_dynamics.hpp:69-74, tiny_algebra.hpp:509-527
        const int q0 = M.q_idx[i];
        const RC qx = RC(qv[q0 * ST]), qy = RC(qv[(q0 + 1) * ST]), qz = RC(qv[(q0 + 2) * ST]), qw = RC(qv[(q0 + 3) * ST]);
        const RC nrm = sqrt_t(qx * qx + qy * qy + qz * qz);
        const RC theta = RC(2) * atan2_t(nrm, qw);
        const RC scaling = nrm < RC(1.220703125e-4) ? RC(1) / (RC(0.5) + theta * theta * RC(1.0 / 48.0)) : theta / nrm;   // eps^(1/4)
        const RA k = RA(M.stiffness[i]);
        u[0] -= k * RA(scaling * qx); u[1] -= k * RA(scaling * qy); u[2] -= k * RA(scaling * qz);
      }
      RA Di[3][3];   // general 3 x 3 inverse (Matrix3::inverse)
      {
        const RA c0 = Dm[1][1] * Dm[2][2] - Dm[1][2] * Dm[2][1], c1 = Dm[1][2] * Dm[2][0] - Dm[1][0] * Dm[2][2], c2 = Dm[1][0] * Dm[2][1] - Dm[1][1] * Dm[2][0];
        const RA sdet = RA(1) / (Dm[0][0] * c0 + Dm[0][1] * c1 + Dm[0][2] * c2);
        Di[0][0] = c0 * sdet; Di[0][1] = (Dm[0][2] * Dm[2][1] - Dm[0][1] * Dm[2][2]) * sdet; Di[0][2] = (Dm[0][1] * Dm[1][2] - Dm[0][2] * Dm[1][1]) * sdet;
        Di[1][0] = c1 * sdet; Di[1][1] = (Dm[0][0] * Dm[2][2] - Dm[0][2] * Dm[2][0]) * sdet; Di[1][2] = (Dm[0][2] * Dm[1][0] - Dm[0][0] * Dm[1][2]) * sdet;
        Di[2][0] = c2 * sdet; Di[2][1] = (Dm[0][1] * Dm[2][0] - Dm[0][0] * Dm[2][1]) * sdet; Di[2][2] = (Dm[0][0] * Dm[1][1] - Dm[0][1] * Dm[1][0]) * sdet;
      }
      st6<RA>(vrec, ST, c);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        st6<RA>(urec + a * 6 * ST, ST, U[a]);
#pragma unroll
        for (int b = 0; b < 3; ++b) urec[(18 + a * 3 + b) * ST] = Di[a][b];
        urec[(27 + a) * ST] = u[a];
      }
      Sv<RA> V[3];   // V = U D^-1
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        V[b].top = U[0].top * Di[0][b] + U[1].top * Di[1][b] + U[2].top * Di[2][b];
        V[b].bot = U[0].bot * Di[0][b] + U[1].bot * Di[1][b] + U[2].bot * Di[2][b];
      }
#pragma unroll
      for (int b = 0; b < 3; ++b) abi_sub_outer(Ia, V[b], U[b]);
      const Sv<RA> Iac = abi_mul(Ia, c);
      pa.top = pA.top + Iac.top + V[0].top * u[0] + V[1].top * u[1] + V[2].top * u[2];
      pa.bot = pA.bot + Iac.bot + V[0].bot * u[0] + V[1].bot * u[1] + V[2].bot * u[2];
      if (any_contact) {   // mass_matrix.hpp:58-84
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const Sv<RC> F = rbi_mul(Ic, Sd[a]);
          for (int b = 0; b <= a; ++b) Mset(d0 + a, d0 + b, RS(dot(Sd[b], F)));
          crba_ancestors(i, d0 + a, F);
        }
      }
    } else {
      const Sv<RC> Sd = ld6<RC>(Sw + i * 6 * ST, ST);
      const Sv<RA> S = cvt_sv<RA>(Sd);
      const int qdi = M.qd_idx[i];
      const RA qdj = RA(qdv[qdi * ST]);
      Sv<RA> vJ; vJ.top = S.top * qdj; vJ.bot = S.bot * qdj;
      const Sv<RA> c = cross_mm(v, vJ);                      // kinematics.hpp:96-97
      const Sv<RA> U = abi_mul(Ia, S);                       // forward_dynamics.hpp:111
      const RA D = dot(S, U);
      const RA invD = RA(1) / D;
      RA tau = RA(tauv[qdi * ST]);
      tau -= RA(M.stiffness[i]) * RA(qv[M.q_idx[i] * ST]);
      tau -= RA(M.damping[i]) * qdj;
      const RA u = tau - dot(S, pA);                         // :129
      st6<RA>(vrec, ST, c);
      st6<RA>(urec, ST, U);
      urec[6 * ST] = invD; urec[7 * ST] = u;
      const V3<RA> ut = U.top * invD, ub = U.bot * invD;     // Ia -= U (U/D)^T, :160-168
      Ia.I.xx -= U.top.x * ut.x; Ia.I.xy -= U.top.x * ut.y; Ia.I.xz -= U.top.x * ut.z;
      Ia.I.yy -= U.top.y * ut.y; Ia.I.yz -= U.top.y * ut.z; Ia.I.zz -= U.top.z * ut.z;
      Ia.H.xx -= U.top.x * ub.x; Ia.H.xy -= U.top.x * ub.y; Ia.H.xz -= U.top.x * ub.z;
      Ia.H.yx -= U.top.y * ub.x; Ia.H.yy -= U.top.y * ub.y; Ia.H.yz -= U.top.y * ub.z;
      Ia.H.zx -= U.top.z * ub.x; Ia.H.zy -= U.top.z * ub.y; Ia.H.zz -= U.top.z * ub.z;
      Ia.M.xx -= U.bot.x * ub.x; Ia.M.xy -= U.bot.x * ub.y; Ia.M.xz -= U.bot.x * ub.z;
      Ia.M.yy -= U.bot.y * ub.y; Ia.M.yz -= U.bot.y * ub.z; Ia.M.zz -= U.bot.z * ub.z;
      const Sv<RA> Iac = abi_mul(Ia, c);                     // :171
      const RA uD = u * invD;
      pa.top = pA.top + Iac.top + U.top * uD;                // :173
      pa.bot = pA.bot + Iac.bot + U.bot * uD;
      if (any_contact) {   // CRBA column, mass_matrix.hpp:86-111: M_ij = S_j . (Ic_i S_i), no transforms needed
        const Sv<RC> F = rbi_mul(Ic, Sd);
        Mset(qdi, qdi, RS(dot(Sd, F)));
        crba_ancestors(i, qdi, F);
      }
    }
    // hand (Ia, pa, Ic) to the parent: plain sums in the common frame
    if (fl & TDS_LF_PARENT_ADJ) { cA = Ia; cP = pa; cC = Ic; }
    else {
      const int slot = (p >= 0) ? M.acc_slot[p] : M.base_acc;
      if (slot >= 0) {
        acc_add27<RA>(A.ptr<RA>(M.x_acc + slot * M.x_acc_words), ST, Ia, pa);
        rbi_acc<RC>(A.ptr<RC>(M.x_acc + slot * M.x_acc_words + M.x_acc_ic_word), ST, Ic);
      }
    }
  }
  TDSW_PHASE();  // 3

  // ---- base acceleration (forward_dynamics.hpp:218-243) ----------------------------------------------------
  Sv<RA> a_prev;
  Sv<RC> base_acc_b;   // base-frame value of the reference (floating) - needed for qdd[0:6]
  base_acc_b.top = v3<RC>(RC(0), RC(0), RC(0)); base_acc_b.bot = base_acc_b.top;
  if (M.floating) {
    // children sums in the common frame -> base frame (pure rotation: O is the base origin)
    Abi<RA> Ach; Sv<RA> pch; Rbi<RC> Icch;
    Ach.I = {RA(0), RA(0), RA(0), RA(0), RA(0), RA(0)}; Ach.M = Ach.I;
    Ach.H.xx = Ach.H.xy = Ach.H.xz = Ach.H.yx = Ach.H.yy = Ach.H.yz = Ach.H.zx = Ach.H.zy = Ach.H.zz = RA(0);
    pch.top = v3<RA>(RA(0), RA(0), RA(0)); pch.bot = pch.top;
    Icch.m = RC(0); Icch.h = v3<RC>(RC(0), RC(0), RC(0)); Icch.I = {RC(0), RC(0), RC(0), RC(0), RC(0), RC(0)};
    if (n_links > 0 && M.parent[0] < 0) { abi_add(Ach, cA); pch = pch + cP; rbi_add(Icch, cC); }
    if (M.base_acc >= 0) {
      Abi<RA> sa; Sv<RA> sp;
      acc_ld27<RA>(A.ptr<RA>(M.x_acc + M.base_acc * M.x_acc_words), ST, sa, sp);
      abi_add(Ach, sa); pch = pch + sp;
      rbi_add(Icch, ld_rbi<RC>(A.ptr<RC>(M.x_acc + M.base_acc * M.x_acc_words + M.x_acc_ic_word), ST));
    }
    const M3<RA> Rt = cvt<RA>(transpose(Rb));
    Abi<RA> Ab;
    {
      Rbi<RA> rbb = model_rbi_of<RA>(M.base_rbi);
      Ab = abi_from_rbi(rbb);
      Abi<RA> Arot;
      Arot.I = rot_sym(Rt, Ach.I); Arot.M = rot_sym(Rt, Ach.M); Arot.H = rot_gen(Rt, Ach.H);
      abi_add(Ab, Arot);
    }
    Sv<RA> pb;
    {
      // gyroscopic bias, kinematics.hpp:54-61 (reference mixes frames here; reproduced as written)
      const M3<RA> RbA = cvt<RA>(Rb);
      M3<RA> Ic0;
      Ic0.xx = RA(M.base_inertia_com[0]); Ic0.xy = RA(M.base_inertia_com[1]); Ic0.xz = RA(M.base_inertia_com[2]);
      Ic0.yx = RA(M.base_inertia_com[3]); Ic0.yy = RA(M.base_inertia_com[4]); Ic0.yz = RA(M.base_inertia_com[5]);
      Ic0.zx = RA(M.base_inertia_com[6]); Ic0.zy = RA(M.base_inertia_com[7]); Ic0.zz = RA(M.base_inertia_com[8]);
      const M3<RA> Iw = rot_gen(RbA, Ic0);
      const V3<RA> wb = v3<RA>(RA(qdv[0]), RA(qdv[ST]), RA(qdv[2 * ST]));
      pb.top = cross(wb, mul(Iw, wb)) + mul(Rt, pch.top);
      pb.bot = mul(Rt, pch.bot);
    }
    if (any_contact) {  // mass_matrix.hpp:114-120: base block = composite inertia in the base frame
      Rbi<RC> Ib = model_rbi_of<RC>(M.base_rbi);
      const M3<RC> RtC = transpose(Rb);
      Rbi<RC> rot; rot.m = Icch.m; rot.h = mul(RtC, Icch.h); rot.I = rot_sym(RtC, Icch.I);
      rbi_add(Ib, rot);
      const RS z = RS(0);
      RS* b00 = Mb + btri(0, 0) * ST; RS* b10 = Mb + btri(1, 0) * ST; RS* b11 = Mb + btri(1, 1) * ST;
      b00[0] = RS(Ib.I.xx); b00[3 * ST] = RS(Ib.I.xy); b00[4 * ST] = RS(Ib.I.yy); b00[6 * ST] = RS(Ib.I.xz); b00[7 * ST] = RS(Ib.I.yz); b00[8 * ST] = RS(Ib.I.zz);
      // rows 3..5, cols 0..2: H^T with H = h x
      b10[0] = z;               b10[ST] = RS(Ib.h.z);      b10[2 * ST] = RS(-Ib.h.y);
      b10[3 * ST] = RS(-Ib.h.z); b10[4 * ST] = z;           b10[5 * ST] = RS(Ib.h.x);
      b10[6 * ST] = RS(Ib.h.y);  b10[7 * ST] = RS(-Ib.h.x); b10[8 * ST] = z;
      b11[0] = RS(Ib.m); b11[3 * ST] = z; b11[4 * ST] = RS(Ib.m); b11[6 * ST] = z; b11[7 * ST] = z; b11[8 * ST] = RS(Ib.m);
    }
    // -base_abi.inv_mul(bias) with the reference's block inverse (C = -H), inertia.hpp:302-328
    {
      M3<RC> I3, H3, M3m;
      I3.xx = Ab.I.xx; I3.xy = Ab.I.xy; I3.xz = Ab.I.xz; I3.yx = Ab.I.xy; I3.yy = Ab.I.yy; I3.yz = Ab.I.yz; I3.zx = Ab.I.xz; I3.zy = Ab.I.yz; I3.zz = Ab.I.zz;
      H3 = cvt<RC>(Ab.H);
      M3m.xx = Ab.M.xx; M3m.xy = Ab.M.xy; M3m.xz = Ab.M.xz; M3m.yx = Ab.M.xy; M3m.yy = Ab.M.yy; M3m.yz = Ab.M.yz; M3m.zx = Ab.M.xz; M3m.zy = Ab.M.yz; M3m.zz = Ab.M.zz;
      auto inv3 = [](const M3<RC>& m) {
        M3<RC> o;
        RC c0 = m.yy * m.zz - m.yz * m.zy, c1 = m.yz * m.zx - m.yx * m.zz, c2 = m.yx * m.zy - m.yy * m.zx;
        RC s = RC(1) / (m.xx * c0 + m.xy * c1 + m.xz * c2);
        o.xx = c0 * s; o.xy = (m.xz * m.zy - m.xy * m.zz) * s; o.xz = (m.xy * m.yz - m.xz * m.yy) * s;
        o.yx = c1 * s; o.yy = (m.xx * m.zz - m.xz * m.zx) * s; o.yz = (m.xz * m.yx - m.xx * m.yz) * s;
        o.zx = c2 * s; o.zy = (m.xy * m.zx - m.xx * m.zy) * s; o.zz = (m.xx * m.yy - m.xy * m.yx) * s;
        return o;
      };
      auto neg = [](M3<RC> m) { m.xx = -m.xx; m.xy = -m.xy; m.xz = -m.xz; m.yx = -m.yx; m.yy = -m.yy; m.yz = -m.yz; m.zx = -m.zx; m.zy = -m.zy; m.zz = -m.zz; return m; };
      auto sub = [](M3<RC> a, const M3<RC>& b) { a.xx -= b.xx; a.xy -= b.xy; a.xz -= b.xz; a.yx -= b.yx; a.yy -= b.yy; a.yz -= b.yz; a.zx -= b.zx; a.zy -= b.zy; a.zz -= b.zz; return a; };
      auto add = [](M3<RC> a, const M3<RC>& b) { a.xx += b.xx; a.xy += b.xy; a.xz += b.xz; a.yx += b.yx; a.yy += b.yy; a.yz += b.yz; a.zx += b.zx; a.zy += b.zy; a.zz += b.zz; return a; };
      M3<RC> Ainv = inv3(I3);
      M3<RC> C = neg(H3);
      M3<RC> D = inv3(sub(M3m, mul(mul(C, Ainv), H3)));
      M3<RC> AinvBD = mul(mul(Ainv, H3), D);
      M3<RC> Ii = add(Ainv, mul(mul(AinvBD, C), Ainv));
      M3<RC> Hi = neg(AinvBD);
      V3<RC> ft = cvt<RC>(pb.top), fb = cvt<RC>(pb.bot);
      V3<RC> at = mul(Ii, ft) + mul(Hi, fb);
      V3<RC> ab = mul(D, fb) + mulT(Hi, ft);
      base_acc_b.top = v3<RC>(-at.x, -at.y, -at.z);
      base_acc_b.bot = v3<RC>(-ab.x, -ab.y, -ab.z);
    }
    a_prev.top = cvt<RA>(mul(Rb, base_acc_b.top));
    a_prev.bot = cvt<RA>(mul(Rb, base_acc_b.bot));
  } else {
    a_prev.top = v3<RA>(RA(0), RA(0), RA(0));
    a_prev.bot = v3<RA>(RA(-P.gravity[0]), RA(-P.gravity[1]), RA(-P.gravity[2]));
  }
  const Sv<RA> a_base = a_prev;
  const RA dtA = RA(P.dt);

  // ---- pass 3: root -> leaf (forward_dynamics.hpp:245-302) + integrate_euler_qdd (integrator.hpp:141-195) ----
  for (int i = 0; i < n_links; ++i) {
    const int p = M.parent[i];
    const int fl = M.flags[i];
    RA* const vrec = A.ptr<RA>(M.x_link + i * LWD + VOFF);
    Sv<RA> a;
    if (fl & TDS_LF_PARENT_ADJ) a = a_prev;
    else if (p >= 0) a = ld6<RA>(A.ptr<RA>(M.x_link + p * LWD + VOFF), ST);
    else a = a_base;
    if (fl & TDS_LF_SPHERICAL) {   // forward_dynamics.hpp:272-284: qdd = D^-1 (u - U^T a)
      const RA* urec = A.ptr<RA>(M.x_link + i * LWD);
      const int d0 = M.qd_idx[i];
      a = a + ld6<RA>(vrec, ST);
      RA t[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) t[k] = urec[(27 + k) * ST] - dot(ld6<RA>(urec + k * 6 * ST, ST), a);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const RA qdd = urec[(18 + j * 3) * ST] * t[0] + urec[(18 + j * 3 + 1) * ST] * t[1] + urec[(18 + j * 3 + 2) * ST] * t[2];
        const Sv<RA> S = cvt_sv<RA>(S_col(i, j));
        a.top = axpy(S.top, qdd, a.top);
        a.bot = axpy(S.bot, qdd, a.bot);
        if (mode == MODE_FD) {
          if constexpr (AD) { if (live) emit_row(d0 + j, qdd.d); }
          else if (live && io.qdd_out) io.qdd_out[(size_t)(d0 + j) * ns + e] = (float)val_of(qdd);
        } else if (!world_step) qdv[(d0 + j) * ST] = RQ(RA(qdv[(d0 + j) * ST]) + qdd * dtA);
      }
    } else if (!(fl & TDS_LF_FIXED)) {
      const RA* urec = A.ptr<RA>(M.x_link + i * LWD);
      const Sv<RA> c = ld6<RA>(vrec, ST);
      const Sv<RA> U = ld6<RA>(urec, ST);
      a = a + c;
      const RA qdd = urec[6 * ST] * (urec[7 * ST] - dot(U, a));
      const Sv<RA> S = cvt_sv<RA>(ld6<RC>(Sw + i * 6 * ST, ST));
      a.top = axpy(S.top, qdd, a.top);
      a.bot = axpy(S.bot, qdd, a.bot);
      const int qdi = M.qd_idx[i];
      if (mode == MODE_FD) {
        if constexpr (AD) { if (live) emit_row(qdi, qdd.d); }
        else if (live && io.qdd_out) io.qdd_out[(size_t)qdi * ns + e] = (float)val_of(qdd);
      } else if (!world_step) qdv[qdi * ST] = RQ(RA(qdv[qdi * ST]) + qdd * dtA);
    }
    st6<RA>(vrec, ST, a);
    a_prev = a;
  }
  if (M.floating) {  // forward_dynamics.hpp:317-322 (gravity added un-rotated), integrator.hpp:153-163
    const RC qb[6] = {base_acc_b.top.x, base_acc_b.top.y, base_acc_b.top.z, base_acc_b.bot.x + RC(P.gravity[0]),
                      base_acc_b.bot.y + RC(P.gravity[1]), base_acc_b.bot.z + RC(P.gravity[2])};
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      if (mode == MODE_FD) {
        if constexpr (AD) { if (live) emit_row(k, qb[k].d); }
        else if (live && io.qdd_out) io.qdd_out[(size_t)k * ns + e] = (float)val_of(qb[k]);
      } else if (!world_step) qdv[k * ST] = RQ(RC(qdv[k * ST]) + qb[k] * RC(P.dt));
    }
  }
  TDSW_PHASE();  // 4
  if (mode == MODE_FD) {
    if constexpr (AD) { if (live) store_vjp(); }
    return;
  }

  // ---- contact solve -------------------------------------------------------------------------------------------
  __syncwarp();   // the Y rows below reuse the per-link records with another lane interleave
  if ((mode == MODE_FULL || world_step) && any_contact) {
    // blocked Cholesky M = L L^T (3x3 blocks, lower): off-diagonal blocks of L overwrite M, diagonal blocks are
    // kept as their inverses.  (The reference inverts M, tiny_matrix_x.h:240-344; only M^-1 products are needed.)
    for (int bi = 0; bi < nb; ++bi) {
      for (int bj = 0; bj <= bi; ++bj) {
        B9<RS> Ab = ldb<RS>(Mb + btri(bi, bj) * ST, ST);
        for (int bk = 0; bk < bj; ++bk)
          gemm_nt_sub(Ab, ldb<RS>(Mb + btri(bi, bk) * ST, ST), ldb<RS>(Mb + btri(bj, bk) * ST, ST));
        if (bj < bi) stb<RS>(Mb + btri(bi, bj) * ST, ST, mul_linvT(Ab, ldl6<RS>(dinv + bj * 6 * ST, ST)));
        else stl6<RS>(dinv + bi * 6 * ST, ST, chol3_inv(Ab));
      }
    }
    TDSW_PHASE();  // 5
    const V3<RC> nbv = v3<RC>(-pn.x, -pn.y, -pn.z);                     // world_normal_on_b of every plane contact
    const V3<RC> f1 = v3<RC>(RC(M.fr1[0]), RC(M.fr1[1]), RC(M.fr1[2]));
    const V3<RC> f2 = v3<RC>(RC(M.fr2[0]), RC(M.fr2[1]), RC(M.fr2[2]));
    // One LCP per list of World::mb_contacts_, solved one after the other, each from the velocities the previous one left
    // (world.hpp:351-355).  Group 0: every plane contact (the plane is multibody 0; its lists (plane, b) share no dof, so
    // their Gauss-Seidel sweeps do not see each other and one LCP over all of them is the same arithmetic).  Groups 1..: the
    // pairs of multibodies (a, b) in lexicographic order, rows J_b - J_a over the dofs of both.
    int pbase = 0;   // first record of the current pair group
    for (int grp = 0; grp <= M.n_pair_groups; ++grp) {
    const int n_act = grp == 0 ? n_active : pgc[grp - 1];
    const RC* const prec = A.ptr<RC>(M.x_pcon + pbase * 9 * RCW);       // records of this pair group
    if (grp > 0) pbase += n_act;
    const int max_active = __reduce_max_sync(0xffffffffu, n_act);
    if (max_active == 0) {
      if (grp == 0) { TDSW_PHASE(); TDSW_PHASE(); }
      continue;
    }
    for (int c = 0; c < max_active; ++c) {
      if (c < n_act) {
        if (grp == 0) {
          const RC* pc = A.ptr<RC>(M.x_con + c * 5 * RCW);
          RS* const Y = A.ptr<RS>(M.x_Y) + c * n3 * 3 * ST;       // [dof k][rhs] : element (3k + rhs)
          const V3<RC> xc = ld3<RC>(pc, ST);
          const RC dist = pc[3 * ST];
          const int L = (int)val_of(pc[4 * ST]);
          for (int k = 0; k < 3 * n3; ++k) Y[k * ST] = RS(0);
          V3<RC> vel = v3<RC>(RC(0), RC(0), RC(0));                  // vel_b = J qd
          if (M.floating) {  // jacobian.hpp:39-58 with r = x_c (O is the base origin)
            const V3<RC> cols[6] = {v3<RC>(RC(0), -xc.z, xc.y), v3<RC>(xc.z, RC(0), -xc.x), v3<RC>(-xc.y, xc.x, RC(0)),
                                    v3<RC>(RC(1), RC(0), RC(0)), v3<RC>(RC(0), RC(1), RC(0)), v3<RC>(RC(0), RC(0), RC(1))};
  #pragma unroll
            for (int k = 0; k < 6; ++k) {
              Y[(3 * k) * ST] = RS(dot(nbv, cols[k])); Y[(3 * k + 1) * ST] = RS(dot(f1, cols[k])); Y[(3 * k + 2) * ST] = RS(dot(f2, cols[k]));
              vel = vel + cols[k] * RC(qdv[k * ST]);
            }
          }
          for (int j = L; j >= 0; j = M.parent[j]) {  // jacobian.hpp:63-80: column = S_j evaluated at the contact point
            const int nc = n_cols(j);
            for (int cj = 0; cj < nc; ++cj) {
              const Sv<RC> S = S_col(j, cj);
              const V3<RC> col = S.bot + cross(S.top, xc);
              const int qj = M.qd_idx[j] + cj;
              Y[(3 * qj) * ST] = RS(dot(nbv, col)); Y[(3 * qj + 1) * ST] = RS(dot(f1, col)); Y[(3 * qj + 2) * ST] = RS(dot(f2, col));
              vel = vel + col * RC(qdv[qj * ST]);
            }
          }
          // rel_vel = vel_a - vel_b = -vel ; mb_constraint_solver.hpp:299-345
          RS* const cs = A.ptr<RS>(M.x_conS) + c * 6 * ST;   // b[3], x[3]
          if (P.contact_model == 1) cs[0] = RS(dot(nbv, vel));   // spring-damper: approach speed n_b . v_b
          else cs[0] = RS((RC(1) + RC(P.restitution)) * dot(nbv, vel) - RC(P.erp) * dist / RC(P.dt));
          cs[ST] = RS(dot(f1, vel));
          cs[2 * ST] = RS(dot(f2, vel));
          cs[3 * ST] = RS(0); cs[4 * ST] = RS(0); cs[5 * ST] = RS(0);
        } else {
          // a contact between two multibodies: point on a / on b at the links la / lb, normal on b, friction directions of
          // plane_space(normal) (mb_constraint_solver.hpp:359-363, 506-520)
          const RC* pc = prec + c * 9 * ST;
          RS* const Y = A.ptr<RS>(M.x_Y) + c * n3 * 3 * ST;
          const V3<RC> xa = ld3<RC>(pc, ST), nrm = ld3<RC>(pc + 3 * ST, ST);
          const RC dist = pc[6 * ST];
          const int la = (int)val_of(pc[7 * ST]), lb = (int)val_of(pc[8 * ST]);
          const V3<RC> xb = xa - nrm * dist;
          V3<RC> g1, g2;
          plane_space_t(nrm, g1, g2);
          for (int k = 0; k < 3 * n3; ++k) Y[k * ST] = RS(0);
          V3<RC> vel = v3<RC>(RC(0), RC(0), RC(0));                  // vel_b - vel_a = -rel_vel
          for (int j = lb; j >= 0; j = M.parent[j]) {
            const int nc = n_cols(j);
            for (int cj = 0; cj < nc; ++cj) {
              const Sv<RC> S = S_col(j, cj);
              const V3<RC> col = S.bot + cross(S.top, xb);
              const int qj = M.qd_idx[j] + cj;
              Y[(3 * qj) * ST] = RS(dot(nrm, col)); Y[(3 * qj + 1) * ST] = RS(dot(g1, col)); Y[(3 * qj + 2) * ST] = RS(dot(g2, col));
              vel = vel + col * RC(qdv[qj * ST]);
            }
          }
          for (int j = la; j >= 0; j = M.parent[j]) {
            const int nc = n_cols(j);
            for (int cj = 0; cj < nc; ++cj) {
              const Sv<RC> S = S_col(j, cj);
              const V3<RC> col = S.bot + cross(S.top, xa);
              const int qj = M.qd_idx[j] + cj;
              Y[(3 * qj) * ST] = RS(-dot(nrm, col)); Y[(3 * qj + 1) * ST] = RS(-dot(g1, col)); Y[(3 * qj + 2) * ST] = RS(-dot(g2, col));
              vel = vel - col * RC(qdv[qj * ST]);
            }
          }
          RS* const cs = A.ptr<RS>(M.x_conS) + c * 6 * ST;   // b[3], x[3]
          if (P.contact_model == 1) cs[0] = RS(dot(nrm, vel));
          else cs[0] = RS((RC(1) + RC(P.restitution)) * dot(nrm, vel) - RC(P.erp) * dist / RC(P.dt));
          cs[ST] = RS(dot(g1, vel));
          cs[2 * ST] = RS(dot(g2, vel));
          cs[3 * ST] = RS(0); cs[4 * ST] = RS(0); cs[5 * ST] = RS(0);
        }
        RS* const Y = A.ptr<RS>(M.x_Y) + c * n3 * 3 * ST;
        // Y <- L^-1 Y (blocked forward substitution, 3 right-hand sides)
        for (int bi = 0; bi < nb; ++bi) {
          B9<RS> a = ldb<RS>(Y + bi * 9 * ST, ST);
          for (int bk = 0; bk < bi; ++bk) gemm_nn_sub(a, ldb<RS>(Mb + btri(bi, bk) * ST, ST), ldb<RS>(Y + bk * 9 * ST, ST));
          stb<RS>(Y + bi * 9 * ST, ST, linv_mul(ldl6<RS>(dinv + bi * 6 * ST, ST), a));
        }
      }
    }
    if (grp == 0) TDSW_PHASE();  // 6
    // matrix-free projected Gauss-Seidel on w = Y p; row order normals | friction-1 | friction-2
    // (solve_pgs, mb_constraint_solver.hpp:101-142; bounds :417-436)
    for (int k = 0; k < n3; ++k) wv[k * ST] = RS(0);
    const RS cfm = RS(P.cfm), mu = RS(P.friction);
    if (P.contact_model == 1) {
      // Spring-damper law instead of the LCP (DESIGN.md "Spring-damper contacts"; parity unpinned): closed-form impulses
      //   p_n = dt max(0, k x^n + d x^n xdot),  x = -distance, xdot = n_b . v_b
      //   p_t = dt mu f_n tanh(|v_t| / v_transition) v_t / |v_t|   along the two friction directions
      // accumulated into w = Y p like the Gauss-Seidel impulses; the back substitution below is shared.
      for (int c = 0; c < max_active; ++c) {
        if (c < n_act) {
          const RS* cs = A.ptr<RS>(M.x_conS) + c * 6 * ST;
          const RS x = RS(-(grp == 0 ? A.ptr<RC>(M.x_con + c * 5 * RCW)[3 * ST] : prec[(c * 9 + 6) * ST]));
          const RS vn = cs[0], v1 = cs[ST], v2 = cs[2 * ST];
          const RS xn = pow_t(x, RS(P.exponent_n));
          RS fn = RS(P.spring_k) * xn + RS(P.damper_d) * xn * vn;
          if (P.hard_contact_condition && fn < RS(0)) fn = RS(0);
          const RS vt = sqrt_t(v1 * v1 + v2 * v2);
          const RS sc = vt > RS(1e-12) ? mu * fn * tanh_t(vt / RS(P.v_transition)) / vt * RS(P.dt) : RS(0);
          const RS p[3] = {fn * RS(P.dt), sc * v1, sc * v2};
          const RS* y = A.ptr<RS>(M.x_Y) + (c * n3 * 3) * ST;
          for (int k = 0; k < n3; ++k)
            wv[k * ST] += p[0] * y[(3 * k) * ST] + p[1] * y[(3 * k + 1) * ST] + p[2] * y[(3 * k + 2) * ST];
        }
      }
    } else
    for (int it = 0; it < P.pgs_iterations; ++it) {
      for (int blk = 0; blk < 3; ++blk) {
        for (int c = 0; c < max_active; ++c) {
          if (c < n_act) {
            RS* const cs = A.ptr<RS>(M.x_conS) + c * 6 * ST;
            const RS* y = A.ptr<RS>(M.x_Y) + (c * n3 * 3 + blk) * ST;     // element k at y[3k * ST]
            RS yy0 = RS(0), yy1 = RS(0), yy2 = RS(0), yw0 = RS(0), yw1 = RS(0), yw2 = RS(0);
            for (int b = 0; b < nb; ++b) {
              const RS y0 = y[(9 * b) * ST], y1 = y[(9 * b + 3) * ST], y2 = y[(9 * b + 6) * ST];
              yy0 += y0 * y0; yy1 += y1 * y1; yy2 += y2 * y2;
              yw0 += y0 * wv[(3 * b) * ST]; yw1 += y1 * wv[(3 * b + 1) * ST]; yw2 += y2 * wv[(3 * b + 2) * ST];
            }
            const RS yy = (yy0 + yy1) + yy2, yw = (yw0 + yw1) + yw2;
            const RS x_old = cs[(3 + blk) * ST];
            RS x = (cs[blk * ST] - yw + yy * x_old) / (yy + cfm);
            if (blk == 0) {
              x = x < RS(0) ? RS(0) : x;
              x = x > RS(100000) ? RS(100000) : x;
            } else {
              RS s = cs[3 * ST];
              s = s < RS(0) ? RS(0) : s;
              const RS lim = mu * s;
              x = x < -lim ? -lim : x;
              x = x > lim ? lim : x;
            }
            cs[(3 + blk) * ST] = x;
            const RS dx = x - x_old;
            for (int b = 0; b < nb; ++b) {
              wv[(3 * b) * ST] += dx * y[(9 * b) * ST];
              wv[(3 * b + 1) * ST] += dx * y[(9 * b + 3) * ST];
              wv[(3 * b + 2) * ST] += dx * y[(9 * b + 6) * ST];
            }
          }
        }
      }
    }
    if (grp == 0) TDSW_PHASE();  // 7
    // qd_b -= M^-1 Jc^T p = L^-T w   (mb_constraint_solver.hpp:476-497), blocked back substitution
    for (int bi = nb - 1; bi >= 0; --bi) {
      RS a0 = wv[(3 * bi) * ST], a1 = wv[(3 * bi + 1) * ST], a2 = wv[(3 * bi + 2) * ST];
      for (int bk = bi + 1; bk < nb; ++bk) {
        const B9<RS> Lb = ldb<RS>(Mb + btri(bk, bi) * ST, ST);
        const RS z0 = wv[(3 * bk) * ST], z1 = wv[(3 * bk + 1) * ST], z2 = wv[(3 * bk + 2) * ST];
        a0 -= Lb.a[0] * z0 + Lb.a[3] * z1 + Lb.a[6] * z2;
        a1 -= Lb.a[1] * z0 + Lb.a[4] * z1 + Lb.a[7] * z2;
        a2 -= Lb.a[2] * z0 + Lb.a[5] * z1 + Lb.a[8] * z2;
      }
      const L6<RS> li = ldl6<RS>(dinv + bi * 6 * ST, ST);
      const RS z0 = li.i00 * a0 + li.i10 * a1 + li.i20 * a2;
      const RS z1 = li.i11 * a1 + li.i21 * a2;
      const RS z2 = li.i22 * a2;
      wv[(3 * bi) * ST] = z0; wv[(3 * bi + 1) * ST] = z1; wv[(3 * bi + 2) * ST] = z2;
    }
    if (n_act > 0)
      for (int k = 0; k < n; ++k) qdv[k * ST] = RQ(RS(qdv[k * ST]) - wv[k * ST]);
    }   // groups
  }
  TDSW_PHASE();  // 8

  // ---- integrate_euler with qdd = 0 (integrator.hpp:10-133) -----------------------------------------------------
  RC up_z = RC(1);
  if (M.floating && !world_step) {
    const RC h = RC(0.5) * RC(P.dt);
    RC qx = RC(qv[0]), qy = RC(qv[ST]), qz = RC(qv[2 * ST]), qw = RC(qv[3 * ST]);
    const RC w0 = RC(qdv[0]), w1 = RC(qdv[ST]), w2 = RC(qdv[2 * ST]);
    const RC dw = (-qx * w0 - qy * w1 - qz * w2) * h;
    const RC dx = (qw * w0 + qz * w1 - qy * w2) * h;
    const RC dy = (qw * w1 + qx * w2 - qz * w0) * h;
    const RC dz = (qw * w2 + qy * w0 - qx * w1) * h;
    qx += dx; qy += dy; qz += dz; qw += dw;
    const RC len = sqrt_t(qx * qx + qy * qy + qz * qz + qw * qw);
    qx /= len; qy /= len; qz /= len; qw /= len;
    qv[0] = RQ(qx); qv[ST] = RQ(qy); qv[2 * ST] = RQ(qz); qv[3 * ST] = RQ(qw);
    for (int k = 0; k < 3; ++k)
      qv[(4 + k) * ST] = RQ(RC(qv[(4 + k) * ST]) + RC(qdv[(3 + k) * ST]) * RC(P.dt));
    up_z = RC(1) - RC(2) * (qx * qx + qy * qy) / (qx * qx + qy * qy + qz * qz + qw * qw);
  }
  for (int i = 0; i < n_links && !world_step; ++i) {
    if (M.flags[i] & TDS_LF_FIXED) continue;
    if (M.flags[i] & TDS_LF_SPHERICAL) {
      // integrator.hpp:97-122: the joint velocity is damped by MultiBody::joint_damping_ ^ (1000 dt) (default 0.995,
      // multi_body.hpp:51) in every integrate_euler, then q += quat_velocity_spherical(q, qd, dt), normalised
      const int q0 = M.q_idx[i], d0 = M.qd_idx[i];
      const RC damp = RC(pow(0.995, P.dt * 1000.0));
      RC w[3];
      for (int k = 0; k < 3; ++k) { w[k] = RC(qdv[(d0 + k) * ST]) * damp; qdv[(d0 + k) * ST] = RQ(w[k]); }
      const RC h = RC(0.5) * RC(P.dt);
      RC qx = RC(qv[q0 * ST]), qy = RC(qv[(q0 + 1) * ST]), qz = RC(qv[(q0 + 2) * ST]), qw = RC(qv[(q0 + 3) * ST]);
      const RC dw = (-qx * w[0] - qy * w[1] - qz * w[2]) * h;      // tiny_algebra.hpp:616-627
      const RC dx = (qw * w[0] + qy * w[2] - qz * w[1]) * h;
      const RC dy = (qw * w[1] + qz * w[0] - qx * w[2]) * h;
      const RC dz = (qw * w[2] + qx * w[1] - qy * w[0]) * h;
      qx += dx; qy += dy; qz += dz; qw += dw;
      const RC len = sqrt_t(qx * qx + qy * qy + qz * qz + qw * qw);
      qv[q0 * ST] = RQ(qx / len); qv[(q0 + 1) * ST] = RQ(qy / len); qv[(q0 + 2) * ST] = RQ(qz / len); qv[(q0 + 3) * ST] = RQ(qw / len);
      continue;
    }
    const int qi = M.q_idx[i];
    qv[qi * ST] = RQ(RC(qv[qi * ST]) + RC(qdv[M.qd_idx[i] * ST]) * RC(P.dt));
  }

  // ---- reward / done / auto-reset, write back ------------------------------------------------------------------------
  if constexpr (AD) {   // the Jacobian column of this lane's direction / the output tangents / the VJP entry: rows q' | qd'
    if (live) {
      for (int k = 0; k < M.n_q; ++k) emit_row(k, qv[k * ST].d);
      for (int k = 0; k < n; ++k) emit_row(M.n_q + k, qdv[k * ST].d);
      store_vjp();
    }
    return;
  }
  if (live) {
    bool done = false;
    if (E.reward_kind == 1) {   // laikago_environment2.h:130-171 (fixed-base emulation)
      const float x = (float)val_of(qv[0]), z = (float)val_of(qv[2 * ST]);
      const float upz = cosf((float)val_of(qv[3 * ST])) * cosf((float)val_of(qv[4 * ST]));
      done = (upz < 0.6f) || (z < 0.2f);
      if (io.reward) io.reward[e] = done ? 0.f : x;
    } else if (E.reward_kind == 2) {
      const float x = (float)val_of(qv[4 * ST]), z = (float)val_of(qv[6 * ST]);
      done = ((float)val_of(up_z) < 0.6f) || (z < 0.2f);
      if (io.reward) io.reward[e] = done ? 0.f : x;
    } else if (E.reward_kind == 3) {   // ant_environment2.h:75-105: done = z < 0.26, reward = (x' - x)/dt, which integrate_euler makes the x velocity
      done = (float)val_of(qv[2 * ST]) < 0.26f;
      if (io.reward) io.reward[e] = done ? 0.f : (float)val_of(qdv[0]);
    }
    if (io.done && E.reward_kind) io.done[e] = done ? 1.f : 0.f;
    if (done && E.auto_reset) {   // ars_vectorized_environment.h:262-283
      for (int k = 0; k < M.n_q; ++k) io.q_out[(size_t)k * ns + e] = E.reset_q[k];
      for (int k = 0; k < n; ++k) io.qd_out[(size_t)k * ns + e] = 0.f;
    } else {
      for (int k = 0; k < M.n_q; ++k) io.q_out[(size_t)k * ns + e] = (float)val_of(qv[k * ST]);
      for (int k = 0; k < n; ++k) io.qd_out[(size_t)k * ns + e] = (float)val_of(qdv[k * ST]);
    }
  }
  TDSW_PHASE();  // 9
}

}  // namespace tdsw

#ifndef TDS_STEPW_KERNEL_ONLY   // (tests/cpp/stepw_host.cpp compiles the kernel above for the host, without the launchers)
extern "C" int tds_launch_stepw(const DevModel* M, const SimParams* P, const EnvParams* E, const StepIO* io,
                                int mode, int use_pd, int precision, char* gscratch, int use_smem,
                                int warps_per_block, cudaStream_t stream) {
  using namespace tdsw;
  const int threads = 32 * warps_per_block;
  const int blocks = (io->n + threads - 1) / threads;
  const size_t smem = use_smem ? (size_t)warps_per_block * M->x_total * 32 * 4 : 0;
  cudaError_t err = cudaSuccess;
#define TDSW_LAUNCH(RA, RC, RS, SM)                                                                     \
  do {                                                                                                  \
    auto k = tds_stepw_kernel<RA, RC, RS, float, SM>;                                                   \
    static size_t smem_set_dev[64] = {0}; int dev_ = 0; cudaGetDevice(&dev_); size_t& smem_set = smem_set_dev[dev_ & 63]; \
    if (smem > 48 * 1024 && smem > smem_set) {                                                          \
      err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
      if (err == cudaSuccess) smem_set = smem;                                                          \
    }                                                                                                   \
    if (err == cudaSuccess) {                                                                           \
      k<<<blocks, threads, smem, stream>>>(*M, *P, *E, *io, mode, use_pd, gscratch, DualIO());          \
      err = cudaGetLastError();                                                                         \
    }                                                                                                   \
  } while (0)
  if (precision == 0) { if (use_smem) TDSW_LAUNCH(float, double, float, true); else TDSW_LAUNCH(float, double, float, false); }
  else if (precision == 1) { if (use_smem) TDSW_LAUNCH(double, double, double, true); else TDSW_LAUNCH(double, double, double, false); }
  else { if (use_smem) TDSW_LAUNCH(float, float, float, true); else TDSW_LAUNCH(float, float, float, false); }
#undef TDSW_LAUNCH
  return (int)err;
}

// Differentiable step: the same kernel on forward-mode dual numbers (fp64).  M must carry the 16-byte layout
// (tds_build_layout_w(..., 16, 16, 16, -1, 16)); gscratch: n_dirs * ceil(n / 32) blocks of x_total * 128 bytes.
// Dense Jacobian (io->jac set) or VJP (dio->vjp_cot set): one lane per (environment, input direction) for directions
// [io->jac_dir0, io->jac_dir0 + n_dirs).  JVP (dio->jvp_out set): one lane per environment, n_dirs = 1.
extern "C" int tds_launch_stepw_dual(const DevModel* M, const SimParams* P, const EnvParams* E, const StepIO* io, const DualIO* dio,
                                     int mode, int use_pd, int n_dirs, char* gscratch, cudaStream_t stream) {
  using namespace tdsw;
  typedef tds::Dual<double> D;
  const dim3 grid((io->n + 31) / 32, n_dirs);
  tds_stepw_kernel<D, D, D, D, false><<<grid, 32, 0, stream>>>(*M, *P, *E, *io, mode, use_pd, gscratch, *dio);
  return (int)cudaGetLastError();
}
#endif  // TDS_STEPW_KERNEL_ONLY
