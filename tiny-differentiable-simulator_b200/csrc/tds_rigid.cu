// The RigidBody path of the reference's World (SURVEY 8f.3): maximal-coordinate rigid bodies with ONE collision shape each,
// sequential-impulse contact solver.  One lane per world; a batch of worlds steps in one launch.
//   World::step                                   src/world.hpp:293-363 (the rigid-body half: :302-318, :336-340, :361-363)
//   RigidBody::apply_gravity / apply_force_impulse / apply_impulse / integrate   src/rigid_body.hpp:84-118
//   World::compute_contacts_rigid_body_internal   src/world.hpp:166-195 (pairs i < j through the dispatcher)
//   CollisionDispatcher                           src/contact_point.hpp:445-506 (direct or swapped call)
//   contact_sphere_sphere / plane_sphere / plane_capsule / plane_box / capsule_sphere   src/contact_point.hpp:44-438
//   RigidBodyConstraintSolver::resolve_collision  src/rb_constraint_solver.hpp:66-163 (the non-CppAD branch)
// State per body, fp64 in HBM as [13 * n_bodies][n_stride]: position [3], orientation xyzw [4], linear velocity [3],
// angular velocity [3].  Everything of a world lives in the lane's registers / local memory: the path is latency-bound
// scalar work (50 Gauss-Seidel sweeps over a handful of contacts), its HBM traffic is 2 x 104 B per body and step call.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include "tds_math.cuh"
#include "tds_dual.cuh"
#include "tds_types.h"
#include "tds_b200_model.h"

#define TDS_RIGID_MAX_BODIES 16
#define TDS_RIGID_MAX_CONTACTS 48

struct RigidWorld {                       // constant for all worlds of a batch (kernel parameter)
  int n_bodies;
  int type[TDS_RIGID_MAX_BODIES];         // TDSG_SPHERE / TDSG_PLANE / TDSG_CAPSULE / TDSG_BOX
  double mass[TDS_RIGID_MAX_BODIES];
  double p[TDS_RIGID_MAX_BODIES][4];      // sphere: radius; capsule: radius, length; box: extents [3]; plane: normal [3], constant
  double dt, gravity[3], friction, restitution, erp;
  int num_solver_iterations;
};

// desc [n_bodies][6] = mass, shape (TDSG_*), p0..p3 -> RigidWorld (host).  The plane normal is normalised like Plane's constructor
// does (src/geometry.hpp:163-168).  Returns 0, -1 on an unknown shape, -2 when the contact list could overflow.
static inline int tds_rigid_world_from_desc(const double* desc, int n_bodies, RigidWorld* W) {
  memset(W, 0, sizeof(*W));
  W->n_bodies = n_bodies;
  for (int i = 0; i < n_bodies; ++i) {
    const double* d = desc + i * 6;
    const int t = (int)d[1];
    if (t != TDSG_SPHERE && t != TDSG_PLANE && t != TDSG_CAPSULE && t != TDSG_BOX) return -1;
    W->mass[i] = d[0]; W->type[i] = t;
    for (int k = 0; k < 4; ++k) W->p[i][k] = d[2 + k];
    if (t == TDSG_PLANE) {
      const double l = sqrt(d[2] * d[2] + d[3] * d[3] + d[4] * d[4]);
      for (int k = 0; k < 3; ++k) W->p[i][k] = d[2 + k] / l;
    }
  }
  // worst case of the contact list (every pair at the point count of its contact function): the kernel's list is fixed-size
  int worst = 0;
  for (int i = 0; i < n_bodies; ++i)
    for (int j = i + 1; j < n_bodies; ++j) {
      auto pts = [](int a, int b) { return (a == TDSG_SPHERE && b == TDSG_SPHERE) ? 1 : (a == TDSG_PLANE && b == TDSG_SPHERE) ? 1 : (a == TDSG_PLANE && b == TDSG_CAPSULE) ? 2
                                    : (a == TDSG_PLANE && b == TDSG_BOX) ? 8 : (a == TDSG_CAPSULE && b == TDSG_SPHERE) ? 2 : 0; };
      const int t = W->type[i], u = W->type[j];
      worst += pts(t, u) ? pts(t, u) : pts(u, t);
    }
  if (worst > TDS_RIGID_MAX_CONTACTS) return -2;
  // World defaults (world.hpp:65-72), RigidBodyConstraintSolver::erp_ (rb_constraint_solver.hpp:45)
  W->dt = 1.0 / 60.0; W->gravity[2] = -9.81; W->friction = 0.5; W->restitution = 0.0; W->erp = 0.1; W->num_solver_iterations = 1;
  return 0;
}

namespace tdsrb {
using namespace tds;

template <typename T> struct Contact { V3<T> n, ra, rb; T dist; int a, b; };   // normal on b, point - position of a / b

// contact_sphere_sphere (contact_point.hpp:44-94) between two spheres given by centre and radius; pa / pb: the bodies' positions
template <typename T>
TDS_D void sphere_sphere(const V3<T>& ca, T ra, const V3<T>& cb, T rb, Contact<T>* cs, int& nc, int a, int b, const V3<T>& pa,
                         const V3<T>& pb, bool swap) {
  const V3<T> diff = ca - cb;
  const T len = sqrt_t(dot(diff, diff));
  if (!(len > T(1e-5)) || nc >= TDS_RIGID_MAX_CONTACTS) return;   // CONTACT_EPSILON
  const T dist = len - (ra + rb);
  const V3<T> n = diff * (T(1) / len);
  const V3<T> point_a = ca - n * ra;
  const V3<T> point_b = point_a - n * dist;
  Contact<T>& c = cs[nc++];
  c.dist = dist;
  if (!swap) { c.n = n; c.ra = point_a - pa; c.rb = point_b - pb; c.a = a; c.b = b; }
  else { c.n = v3<T>(-n.x, -n.y, -n.z); c.ra = point_b - pb; c.rb = point_a - pa; c.a = b; c.b = a; }   // dispatcher :478-492
}

// contact_plane_sphere (contact_point.hpp:97-124): plane = body a (its pose is not used), sphere centre c
template <typename T>
TDS_D void plane_sphere(const V3<T>& pn, T pc, const V3<T>& c, T r, Contact<T>* cs, int& nc, int a, int b, const V3<T>& pa,
                        const V3<T>& pb, bool swap) {
  if (nc >= TDS_RIGID_MAX_CONTACTS) return;
  const V3<T> mn = v3<T>(-pn.x, -pn.y, -pn.z);
  const T t = -(dot(c, mn) + pc);
  const V3<T> point_a = c + mn * t;
  const V3<T> point_b = c - pn * r;
  Contact<T>& k = cs[nc++];
  k.dist = t - r;
  if (!swap) { k.n = mn; k.ra = point_a - pa; k.rb = point_b - pb; k.a = a; k.b = b; }
  else { k.n = pn; k.ra = point_b - pb; k.rb = point_a - pa; k.a = b; k.b = a; }
}

template <typename T, typename TS>
__global__ void __launch_bounds__(128) tds_rigid_step_kernel(const __grid_constant__ RigidWorld W, const TS* s_in,
                                                             TS* s_out, const TS* __restrict__ force, int steps,
                                                             int n, int ns, double* __restrict__ jac, int jac_dir0,
                                                             const DualIO dio = DualIO()) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  constexpr bool AD = is_dual<T>::value;
  const int dir = AD ? (int)blockIdx.y + jac_dir0 : -1;      // differentiable instance: input direction of this lane
  const int nb = W.n_bodies;
  // derivative part of input idx (blocks state 13 nb | force 3 nb): the caller's tangent (JVP), else d input_idx / d direction
  auto seed = [&](T x, int idx) -> T {
    if constexpr (AD) {
      if (dio.jvp_out) {
        const int blk = idx < 13 * nb ? 0 : 1, r = blk ? idx - 13 * nb : idx;
        x.d = dio.jvp_tan[blk] ? dio.jvp_tan[blk][(size_t)r * ns + e] : 0.0;
      } else if (idx == dir) x.d = 1.0;
    }
    return x;
  };
  V3<T> pos[TDS_RIGID_MAX_BODIES], lin[TDS_RIGID_MAX_BODIES], ang[TDS_RIGID_MAX_BODIES];
  T qx[TDS_RIGID_MAX_BODIES], qy[TDS_RIGID_MAX_BODIES], qz[TDS_RIGID_MAX_BODIES], qw[TDS_RIGID_MAX_BODIES];
  // input directions: the 13 * n_bodies state entries, then the 3 * n_bodies force entries
  for (int b = 0; b < nb; ++b) {
    auto ld = [&](int k) { return seed(T(s_in[(size_t)(b * 13 + k) * ns + e]), b * 13 + k); };
    pos[b] = v3<T>(ld(0), ld(1), ld(2));
    qx[b] = ld(3); qy[b] = ld(4); qz[b] = ld(5); qw[b] = ld(6);
    lin[b] = v3<T>(ld(7), ld(8), ld(9));
    ang[b] = v3<T>(ld(10), ld(11), ld(12));
  }
  const T dt = T(W.dt);
  Contact<T> cs[TDS_RIGID_MAX_CONTACTS];
  for (int s = 0; s < steps; ++s) {
    // apply_gravity, apply_force_impulse, clear_forces (rigid_body.hpp:84-101; the torque is always zero on this path)
    for (int b = 0; b < nb; ++b) {
      const T m = T(W.mass[b]);
      const T inv_m = W.mass[b] == 0.0 ? T(0) : T(1) / m;
      V3<T> f = v3<T>(m * T(W.gravity[0]), m * T(W.gravity[1]), m * T(W.gravity[2]));
      if (s == 0 && force) {
        const int f0 = 13 * nb + 3 * b;
        f = f + v3<T>(seed(T(force[(size_t)(3 * b) * ns + e]), f0), seed(T(force[(size_t)(3 * b + 1) * ns + e]), f0 + 1),
                      seed(T(force[(size_t)(3 * b + 2) * ns + e]), f0 + 2));
      }
      lin[b] = lin[b] + f * inv_m * dt;
    }
    // contacts of every pair i < j (world.hpp:166-195)
    int nc = 0;
    for (int i = 0; i < nb; ++i)
      for (int j = i + 1; j < nb; ++j) {
        int a = i, b = j;
        int ta = W.type[a], tb = W.type[b];
        // direct function f[ta][tb], else the swapped one f[tb][ta] with points exchanged and normal negated
        const bool direct = (ta == TDSG_SPHERE && tb == TDSG_SPHERE) || (ta == TDSG_PLANE && (tb == TDSG_SPHERE || tb == TDSG_CAPSULE || tb == TDSG_BOX)) ||
                            (ta == TDSG_CAPSULE && tb == TDSG_SPHERE);
        const bool swapped = !direct && ((tb == TDSG_PLANE && (ta == TDSG_SPHERE || ta == TDSG_CAPSULE || ta == TDSG_BOX)) || (tb == TDSG_CAPSULE && ta == TDSG_SPHERE));
        if (!direct && !swapped) continue;
        if (swapped) { a = j; b = i; ta = W.type[a]; tb = W.type[b]; }     // the function runs on (a, b) = (j, i)
        const M3<T> Rb = quat_to_matrix<T>(qx[b], qy[b], qz[b], qw[b]);
        if (ta == TDSG_SPHERE) {
          sphere_sphere(pos[a], T(W.p[a][0]), pos[b], T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
        } else if (ta == TDSG_CAPSULE) {   // contact_capsule_sphere: end spheres at +L/2, then -L/2
          const M3<T> Ra = quat_to_matrix<T>(qx[a], qy[a], qz[a], qw[a]);
          const V3<T> half = mul(Ra, v3<T>(T(0), T(0), T(0.5 * W.p[a][1])));
          sphere_sphere(pos[a] + half, T(W.p[a][0]), pos[b], T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
          sphere_sphere(pos[a] - half, T(W.p[a][0]), pos[b], T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
        } else {                           // plane x sphere / capsule / box
          const V3<T> pn = v3<T>(T(W.p[a][0]), T(W.p[a][1]), T(W.p[a][2]));
          const T pc = T(W.p[a][3]);
          if (tb == TDSG_SPHERE) plane_sphere(pn, pc, pos[b], T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
          else if (tb == TDSG_CAPSULE) {
            const V3<T> half = mul(Rb, v3<T>(T(0), T(0), T(0.5 * W.p[b][1])));
            plane_sphere(pn, pc, pos[b] + half, T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
            plane_sphere(pn, pc, pos[b] - half, T(W.p[b][0]), cs, nc, a, b, pos[a], pos[b], swapped);
          } else {                         // contact_plane_box: spheres of radius max(1e-2, 0) at the corners, x outermost
            const double r = 1e-2;
            const double dx = 0.5 * W.p[b][0] - r, dy = 0.5 * W.p[b][1] - r, dz = 0.5 * W.p[b][2] - r;
            for (int k = 0; k < 8; ++k) {
              const V3<T> corner = v3<T>(T((k & 4) ? -dx : dx), T((k & 2) ? -dy : dy), T((k & 1) ? -dz : dz));
              plane_sphere(pn, pc, pos[b] + mul(Rb, corner), T(r), cs, nc, a, b, pos[a], pos[b], swapped);
            }
          }
        }
      }
    // sequential impulses (world.hpp:336-340, rb_constraint_solver.hpp:113-160)
    for (int it = 0; it < W.num_solver_iterations; ++it)
      for (int c = 0; c < nc; ++c) {
        const Contact<T>& k = cs[c];
        if (!(k.dist < T(0))) continue;
        const int a = k.a, b = k.b;
        const T ima = W.mass[a] == 0.0 ? T(0) : T(1) / T(W.mass[a]), imb = W.mass[b] == 0.0 ? T(0) : T(1) / T(W.mass[b]);
        const T iia = W.mass[a] == 0.0 ? T(0) : T(1), iib = W.mass[b] == 0.0 ? T(0) : T(1);   // inv_inertia_world_: identity or zero (rigid_body.hpp:53-54)
        const T baumgarte = T(W.erp) * k.dist / dt;
        const V3<T> rel_vel = (lin[a] + cross(ang[a], k.ra)) - (lin[b] + cross(ang[b], k.rb));
        const T nrv = dot(k.n, rel_vel);
        if (!(nrv < T(0))) continue;
        const V3<T> t1 = cross(k.ra, k.n) * iia, t2 = cross(k.rb, k.n) * iib;
        const T angt = dot(k.n, cross(t1, k.ra) + cross(t2, k.rb));
        const T den = ima + imb + angt;
        const T impulse = (-(T(1) + T(W.restitution)) * nrv - baumgarte) / den;
        if (!(impulse > T(0))) continue;
        auto apply = [&](int body, const V3<T>& imp, const V3<T>& r, T im, T ii) {   // RigidBody::apply_impulse
          lin[body] = lin[body] + imp * im;
          ang[body] = ang[body] + cross(r, imp) * ii;
        };
        const V3<T> iv = k.n * impulse;
        apply(a, iv, k.ra, ima, iia);
        apply(b, v3<T>(-iv.x, -iv.y, -iv.z), k.rb, imb, iib);
        const V3<T> lat = rel_vel - k.n * nrv;             // (rel_vel from BEFORE the normal impulse, as the reference)
        const T lat_n = sqrt_t(dot(lat, lat));
        const T trial = lat_n / den;
        const T fi = trial < T(W.friction) * impulse ? trial : T(W.friction) * impulse;
        if (lat_n > T(1e-4)) {
          const V3<T> fd = lat * (T(1) / lat_n);
          apply(a, fd * (-fi), k.ra, ima, iia);
          apply(b, fd * fi, k.rb, imb, iib);
        }
      }
    // integrate (rigid_body.hpp:110-118; quat_velocity, tiny_algebra.hpp:604-614)
    for (int b = 0; b < nb; ++b) {
      pos[b] = pos[b] + lin[b] * dt;
      const T h = T(0.5) * dt;
      const V3<T> w = ang[b];
      const T dw = (-qx[b] * w.x - qy[b] * w.y - qz[b] * w.z) * h;
      const T dx = (qw[b] * w.x + qz[b] * w.y - qy[b] * w.z) * h;
      const T dy = (qw[b] * w.y + qx[b] * w.z - qz[b] * w.x) * h;
      const T dz = (qw[b] * w.z + qy[b] * w.x - qx[b] * w.y) * h;
      T x = qx[b] + dx, y = qy[b] + dy, z = qz[b] + dz, ww = qw[b] + dw;
      const T inv = T(1) / sqrt_t(x * x + y * y + z * z + ww * ww);
      qx[b] = x * inv; qy[b] = y * inv; qz[b] = z * inv; qw[b] = ww * inv;
    }
  }
  double vjp_acc = 0.0;   // VJP: sum_r cot_r * d out_r / d direction
  for (int b = 0; b < nb; ++b) {
    const T out[13] = {pos[b].x, pos[b].y, pos[b].z, qx[b], qy[b], qz[b], qw[b], lin[b].x, lin[b].y, lin[b].z, ang[b].x, ang[b].y, ang[b].z};
    for (int k = 0; k < 13; ++k) {
      if constexpr (AD) {
        const size_t r = (size_t)(b * 13 + k);
        if (jac) jac[(r * (16 * nb) + dir) * ns + e] = out[k].d;     // [row][column][world]
        if (dio.jvp_out) dio.jvp_out[r * ns + e] = out[k].d;
        if (dio.vjp_cot) vjp_acc += dio.vjp_cot[r * ns + e] * out[k].d;
        if (blockIdx.y == 0 && s_out) s_out[r * ns + e] = (TS)val_of(out[k]);
      } else {
        s_out[(size_t)(b * 13 + k) * ns + e] = (TS)out[k];
      }
    }
  }
  if constexpr (AD) {
    if (dio.vjp_cot) {
      const int blk = dir < 13 * nb ? 0 : 1, r = blk ? dir - 13 * nb : dir;
      if (dio.vjp_out[blk]) dio.vjp_out[blk][(size_t)r * ns + e] = vjp_acc;
    }
  }
}
}  // namespace tdsrb

#ifndef TDS_RIGID_KERNEL_ONLY   // (tests/cpp/rigid_host.cpp compiles the kernel above for the host)
#include <string>
#include <vector>

extern "C" void tds_b200_set_error(const char* msg);

struct tds_b200_rigid {
  RigidWorld W;
  int n = 0, ns = 0, device = 0;
  double *state = nullptr, *state2 = nullptr, *force = nullptr, *jac = nullptr;   // state2: output of the differentiable instance
  cudaStream_t stream = nullptr;
};

static int rigid_fail(const std::string& m, int rc) { tds_b200_set_error(m.c_str()); return rc; }
#define RB_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return rigid_fail(std::string(#expr) + ": " + cudaGetErrorString(e_), (int)e_); } while (0)

extern "C" {
// desc: [n_bodies][6] = mass, shape (TDSG_*), p0, p1, p2, p3 (see RigidWorld::p).  NULL on a refused description / no GPU.
tds_b200_rigid* tds_b200_rigid_create(const double* desc, int n_bodies, int n_worlds, int device) {
  if (!desc || n_bodies < 1 || n_bodies > TDS_RIGID_MAX_BODIES || n_worlds < 1) { tds_b200_set_error("rigid world: 1..16 bodies, >= 1 world"); return nullptr; }
  RigidWorld W0;
  const int rcw = tds_rigid_world_from_desc(desc, n_bodies, &W0);
  if (rcw == -1) { tds_b200_set_error("rigid world: shapes are sphere, plane, capsule, box"); return nullptr; }
  if (rcw == -2) { tds_b200_set_error("rigid world: more than 48 candidate contact points"); return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { tds_b200_set_error("cudaSetDevice failed"); return nullptr; }
  tds_b200_rigid* h = new tds_b200_rigid;
  h->W = W0;
  h->n = n_worlds; h->ns = (n_worlds + 31) & ~31; h->device = device;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMalloc((void**)&h->state, sizeof(double) * 13 * n_bodies * h->ns) != cudaSuccess ||
      cudaMalloc((void**)&h->force, sizeof(double) * 3 * n_bodies * h->ns) != cudaSuccess) {
    tds_b200_set_error("rigid world: allocation failed");
    cudaFree(h->state); cudaFree(h->force); if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return nullptr;
  }
  return h;
}

void tds_b200_rigid_destroy(tds_b200_rigid* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->state); cudaFree(h->state2); cudaFree(h->force); cudaFree(h->jac);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int tds_b200_rigid_set_params(tds_b200_rigid* h, double dt, const double* gravity, double friction, double restitution, double erp,
                              int num_solver_iterations) {
  if (!h || !gravity || !(dt > 0) || num_solver_iterations < 0) return rigid_fail("rigid_set_params: bad argument", -1);
  h->W.dt = dt; for (int k = 0; k < 3; ++k) h->W.gravity[k] = gravity[k];
  h->W.friction = friction; h->W.restitution = restitution; h->W.erp = erp; h->W.num_solver_iterations = num_solver_iterations;
  return 0;
}

// `steps` calls of World::step on device arrays [13 * n_bodies][n_stride] fp64 (n_stride = n_worlds rounded up to 32); force
// [3 * n_bodies][n_stride] or NULL = RigidBody::apply_central_force before the first step (forces are cleared by every step).
int tds_b200_rigid_step_device(tds_b200_rigid* h, const double* state_in, double* state_out, const double* force, int steps, void* stream) {
  if (!h || !state_in || !state_out || steps < 0) return rigid_fail("rigid_step_device: bad argument", -1);
  const int T = 128, B = (h->n + T - 1) / T;
  tdsrb::tds_rigid_step_kernel<double, double><<<B, T, 0, stream ? (cudaStream_t)stream : h->stream>>>(h->W, state_in, state_out, force, steps, h->n, h->ns, nullptr, 0);
  RB_TRY(cudaGetLastError());
  return 0;
}

static int rigid_upload(tds_b200_rigid* h, const double* state, const double* force) {
  const int nb = h->W.n_bodies, n = h->n, ns = h->ns;
  std::vector<double> t((size_t)13 * nb * ns, 0.0);
  for (int e = 0; e < n; ++e) for (int k = 0; k < 13 * nb; ++k) t[(size_t)k * ns + e] = state[(size_t)e * 13 * nb + k];
  for (int e = n; e < ns; ++e) for (int b = 0; b < nb; ++b) t[(size_t)(b * 13 + 6) * ns + e] = 1.0;
  RB_TRY(cudaMemcpyAsync(h->state, t.data(), sizeof(double) * t.size(), cudaMemcpyHostToDevice, h->stream));
  if (force) {
    std::vector<double> f((size_t)3 * nb * ns, 0.0);
    for (int e = 0; e < n; ++e) for (int k = 0; k < 3 * nb; ++k) f[(size_t)k * ns + e] = force[(size_t)e * 3 * nb + k];
    RB_TRY(cudaMemcpyAsync(h->force, f.data(), sizeof(double) * f.size(), cudaMemcpyHostToDevice, h->stream));
    RB_TRY(cudaStreamSynchronize(h->stream));
  }
  RB_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

// host arrays: state [n_worlds][n_bodies][13], force [n_worlds][n_bodies][3] or NULL, state_out like state
int tds_b200_rigid_step_host(tds_b200_rigid* h, const double* state, const double* force, int steps, double* state_out) {
  if (!h || !state || !state_out) return rigid_fail("rigid_step_host: bad argument", -1);
  RB_TRY(cudaSetDevice(h->device));
  int rc = rigid_upload(h, state, force);
  if (rc) return rc;
  rc = tds_b200_rigid_step_device(h, h->state, h->state, force ? h->force : nullptr, steps, h->stream);
  if (rc) return rc;
  const int nb = h->W.n_bodies, n = h->n, ns = h->ns;
  std::vector<double> t((size_t)13 * nb * ns);
  RB_TRY(cudaMemcpyAsync(t.data(), h->state, sizeof(double) * t.size(), cudaMemcpyDeviceToHost, h->stream));
  RB_TRY(cudaStreamSynchronize(h->stream));
  for (int e = 0; e < n; ++e) for (int k = 0; k < 13 * nb; ++k) state_out[(size_t)e * 13 * nb + k] = t[(size_t)k * ns + e];
  return 0;
}

// d state_out / d (state_in | force) by forward-mode dual numbers, one lane per (world, input direction):
// jac [n_worlds][13 * n_bodies][16 * n_bodies] (the billiard gradients of the reference's python/examples/billiard_optimization.py)
int tds_b200_rigid_jacobian_host(tds_b200_rigid* h, const double* state, const double* force, int steps, double* state_out, double* jac) {
  if (!h || !state || !jac) return rigid_fail("rigid_jacobian_host: bad argument", -1);
  RB_TRY(cudaSetDevice(h->device));
  const int nb = h->W.n_bodies, n = h->n, ns = h->ns, rows = 13 * nb, cols = 16 * nb;
  std::vector<double> zero_f;
  if (!force) { zero_f.assign((size_t)n * 3 * nb, 0.0); force = zero_f.data(); }
  int rc = rigid_upload(h, state, force);
  if (rc) return rc;
  if (!h->jac) RB_TRY(cudaMalloc((void**)&h->jac, sizeof(double) * (size_t)rows * cols * ns));
  if (!h->state2) RB_TRY(cudaMalloc((void**)&h->state2, sizeof(double) * (size_t)rows * ns));   // (the lanes of other directions still read the input)
  const int T = 128;
  dim3 grid((n + T - 1) / T, cols);
  tdsrb::tds_rigid_step_kernel<tds::Dual<double>, double><<<grid, T, 0, h->stream>>>(h->W, h->state, h->state2, h->force, steps, n, ns, h->jac, 0);
  RB_TRY(cudaGetLastError());
  std::vector<double> t((size_t)rows * cols * ns), so((size_t)rows * ns);
  RB_TRY(cudaMemcpyAsync(t.data(), h->jac, sizeof(double) * t.size(), cudaMemcpyDeviceToHost, h->stream));
  RB_TRY(cudaMemcpyAsync(so.data(), h->state2, sizeof(double) * so.size(), cudaMemcpyDeviceToHost, h->stream));
  RB_TRY(cudaStreamSynchronize(h->stream));
  for (int e = 0; e < n; ++e) {
    for (int k = 0; k < rows * cols; ++k) jac[(size_t)e * rows * cols + k] = t[(size_t)k * ns + e];
    if (state_out) for (int k = 0; k < rows; ++k) state_out[(size_t)e * rows + k] = so[(size_t)k * ns + e];
  }
  return 0;
}

// Products with d state_out / d (state | force) of `steps` steps, on device arrays in the layout of tds_b200_rigid_step_device; one
// lane carries its derivative through all the steps.  A null force is zero force (a requested force block then differentiates at 0).
static const double* rigid_force_or_zero(tds_b200_rigid* h, const double* force, bool needed, cudaStream_t sm) {
  if (force || !needed) return force;
  if (cudaMemsetAsync(h->force, 0, sizeof(double) * 3 * h->W.n_bodies * h->ns, sm) != cudaSuccess) return nullptr;
  return h->force;
}

int tds_b200_rigid_jvp_device(tds_b200_rigid* h, const double* state, const double* force, int steps, const double* t_state,
                              const double* t_force, double* t_out, void* stream) {
  if (!h || !state || !t_out || steps < 0) return rigid_fail("rigid_jvp_device: bad argument", -1);
  cudaStream_t sm = stream ? (cudaStream_t)stream : h->stream;
  force = rigid_force_or_zero(h, force, t_force != nullptr, sm);
  if (t_force && !force) return rigid_fail("rigid_jvp_device: zeroing the force failed", -1);
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  dio.jvp_tan[0] = t_state; dio.jvp_tan[1] = t_force; dio.jvp_out = t_out;
  const int T = 128;
  tdsrb::tds_rigid_step_kernel<tds::Dual<double>, double><<<(h->n + T - 1) / T, T, 0, sm>>>(h->W, state, nullptr, force, steps, h->n, h->ns,
                                                                                         nullptr, 0, dio);
  RB_TRY(cudaGetLastError());
  return 0;
}

int tds_b200_rigid_vjp_device(tds_b200_rigid* h, const double* state, const double* force, int steps, const double* g_out,
                              double* g_state, double* g_force, void* stream) {
  if (!h || !state || !g_out || steps < 0) return rigid_fail("rigid_vjp_device: bad argument", -1);
  cudaStream_t sm = stream ? (cudaStream_t)stream : h->stream;
  force = rigid_force_or_zero(h, force, g_force != nullptr, sm);
  if (g_force && !force) return rigid_fail("rigid_vjp_device: zeroing the force failed", -1);
  DualIO dio;
  memset(&dio, 0, sizeof(dio));
  dio.vjp_cot = g_out; dio.vjp_out[0] = g_state; dio.vjp_out[1] = g_force;
  const int T = 128, nb = h->W.n_bodies;
  // only the requested blocks are launched: directions [0, 13 nb) of the state, [13 nb, 16 nb) of the force
  if (g_state) {
    tdsrb::tds_rigid_step_kernel<tds::Dual<double>, double><<<dim3((h->n + T - 1) / T, 13 * nb), T, 0, sm>>>(
        h->W, state, nullptr, force, steps, h->n, h->ns, nullptr, 0, dio);
    RB_TRY(cudaGetLastError());
  }
  if (g_force) {
    tdsrb::tds_rigid_step_kernel<tds::Dual<double>, double><<<dim3((h->n + T - 1) / T, 3 * nb), T, 0, sm>>>(
        h->W, state, nullptr, force, steps, h->n, h->ns, nullptr, 13 * nb, dio);
    RB_TRY(cudaGetLastError());
  }
  return 0;
}
}  // extern "C"
#endif  // TDS_RIGID_KERNEL_ONLY
