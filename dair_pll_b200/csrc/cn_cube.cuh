// Single floating rigid body with one box geometry against the ground plane
// (assets/contactnets_cube.urdf): n_q = 7, n_v = 6, 4 contacts (top-4 of the 8 box
// corners, geometry.py:162-202, 487-491), k = 12.
//
// Replaces, per sample, what the reference computes with ~5.5k ATen calls:
//   LagrangianTerms.forward        multibody_terms.py:214-237   (M, M^-1 F)
//   ContactTerms.forward           multibody_terms.py:428-521   (phi, J)
//   collide_plane_convex / top-k   geometry.py:553-582, 162-202
//   contactnets_loss               multibody_learnable_system.py:104-197
//   forward_dynamics               multibody_learnable_system.py:199-304
//   SAPSolver.apply                (un-vendored; restated, see oracle/cone_qp.c)
//
// Internal velocity coordinates are the WORLD-frame twist u^ = [R w_B ; v_W]: in
// them a contact Jacobian is [-S(rho_c), I3] with rho_c the world-frame lever arm,
// so J u, J^T f and J^T K J reduce to cross products and no dense 12x6 J is ever
// formed; the mass matrix becomes [[R I_o R^T, m S(R c)], [-m S(R c), m I3]] and its
// inverse is closed-form (Schur complement = R I_sym R^T).  The QP is solved in
// primal (velocity) form:  min_u 1/2 u^T M u + eps/2 sum_c |Pi(-(D_mu J_c u + q_c)/eps)|^2
// by Newton with a derivative-based line search; f_c = Pi(...) at the optimum.
//
// Code-size discipline: the kernels are instruction-cache sensitive (warps of one SM run
// different phases), so per-contact work is written as loops over c whose unroll factor
// UNR is a template parameter: UNR = 1 (rolled) when the per-sample problem lives in a
// shared-memory slot (dynamic indexing is free there), UNR = 4 for register-resident use.
#pragma once
#include "cn_common.cuh"

#ifndef CN_STAT_LS
#define CN_STAT_LS()
#define CN_STAT_UNIT()
#endif

namespace cn {

constexpr int CUBE_NQ = 7, CUBE_NV = 6, CUBE_NX = 13, CUBE_NC = 4, CUBE_K = 12;
constexpr int CUBE_NPARAM = 14;      // [inertia 10 | mu_pair 1 | half_lengths 3]
constexpr int CUBE_PROB_FIELDS = 33; // IW 6 | mcW 3 | rho 12 | q 12

template <typename T> struct CubeParams {
  T m, c[3], Isym[6];   // the 10-vector the generated callables take (multibody_terms.py:198-205)
  T mu;                 // combined pair friction 2 mu_a mu_b/(mu_a+mu_b) (multibody_terms.py:471)
  T h[3];               // |length_params| (geometry.py:394-397)
  T dt, eps, inv_eps, grav;
  // derived
  T Io[6];              // I_sym - m S(c)^2  (inertia about the body origin)
  T Isym_inv[6];
  T inv_m;
  T dscale[6];          // 1/diag(M) in body coordinates, for the scaled stopping test
};

template <typename T>
CN_HD void cube_params_init(CubeParams<T>& P, const T* inertia, const T* mu, const T* half, T dt, T eps) {
  P.m = inertia[0];
  for (int i = 0; i < 3; ++i) P.c[i] = inertia[1 + i];
  for (int i = 0; i < 6; ++i) P.Isym[i] = inertia[4 + i];
  P.mu = mu[0];
  for (int i = 0; i < 3; ++i) P.h[i] = half[i];
  P.dt = dt; P.eps = eps; P.inv_eps = T(1) / eps; P.grav = T(9.81);
  const T cx = P.c[0], cy = P.c[1], cz = P.c[2], m = P.m;
  // -S(c)^2 = |c|^2 I - c c^T
  P.Io[0] = P.Isym[0] + m * (cy * cy + cz * cz);
  P.Io[1] = P.Isym[1] + m * (cx * cx + cz * cz);
  P.Io[2] = P.Isym[2] + m * (cx * cx + cy * cy);
  P.Io[3] = P.Isym[3] - m * cx * cy;
  P.Io[4] = P.Isym[4] - m * cx * cz;
  P.Io[5] = P.Isym[5] - m * cy * cz;
  sym3_inv(P.Isym, P.Isym_inv);
  P.inv_m = T(1) / m;
  P.dscale[0] = T(1) / P.Io[0]; P.dscale[1] = T(1) / P.Io[1]; P.dscale[2] = T(1) / P.Io[2];
  P.dscale[3] = P.dscale[4] = P.dscale[5] = P.inv_m;
}

// View of the per-sample quantities that stay fixed during the Newton solve: element k of
// the 33-field record at p[k * s].  s = 1 over a local array (registers), s = #slots over a
// shared-memory pool laid out field-major (bank-conflict-free across lanes).
template <typename T> struct CubeProb {
  T* p;
  int s;
  CN_HD T& IW(int i) const { return p[i * s]; }          // R Io R^T  [xx,yy,zz,xy,xz,yz]
  CN_HD T& mcW(int i) const { return p[(6 + i) * s]; }   // m R c
  CN_HD T& rho(int k) const { return p[(9 + k) * s]; }   // world lever arms, 3 per contact
  CN_HD T& q(int k) const { return p[(21 + k) * s]; }    // QP linear term, sappy order [tx,ty,n] per contact
};

// [aw; av] = M^-1 [tau; frc]  (tau, aw body frame; frc, av world frame); Schur complement = I_sym.
template <typename T>
CN_HD void cube_minv(const CubeParams<T>& P, const T* R, const T* tau, const T* frc, T* aw, T* av) {
  T fb[3], cxf[3], rhs[3], cxa[3], rc[3];
  rot3t(R, frc, fb);
  cross3(P.c, fb, cxf);
  for (int i = 0; i < 3; ++i) rhs[i] = tau[i] - cxf[i];
  sym3_mul(P.Isym_inv, rhs, aw);
  cross3(P.c, aw, cxa);
  rot3(R, cxa, rc);
  for (int i = 0; i < 3; ++i) av[i] = frc[i] * P.inv_m + rc[i];
}

// u^ -> M^ u^ in world-twist coordinates
template <typename T>
CN_HD void cube_mass_mul(const CubeParams<T>& P, const CubeProb<T>& S, const T* u, T* o) {
  const T I0 = S.IW(0), I1 = S.IW(1), I2 = S.IW(2), I3 = S.IW(3), I4 = S.IW(4), I5 = S.IW(5);
  const T mc[3] = {S.mcW(0), S.mcW(1), S.mcW(2)};
  T b[3], c[3];
  cross3(mc, u + 3, b);
  cross3(mc, u, c);
  o[0] = I0 * u[0] + I3 * u[1] + I4 * u[2] + b[0];
  o[1] = I3 * u[0] + I1 * u[1] + I5 * u[2] + b[1];
  o[2] = I4 * u[0] + I5 * u[1] + I2 * u[2] + b[2];
  for (int i = 0; i < 3; ++i) o[3 + i] = P.m * u[3 + i] - c[i];
}

// The 4 corners with the largest support d . (sigma o h) (top-k of the reference,
// geometry.py:191-197), in ascending vertex-index order (the reference's order is unspecified).
// Closed form: with a_k = |d_k| h_k sorted s <= m <= l, the support values in decreasing order
// are {none flipped, flip s, flip m, then flip s+m or flip l, whichever costs less}.
// Returns the 4 vertex indices (i = 4 x + 2 y + z with bit set = +h, geometry.py:39-41)
// packed 3 bits each, corner c at bits 3c..3c+2.
template <typename T> CN_HD uint32_t cube_select_corners(const T* d, const T* h) {
  const T a0 = t_abs(d[0]) * h[0], a1 = t_abs(d[1]) * h[1], a2 = t_abs(d[2]) * h[2];
  const uint32_t best = (d[0] >= T(0) ? 4u : 0u) | (d[1] >= T(0) ? 2u : 0u) | (d[2] >= T(0) ? 1u : 0u);
  const bool c01 = a0 <= a1, c12 = a1 <= a2, c02 = a0 <= a2;
  // axis of the smallest / largest a (ties towards the lower axis); axis k flips vertex bit 4 >> k
  const int is = c01 ? (c02 ? 0 : 2) : (c12 ? 1 : 2);
  const int il = c01 ? (c12 ? 2 : 1) : (c02 ? 2 : 0);
  const int im = 3 - is - il;
  const T lo01 = t_min(a0, a1), hi01 = t_max(a0, a1);
  const T as = t_min(lo01, a2), al = t_max(hi01, a2), am = t_max(lo01, t_min(hi01, a2));
  const uint32_t bs = 4u >> is, bm = 4u >> im, bl = 4u >> il;
  const uint32_t v3 = (as + am <= al) ? (best ^ bs ^ bm) : (best ^ bl);
  uint32_t mask = (1u << best) | (1u << (best ^ bs)) | (1u << (best ^ bm)) | (1u << v3);
  uint32_t sel = 0;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
#if defined(__CUDA_ARCH__)
    const uint32_t i = (uint32_t)(__ffs((int)mask) - 1);
#else
    const uint32_t i = (uint32_t)(__builtin_ffs((int)mask) - 1);
#endif
    mask &= mask - 1u;
    sel |= i << (3 * c);
  }
  return sel;
}

// sign (+1 / -1) of corner c of `sel` along axis (0 = x, 1 = y, 2 = z)
template <typename T> CN_HD T sgn_bit(uint32_t sel, int c, int axis) {
  return ((sel >> (3 * c + 2 - axis)) & 1u) ? T(1) : T(-1);
}

// Shared geometry set-up: R, world inertia, corner selection, lever arms (phi_c = rho_c,z + pos_z,
// geometry.py:568-571, is formed where it is used).
template <typename T, int UNR>
CN_HD void cube_geometry(const CubeParams<T>& P, const T* quat, T* R, uint32_t& sel, const CubeProb<T>& S) {
  quat_to_rot(quat, R);
  // IW = R Io R^T
  T A[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const T r0 = R[3 * i], r1 = R[3 * i + 1], r2 = R[3 * i + 2];
    A[3 * i + 0] = r0 * P.Io[0] + r1 * P.Io[3] + r2 * P.Io[4];
    A[3 * i + 1] = r0 * P.Io[3] + r1 * P.Io[1] + r2 * P.Io[5];
    A[3 * i + 2] = r0 * P.Io[4] + r1 * P.Io[5] + r2 * P.Io[2];
  }
  S.IW(0) = A[0] * R[0] + A[1] * R[1] + A[2] * R[2];
  S.IW(1) = A[3] * R[3] + A[4] * R[4] + A[5] * R[5];
  S.IW(2) = A[6] * R[6] + A[7] * R[7] + A[8] * R[8];
  S.IW(3) = A[0] * R[3] + A[1] * R[4] + A[2] * R[5];
  S.IW(4) = A[0] * R[6] + A[1] * R[7] + A[2] * R[8];
  S.IW(5) = A[3] * R[6] + A[4] * R[7] + A[5] * R[8];
  T cW[3];
  rot3(R, P.c, cW);
#pragma unroll
  for (int i = 0; i < 3; ++i) S.mcW(i) = P.m * cW[i];
  // support direction in the body frame: -(third row of R)  (geometry.py:560-564)
  const T d[3] = {-R[6], -R[7], -R[8]};
  sel = cube_select_corners(d, P.h);
  T Rh[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) Rh[3 * i + k] = R[3 * i + k] * P.h[k];
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    const T sx = sgn_bit<T>(sel, c, 0), sy = sgn_bit<T>(sel, c, 1), sz = sgn_bit<T>(sel, c, 2);
#pragma unroll
    for (int i = 0; i < 3; ++i) S.rho(3 * c + i) = sx * Rh[3 * i] + sy * Rh[3 * i + 1] + sz * Rh[3 * i + 2];
  }
}

// Contact-free acceleration M^-1 F at (R, w_B), in body(w)/world(v) state coordinates
// (closed form of the generated lagrangian_forces, see oracle/callables.py).
template <typename T>
CN_HD void cube_free_accel(const CubeParams<T>& P, const T* R, const T* wB, T* aw, T* av) {
  T Iw[3], wIw[3], gB[3], cg[3], tau[3], wc[3], wwc[3], Rwwc[3], frc[3];
  sym3_mul(P.Io, wB, Iw);
  cross3(wB, Iw, wIw);
  gB[0] = -P.grav * R[6]; gB[1] = -P.grav * R[7]; gB[2] = -P.grav * R[8];
  cross3(P.c, gB, cg);
  for (int i = 0; i < 3; ++i) tau[i] = -wIw[i] + P.m * cg[i];
  cross3(wB, P.c, wc);
  cross3(wB, wc, wwc);
  rot3(R, wwc, Rwwc);
  for (int i = 0; i < 3; ++i) frc[i] = -P.m * Rwwc[i];
  frc[2] -= P.m * P.grav;
  cube_minv(P, R, tau, frc, aw, av);
}

// residual of contact c at twist u:  r = D_mu (u_w x rho_c + u_v) + q_c
template <typename T>
CN_HD void cube_contact_residual(const CubeParams<T>& P, const CubeProb<T>& S, int c, const T* u, T* rho, T* r) {
  rho[0] = S.rho(3 * c); rho[1] = S.rho(3 * c + 1); rho[2] = S.rho(3 * c + 2);
  T e[3];
  cross3_add(u, rho, u + 3, e);
  r[0] = P.mu * e[0] + S.q(3 * c);
  r[1] = P.mu * e[1] + S.q(3 * c + 1);
  r[2] = e[2] + S.q(3 * c + 2);
}

// Gradient (and optionally Hessian) of the primal objective at u (world twist).
//   g = M u - sum_c J_c^T f~_c ;  H = M + sum_c J_c^T K_c J_c   (H: full 6x6 row-major, lower part)
// Also returns the scaled norms used by the stopping test.
template <typename T, bool WANT_H, int UNR>
CN_HD void cube_eval(const CubeParams<T>& P, const CubeProb<T>& S, const T* u, T* g, T* H, T& res2, T& scale2) {
  T Mu[6];
  cube_mass_mul(P, S, u, Mu);
  T z[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  if (WANT_H) {
    const T m0 = S.mcW(0), m1 = S.mcW(1), m2 = S.mcW(2);
    H[0] = S.IW(0); H[7] = S.IW(1); H[14] = S.IW(2);
    H[6] = S.IW(3); H[12] = S.IW(4); H[13] = S.IW(5);
    // M_vw = -S(mcW): rows 3..5, cols 0..2
    H[18] = T(0); H[19] = m2;   H[20] = -m1;
    H[24] = -m2;  H[25] = T(0); H[26] = m0;
    H[30] = m1;   H[31] = -m0;  H[32] = T(0);
    H[21] = P.m; H[28] = P.m; H[35] = P.m; H[27] = T(0); H[33] = T(0); H[34] = T(0);
  }
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    T rho[3], r[3], f[3], K[6];
    cube_contact_residual(P, S, c, u, rho, r);
    cone_eval<T, WANT_H>(r, P.inv_eps, P.mu, f, K);
    const T ft[3] = {P.mu * f[0], P.mu * f[1], f[2]};
    cross3_add(rho, ft, z, z);
#pragma unroll
    for (int i = 0; i < 3; ++i) z[3 + i] += ft[i];
    if (WANT_H) {
      const T K0[3] = {K[0], K[1], K[2]}, K1[3] = {K[1], K[3], K[4]}, K2[3] = {K[2], K[4], K[5]};
      // Pm = S(rho) K : column j = rho x K_j  (K symmetric)
      T P0[3], P1[3], P2[3];
      cross3(rho, K0, P0); cross3(rho, K1, P1); cross3(rho, K2, P2);
      // H_vw (rows 3+j, cols i) += Pm^T
#pragma unroll
      for (int i = 0; i < 3; ++i) { H[18 + i] += P0[i]; H[24 + i] += P1[i]; H[30 + i] += P2[i]; }
      // H_ww += -Pm S(rho) = S(rho) K S(rho)^T: row i = rho x (row i of Pm); only the lower triangle, each entry one
      // FMA chain ending on H
      const T a = rho[0], b = rho[1], cz = rho[2];
      H[0] = H[0] + b * P2[0] - cz * P1[0];
      H[6] = H[6] + b * P2[1] - cz * P1[1];
      H[7] = H[7] + cz * P0[1] - a * P2[1];
      H[12] = H[12] + b * P2[2] - cz * P1[2];
      H[13] = H[13] + cz * P0[2] - a * P2[2];
      H[14] = H[14] + a * P1[2] - b * P0[2];
      // H_vv += K
      H[21] += K[0]; H[27] += K[1]; H[28] += K[3]; H[33] += K[2]; H[34] += K[4]; H[35] += K[5];
    }
  }
  // scaled residual test quantities: D = 1/diag(M) (body-frame diagonal as a fixed scale)
  res2 = T(0); T a2 = T(0), b2 = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    g[i] = Mu[i] - z[i];
    res2 += g[i] * g[i] * P.dscale[i];
    a2 += Mu[i] * Mu[i] * P.dscale[i];
    b2 += z[i] * z[i] * P.dscale[i];
  }
  scale2 = t_max(a2, b2);
}

// True iff u = 0 is already optimal: every contact's y = -q/eps lies in the polar cone, so
// all forces vanish and the gradient M*0 - J^T 0 is exactly zero (free flight).
template <typename T, int UNR> CN_HD bool cube_trivially_solved(const CubeProb<T>& S) {
  bool open = true;
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    const T q0 = S.q(3 * c), q1 = S.q(3 * c + 1), qn = S.q(3 * c + 2);
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
  }
  return open;
}

template <typename T> CN_HD bool cube_converged(const SolverCfg<T>& cfg, T res2, T scale2) {
  return !(res2 > cfg.tol_rel * cfg.tol_rel * scale2);   // also true for NaN
}

enum { NEWTON_DONE = 0, NEWTON_CONTINUE = 1 };

// Line-search state of the unified Newton visit below (one bracket on the pending direction).
template <typename T> struct CubeTrial {
  T alpha, lo, hi;   // u = u0 + alpha d is the tentative point; phi' < 0 at lo, > 0 at hi
};

// One Newton VISIT = exactly one gradient/Hessian evaluation, no inner loop (the unit the wavefront
// kernel schedules; the per-thread kernels simply loop over visits).  State: u (current, possibly
// tentative point u0 + alpha d), d / d0 = phi'(0) of the pending direction (d0 = 0: nothing pending),
// the bracket tr, best_res2, it.  The step taken by the previous visit is accepted or rejected
// lazily from the gradient at the new point, which the evaluation for the next direction provides
// anyway: the full step one-sidedly (phi'(1) <= ls_c |phi'(0)|), an interior trial on
// |phi'(alpha)| <= ls_c |phi'(0)|.  A rejected point moves the bracket and the next trial is one
// safeguarded Newton iteration on phi'(alpha), with phi'' = d^T H d exact from this evaluation.
// Stops: scaled gradient below tol_rel; three evaluations without a 4x reduction of the best residual
// below tol_stall (rounding floor of the sample's conditioning); iteration cap.  A gradient below
// cfg.tol_final (quadratic regime: the next step lands at rounding level) takes the step and
// finishes without the confirming evaluation.
//   it: bits 0-7 Newton directions taken, 8-15 trials on the pending direction (0xff = forced
//   accept), 16+ rounding-floor counter.  Returns NEWTON_DONE or NEWTON_CONTINUE.
template <typename T, int UNR>
CN_HD int cube_newton_visit(const CubeParams<T>& P, const CubeProb<T>& S, const SolverCfg<T>& cfg, T* u, T* d,
                            T& d0, T& best_res2, CubeTrial<T>& tr, int& it) {
  T g[6], H[36], res2, scale2;
  CN_STAT_UNIT();
  cube_eval<T, true, UNR>(P, S, u, g, H, res2, scale2);
  if (cube_converged(cfg, res2, scale2)) {
    if (cfg.polish && res2 == res2) {
      block_solve6_neg<T>(H, g, d);
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] += d[i];
    }
    return NEWTON_DONE;
  }
  if (res2 <= cfg.tol_stall * cfg.tol_stall * scale2 && !(res2 < T(0.25) * best_res2)) {
    it += 1 << 16;
    if ((it >> 16) >= 3) return NEWTON_DONE;
  } else if (res2 < best_res2 || best_res2 < T(0)) {
    it &= 0xffff;
  }
  if (res2 < best_res2 || best_res2 < T(0)) best_res2 = res2;
  const int trials = (it >> 8) & 0xff;
  if (d0 < T(0) && trials != 0xff) {
    T d1 = T(0);
#pragma unroll
    for (int i = 0; i < 6; ++i) d1 += g[i] * d[i];
    const T thresh = -cfg.ls_c * d0;
    // the full step is accepted one-sidedly (still descending is fine); interior trials on |phi'|
    const bool accept = trials == 0 ? (d1 <= thresh) : (t_abs(d1) <= thresh);
    if (!accept) {
      if (d1 < T(0)) tr.lo = tr.alpha; else tr.hi = tr.alpha;
      T d2 = T(0);                                  // phi''(alpha) = d^T H d (lower triangle of H is filled)
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        T row = T(0);
#pragma unroll
        for (int j = 0; j < 6; ++j) row += H[j <= i ? 6 * i + j : 6 * j + i] * d[j];
        d2 += d[i] * row;
      }
      T an = tr.alpha - d1 * t_rcp(d2);
      if (!(an > tr.lo && an < tr.hi)) an = T(0.5) * (tr.lo + tr.hi);
      int nt = trials + 1;
      if (tr.hi - tr.lo <= T(4) * eps_of<T>() * tr.hi || nt >= 7) {   // budget spent: keep a point with phi' <= 0
        an = tr.lo > T(0) ? tr.lo : an;
        nt = 0xff;
      }
      const T step = an - tr.alpha;
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] += step * d[i];
      tr.alpha = an;
      it = (it & ~0xff00) | (nt << 8);
      return NEWTON_CONTINUE;
    }
  }
  if ((it & 0xff) >= cfg.max_iter) return NEWTON_DONE;
  block_solve6_neg<T>(H, g, d);
  T dd = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) { dd += g[i] * d[i]; u[i] += d[i]; }
  d0 = dd < T(0) ? dd : T(0);
  tr.alpha = T(1); tr.lo = T(0); tr.hi = T(1);
  it = (it & ~0xff00) + 1;
  if (res2 <= cfg.tol_final * cfg.tol_final * scale2) return NEWTON_DONE;
  return NEWTON_CONTINUE;
}

// Newton solve from u (in: start point -- zero, or the previous step's solution as a warm start;
// out: optimum).  Returns the number of Newton directions taken.
template <typename T, int UNR>
CN_HD int cube_solve(const CubeParams<T>& P, const CubeProb<T>& S, const SolverCfg<T>& cfg, T* u) {
  int it = 0;
  if (cube_trivially_solved<T, UNR>(S)) {
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] = T(0);
  } else {
    T d[6], d0 = T(0), best = T(-1);
    CubeTrial<T> tr{T(1), T(0), T(1)};
    while (cube_newton_visit<T, UNR>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
  }
  return it & 0xff;
}

// ---------------------------------------------------------------------------
// ContactNets loss (multibody_learnable_system.py:104-197): prologue builds the QP
// at (q+, v+); epilogue evaluates the loss at the solved (detached) forces and, by
// the envelope theorem (:172-175), the parameter gradient in the same pass.
// ---------------------------------------------------------------------------
template <typename T> struct CubeLossAux {
  T R[9];       // world <- body rotation at q+
  T dv[6];      // v+ - (v + dt a), state coordinates [body w ; world v]   (:156)
  T acc[6];     // contact-free acceleration, state coordinates
  T vp[6];      // v+, state coordinates
  T pos_z;
  T konst;      // 1/2 dv^T M dv + sum max(-phi,0)^2   (:163-170)
  T dvW[6];     // dv as a world twist: the always-feasible end of the start segment (cube_loss_start)
  T a_min;      // fraction of the segment dv -> 0 at which the first contact leaves its polar cone
  uint32_t sel; // selected corners (sign bits)
};

// Start point of the loss QP's solve.  In the primal form every contact's residual is r_c(u) = D_mu J_c (u - dv) + s_c with
// s_c = [dt mu v_t ; |phi| + dt |mu v_t|] inside the polar cone: u = dv (the measured velocity change, world twist) is always
// feasible with zero forces, u = 0 minimises the kinetic term, and the optimum is (up to eps) the M-projection of 0 onto the
// feasible set.  Along the segment u = (1 - a) dv the residual is the interpolation (1 - a) s_c + a q_c, so the a at which
// contact c leaves the polar cone is the root of one quadratic; a_b = min_c a_c is where the segment leaves the feasible set.
// Starting the Newton iteration at a = min(1, CN_LOSS_START_FACTOR a_b) instead of u = 0 (a = 1) puts it next to the
// contacts that actually activate: measured on the bench batch 11.1 -> 7.4 evaluations per solve, on recorded tosses 8.5 ->
// 7.6 (tools/exp_solver_trace.py; factors 3..9 are within 3% of each other, 1 -- the boundary itself -- gains nothing because
// the curvature there is still M alone).  The optimum is unique, so only the iteration count changes.  0 disables it.
#ifndef CN_LOSS_START_FACTOR
#define CN_LOSS_START_FACTOR 7.0
#endif

template <typename T, int UNR>
CN_HD void cube_loss_prologue(const CubeParams<T>& P, const T* x, const T* xp, const CubeProb<T>& S,
                              CubeLossAux<T>& A) {
  cube_geometry<T, UNR>(P, xp, A.R, A.sel, S);
  A.pos_z = xp[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) A.vp[i] = xp[7 + i];
  cube_free_accel(P, A.R, A.vp, A.acc, A.acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) A.dv[i] = A.vp[i] - (x[7 + i] + P.dt * A.acc[i]);
  // world twists
  T dvW[6], vW[6];
  rot3(A.R, A.dv, dvW); rot3(A.R, A.vp, vW);
#pragma unroll
  for (int i = 0; i < 3; ++i) { dvW[3 + i] = A.dv[3 + i]; vW[3 + i] = A.vp[3 + i]; }
  T pen4 = T(0), a_min = T(2);
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
    T ed[3], ev[3];
    cross3_add(dvW, rho, dvW + 3, ed); cross3_add(vW, rho, vW + 3, ev);
    const T sx = P.mu * ev[0], sy = P.mu * ev[1];
    const T speed2 = sx * sx + sy * sy;
    const T speed = speed2 * t_rsqrt0(speed2);
    const T phic = rho[2] + A.pos_z;
    const T s0 = P.dt * sx, s1 = P.dt * sy, s2 = t_abs(phic) + P.dt * speed;
    const T e0 = -P.mu * ed[0], e1 = -P.mu * ed[1], e2 = -ed[2];
    S.q(3 * c) = e0 + s0;                                          // :158-161
    S.q(3 * c + 1) = e1 + s1;
    S.q(3 * c + 2) = e2 + s2;
    const T pneg2 = t_abs(phic) - phic;                            // 2 max(-phi_c, 0), exactly
    pen4 += pneg2 * pneg2;
    if (CN_LOSS_START_FACTOR > 0) {
      // |s_t + a e_t|^2 = (s_n + a e_n)^2, i.e. Aq a^2 + 2 Bh a + Cq = 0: smallest positive root, in the cancellation-free
      // form -Cq / (Bh + sqrt(disc)).  Cq = min(cs, 0) = (cs - |cs|) / 2, exactly.  disc < 0 (no root) makes den NaN, so
      // den > 0 alone selects the samples with a root.
      const T Aq = e0 * e0 + e1 * e1 - e2 * e2, Bh = s0 * e0 + s1 * e1 - s2 * e2;
      const T cs = s0 * s0 + s1 * s1 - s2 * s2;
      const T Cq = T(0.5) * (cs - t_abs(cs));
      const T disc = Bh * Bh - Aq * Cq;
      const T den = Bh + disc * t_rsqrt0(disc);
      const T a_c = den > T(0) ? -Cq * t_rcp(den) : T(2);
      a_min = a_c < a_min ? a_c : a_min;
    }
  }
  const T pen = T(0.25) * pen4;
  A.a_min = a_min;
#pragma unroll
  for (int i = 0; i < 6; ++i) A.dvW[i] = dvW[i];
  T Mdv[6];
  cube_mass_mul(P, S, dvW, Mdv);
  T e = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) e += dvW[i] * Mdv[i];
  A.konst = T(0.5) * e + pen;
}

// vex(X) with <X, S(a)> = a . vex(X);  X row-major 3x3
// Start point u = (1 - a) dv with a = min(1, factor a_min) (factor <= 0: a = 1, the round-1 start u = 0; factor < 0 is
// reserved for callers that pass a fixed fraction through cube_loss_start_fraction).
template <typename T> CN_HD void cube_loss_start_fraction(const CubeLossAux<T>& A, T a, T* u) {
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = (T(1) - a) * A.dvW[i];
}
template <typename T> CN_HD void cube_loss_start(const CubeLossAux<T>& A, T factor, T* u) {
  cube_loss_start_fraction<T>(A, factor > T(0) ? t_min(factor * A.a_min, T(1)) : T(1), u);
}

template <typename T> CN_HD void vex3(const T* X, T* o) {
  o[0] = X[7] - X[5]; o[1] = X[2] - X[6]; o[2] = X[3] - X[1];
}

// Adjoint of a rigid body's mass matrix and force vector w.r.t. its inertia 10-vector
// [m, c(3), Ixx, Iyy, Izz, Ixy, Ixz, Iyz] (body-frame angular / world-frame linear coordinates):
//   M = [[I_o, m S(c) R^T], [-m R S(c), m I3]],  I_o = I_sym - m S(c)^2,
//   F = [-w x (I_o w) + m c x (R^T g) ; -m R (w x (w x c)) + m g]
// given the loss differential  <Kww, dM_ww> + <N, dM_wv> + trvv dm (from M_vv) + lam . dF,
// with N = Mbar_wv + Mbar_vw^T.  grad[0..9] += d loss / d inertia-vector.
template <typename T>
CN_HD void rigid_body_inertia_adjoint(T m, const T* c, const T* R, const T* w, T grav, T* Kww, const T* N, T trvv,
                                      const T* lam, T* grad) {
  // F-term into the I_o adjoint: (w x lam_w) w^T
  T wxl[3];
  cross3(w, lam, wxl);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Kww[3 * i + j] += wxl[i] * w[j];
  // I_sym
  grad[4] += Kww[0]; grad[5] += Kww[4]; grad[6] += Kww[8];
  grad[7] += Kww[1] + Kww[3]; grad[8] += Kww[2] + Kww[6]; grad[9] += Kww[5] + Kww[7];
  const T trK = Kww[0] + Kww[4] + Kww[8];
  T Kc[3], Ktc[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Kc[i] = Kww[3 * i] * c[0] + Kww[3 * i + 1] * c[1] + Kww[3 * i + 2] * c[2];
    Ktc[i] = Kww[i] * c[0] + Kww[3 + i] * c[1] + Kww[6 + i] * c[2];
  }
  const T cc = dot3(c, c);
  T NR[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) NR[3 * i + j] = N[3 * i] * R[j] + N[3 * i + 1] * R[3 + j] + N[3 * i + 2] * R[6 + j];
  T vNR[3];
  vex3(NR, vNR);
  const T gB[3] = {-grav * R[6], -grav * R[7], -grav * R[8]};
  T ell[3];
  rot3t(R, lam + 3, ell);
  T cxg[3], wc[3], wwc[3], wl[3], wwl[3], gxl[3];
  cross3(c, gB, cxg);
  cross3(w, c, wc); cross3(w, wc, wwc);
  cross3(w, ell, wl); cross3(w, wl, wwl);
  cross3(gB, lam, gxl);
  grad[0] += cc * trK - dot3(c, Kc) + dot3(c, vNR) + trvv + dot3(lam, cxg) - dot3(ell, wwc) - grav * lam[5];
#pragma unroll
  for (int i = 0; i < 3; ++i)
    grad[1 + i] += m * (T(2) * trK * c[i] - Kc[i] - Ktc[i] + vNR[i] + gxl[i] - wwl[i]);
}

// Loss value at the optimum u and (if grad != nullptr) += d loss / d [inertia(10), mu, half(3)].
// force_out (nullable): reference order [n(4); (tx,ty)(4)].
// PARK: pass 1 overwrites the slot's q_c (dead after q.f) with the force f_c so that pass 2 reads it back
// instead of re-evaluating the cone projection (the wavefront kernel; S is consumed).
template <typename T, int UNR, bool PARK = false>
CN_HD T cube_loss_epilogue(const CubeParams<T>& P, const CubeProb<T>& S, const CubeLossAux<T>& A, const T* u,
                           T* grad, T* force_out) {
  const T* R = A.R;
  // pass 1: forces f_c = Pi(-(D_mu J_c u + q_c)/eps), z = J^T f (world twist), q.f, f.f, validity
  T zW[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  T qf = T(0), ff = T(0);
  bool fok = true;                         // every |f_i| <= 1e3 (false for NaN)
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    T rho[3], r[3], f[3];
    cube_contact_residual(P, S, c, u, rho, r);
    cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
    const T ft[3] = {P.mu * f[0], P.mu * f[1], f[2]};
    cross3_add(rho, ft, zW, zW);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      zW[3 + i] += ft[i];
      qf += S.q(3 * c + i) * f[i]; ff += f[i] * f[i];
      fok = fok && t_abs(f[i]) <= T(1e3);
    }
    if (PARK) {
#pragma unroll
      for (int i = 0; i < 3; ++i) S.q(3 * c + i) = f[i];
    }
    if (force_out) { force_out[c] = f[2]; force_out[4 + 2 * c] = f[0]; force_out[4 + 2 * c + 1] = f[1]; }
  }
  if (!fok) {                              // |f| > 1e3, NaN or Inf: force := 0, constant := 0 (:186-192)
    if (force_out) for (int i = 0; i < 12; ++i) force_out[i] = T(0);
    return T(0);
  }
  T z[6], y[6];
  rot3t(R, zW, z);
#pragma unroll
  for (int i = 0; i < 3; ++i) z[3 + i] = zW[3 + i];
  cube_minv(P, R, z, z + 3, y, y + 3);
  T zy = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + A.konst;   // :194-195
  if (!grad) return loss;

  // ---- envelope backward (forces fixed) ----
  const T* dv = A.dv; const T* a = A.acc; const T* w = A.vp;   // w = body angular velocity (first 3)
  T lam[6], b[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { b[i] = y[i] - dv[i]; lam[i] = P.dt * b[i]; }   // lam = -dt (dv - y)
  // Mbar = -1/2 y y^T + 1/2 dv dv^T - lam a^T
  T Kww[9], N[9], trvv = T(0);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Kww[3 * i + j] = T(0.5) * (dv[i] * dv[j] - y[i] * y[j]) - lam[i] * a[j];
      N[3 * i + j] = (dv[i] * dv[3 + j] - y[i] * y[3 + j]) - lam[i] * a[3 + j] - lam[3 + j] * a[i];
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) trvv += T(0.5) * (dv[3 + i] * dv[3 + i] - y[3 + i] * y[3 + i]) - lam[3 + i] * a[3 + i];
  rigid_body_inertia_adjoint<T>(P.m, P.c, R, w, P.grav, Kww, N, trvv, lam, grad);
  // pass 2: contacts -> mu and half lengths (forces recomputed: cheaper than parking them)
  T bW[3], wW[3];
  rot3(R, b, bW); rot3(R, w, wW);
  T gmu = T(0), gh0 = T(0), gh1 = T(0), gh2 = T(0);
#pragma unroll UNR
  for (int cidx = 0; cidx < CUBE_NC; ++cidx) {
    T rho[3], r[3], f[3];
    if (PARK) {
#pragma unroll
      for (int i = 0; i < 3; ++i) { rho[i] = S.rho(3 * cidx + i); f[i] = S.q(3 * cidx + i); }
    } else {
      cube_contact_residual(P, S, cidx, u, rho, r);
      cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
    }
    T eb[3], ev[3];
    cross3_add(bW, rho, b + 3, eb); cross3_add(wW, rho, A.vp + 3, ev);
    const T ftx = f[0], fty = f[1], fn = f[2];
    const T sx = P.mu * ev[0], sy = P.mu * ev[1];
    const T sinv = t_rsqrt0(sx * sx + sy * sy);                     // speed 0: sx = sy = 0, so ux = uy = 0
    const T ux = sx * sinv, uy = sy * sinv;
    const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
    gmu = gmu + ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
    const T phic = rho[2] + A.pos_z;
    const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - (t_abs(phic) - phic);
    // (R^T ft) x b + (R^T gt) x w + phibar R^T e_z = R^T (ft x bW + gt x wW + phibar e_z)
    const T ft[3] = {P.mu * ftx, P.mu * fty, fn};
    const T gt[3] = {P.mu * gx, P.mu * gy, T(0)};
    T p[3], pB[3];
    cross3(ft, bW, p);
    cross3_add(gt, wW, p, p);
    p[2] += phibar;
    rot3t(R, p, pB);
    gh0 += sgn_bit<T>(A.sel, cidx, 0) * pB[0];
    gh1 += sgn_bit<T>(A.sel, cidx, 1) * pB[1];
    gh2 += sgn_bit<T>(A.sel, cidx, 2) * pB[2];
  }
  grad[10] += gmu;
  grad[11] += gh0; grad[12] += gh1; grad[13] += gh2;
  return loss;
}

// Free-flight fast path of the loss (wavefront kernel's triage phase).  70% of a toss data set is flight:
// every contact's q lies in the polar cone, so u = 0, f = 0 (cube_trivially_solved) and
//   loss = 1/2 dv^T M dv + sum max(-phi,0)^2,
// whose parameter gradient needs only the inertia adjoint and the penetration term.  Everything is
// evaluated in registers -- no problem record is built -- at about a third of the generic
// prologue + epilogue.  Returns false (nothing written) when the sample needs the solver.
template <typename T>
CN_HD bool cube_loss_free_flight(const CubeParams<T>& P, const T* x, const T* xp, T* grad, T* loss_out) {
  T R[9], vp[6], acc[6], dv[6];
  quat_to_rot(xp, R);
  const T dsup[3] = {-R[6], -R[7], -R[8]};
  const uint32_t sel = cube_select_corners(dsup, P.h);
#pragma unroll
  for (int i = 0; i < 6; ++i) vp[i] = xp[7 + i];
  cube_free_accel(P, R, vp, acc, acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) dv[i] = vp[i] - (x[7 + i] + P.dt * acc[i]);
  T dvW[3], vW[3], Rh[9];
  rot3(R, dv, dvW); rot3(R, vp, vW);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) Rh[3 * i + k] = R[3 * i + k] * P.h[k];
  bool open = true;
  T pen4 = T(0), gs[3] = {T(0), T(0), T(0)};
#pragma unroll 1
  for (int c = 0; c < CUBE_NC; ++c) {
    const T sx = sgn_bit<T>(sel, c, 0), sy = sgn_bit<T>(sel, c, 1), sz = sgn_bit<T>(sel, c, 2);
    T rho[3], ed[3], ev[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) rho[i] = sx * Rh[3 * i] + sy * Rh[3 * i + 1] + sz * Rh[3 * i + 2];
    cross3_add(dvW, rho, dv + 3, ed); cross3_add(vW, rho, vp + 3, ev);
    const T tx = P.mu * ev[0], ty = P.mu * ev[1];
    const T speed2 = tx * tx + ty * ty;
    const T speed = speed2 * t_rsqrt0(speed2);
    const T phic = rho[2] + xp[6];
    const T q0 = -P.mu * ed[0] + P.dt * tx, q1 = -P.mu * ed[1] + P.dt * ty;
    const T qn = -ed[2] + t_abs(phic) + P.dt * speed;
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
    const T pneg2 = t_abs(phic) - phic;              // 2 max(-phi_c, 0) = -d loss / d phi_c at f = 0, exactly
    pen4 += pneg2 * pneg2;
    gs[0] -= sx * pneg2; gs[1] -= sy * pneg2; gs[2] -= sz * pneg2;
  }
  if (!open) return false;
  const T pen = T(0.25) * pen4;
  const T gh[3] = {gs[0] * R[6], gs[1] * R[7], gs[2] * R[8]};
  // 1/2 dv^T M dv in state coordinates: w^T Io w + 2 m w . (c x R^T v) + m v . v
  T vB[3], Iw[3], cxv[3];
  rot3t(R, dv + 3, vB);
  sym3_mul(P.Io, dv, Iw);
  cross3(P.c, vB, cxv);
  const T e = dot3(dv, Iw) + T(2) * P.m * dot3(dv, cxv) + P.m * dot3(dv + 3, dv + 3);
  *loss_out = T(0.5) * e + pen;
  if (grad) {
    // the generic envelope backward (cube_loss_epilogue) with y = 0: b = -dv, lam = -dt dv
    T lam[6], Kww[9], N[9], trvv = T(0);
#pragma unroll
    for (int i = 0; i < 6; ++i) lam[i] = -P.dt * dv[i];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        Kww[3 * i + j] = T(0.5) * dv[i] * dv[j] - lam[i] * acc[j];
        N[3 * i + j] = dv[i] * dv[3 + j] - lam[i] * acc[3 + j] - lam[3 + j] * acc[i];
      }
#pragma unroll
    for (int i = 0; i < 3; ++i) trvv += T(0.5) * dv[3 + i] * dv[3 + i] - lam[3 + i] * acc[3 + i];
    rigid_body_inertia_adjoint<T>(P.m, P.c, R, vp, P.grav, Kww, N, trvv, lam, grad);
    grad[11] += gh[0]; grad[12] += gh[1]; grad[13] += gh[2];
  }
  return true;
}

// Whole per-sample loss path (the simple, one-thread-per-sample composition; registers).
template <typename T>
CN_HD T cube_loss_sample(const CubeParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, T* grad,
                         T* force_out, int* iters_out) {
  T store[CUBE_PROB_FIELDS];
  const CubeProb<T> S{store, 1};
  CubeLossAux<T> A;
  cube_loss_prologue<T, 4>(P, x, xp, S, A);
  T u[6];
  cube_loss_start<T>(A, T(CN_LOSS_START_FACTOR), u);
  const int it = cube_solve<T, 4>(P, S, cfg, u);
  if (iters_out) *iters_out = it;
  return cube_loss_epilogue<T, 4>(P, S, A, u, grad, force_out);
}

// ---------------------------------------------------------------------------
// Learnable time step: forward_dynamics (multibody_learnable_system.py:260-304) +
// VelocityIntegrator.step (integrator.py:153-162) + FloatingBaseSpace.exponential
// (state_space.py:466-486, quaternion.py:89-104, 276-309).  No quaternion renormalisation.
// ---------------------------------------------------------------------------
template <typename T> struct CubeStepAux {
  T R[9];
  T vm[6];     // v + dt a  (state coordinates)   (:285)
  uint32_t sel;
};

// builds the step QP at (q, v): q_c = D_mu J_c v_minus + [0, 0, phi_c / dt]   (:286)
template <typename T, int UNR>
CN_HD void cube_step_prologue(const CubeParams<T>& P, const T* x, const CubeProb<T>& S, CubeStepAux<T>& A) {
  T acc[6], vmW[6];
  cube_geometry<T, UNR>(P, x, A.R, A.sel, S);
  cube_free_accel(P, A.R, x + 7, acc, acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) A.vm[i] = x[7 + i] + P.dt * acc[i];
  rot3(A.R, A.vm, vmW);
#pragma unroll
  for (int i = 0; i < 3; ++i) vmW[3 + i] = A.vm[3 + i];
  const T inv_dt = T(1) / P.dt;
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
    T e[3];
    cross3(vmW, rho, e);
    S.q(3 * c) = P.mu * (e[0] + vmW[3]);
    S.q(3 * c + 1) = P.mu * (e[1] + vmW[4]);
    S.q(3 * c + 2) = (e[2] + vmW[5]) + (rho[2] + x[6]) * inv_dt;
  }
}

// x_next from the solved twist u.  The reference forms v+ = v- + M^-1 J^T f (:303-304); at the
// optimum M u = J^T f, so v+ = v- + u, which is used here because u is the better-conditioned
// quantity (f = Pi(-(J u + q)/eps) amplifies rounding in u by 1/eps).  q+ = q (+) v+ dt.
template <typename T, int UNR>
CN_HD void cube_step_epilogue(const CubeParams<T>& P, const CubeProb<T>& S, const CubeStepAux<T>& A, const T* x,
                              const T* u, T* xn, T* force_out) {
  if (force_out) {
#pragma unroll UNR
    for (int c = 0; c < CUBE_NC; ++c) {
      T rho[3], r[3], f[3];
      cube_contact_residual(P, S, c, u, rho, r);
      cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
      force_out[c] = f[2]; force_out[4 + 2 * c] = f[0]; force_out[4 + 2 * c + 1] = f[1];
    }
  }
  T uB[3], vn[6];
  rot3t(A.R, u, uB);
#pragma unroll
  for (int i = 0; i < 3; ++i) { vn[i] = A.vm[i] + uB[i]; vn[3 + i] = A.vm[3 + i] + u[3 + i]; }
  const T rx = vn[0] * P.dt, ry = vn[1] * P.dt, rz = vn[2] * P.dt;
  const T ang = t_sqrt(rx * rx + ry * ry + rz * rz);
  const T half = T(0.5) * ang;
  const T sinc = half > T(0) ? sin(half) / half : T(1);      // quaternion.py:208-229
  const T dw = cos(half), k = T(0.5) * sinc;
  const T dx = rx * k, dy = ry * k, dz = rz * k;
  const T qw = x[0], qx = x[1], qy = x[2], qz = x[3];
  xn[0] = qw * dw - (qx * dx + qy * dy + qz * dz);
  xn[1] = qw * dx + dw * qx + (qy * dz - qz * dy);
  xn[2] = qw * dy + dw * qy + (qz * dx - qx * dz);
  xn[3] = qw * dz + dw * qz + (qx * dy - qy * dx);
#pragma unroll
  for (int i = 0; i < 3; ++i) xn[4 + i] = x[4 + i] + vn[3 + i] * P.dt;
#pragma unroll
  for (int i = 0; i < 6; ++i) xn[7 + i] = vn[i];
}

// warm (nullable, in/out): the contact velocity change u of the toss's previous step as the start
// point of this step's solve (the optimum is unique, so only the iteration count depends on it).
template <typename T>
CN_HD int cube_step_sample(const CubeParams<T>& P, const SolverCfg<T>& cfg, const T* x, T* xn, T* force_out,
                           T* warm = nullptr) {
  T store[CUBE_PROB_FIELDS];
  const CubeProb<T> S{store, 1};
  CubeStepAux<T> A;
  cube_step_prologue<T, 4>(P, x, S, A);
  T u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = warm ? warm[i] : T(0);
  const int it = cube_solve<T, 4>(P, S, cfg, u);
  cube_step_epilogue<T, 4>(P, S, A, x, u, xn, force_out);
  if (warm) {
#pragma unroll
    for (int i = 0; i < 6; ++i) warm[i] = u[i];
  }
  return it;
}

// ---------------------------------------------------------------------------
// The same single floating body with WITNESS POINTS instead of box corners: the contact set of any plane-convex
// pair (GeometryCollider.collide_plane_convex, geometry.py:553-582) is "n_c <= 4 support points p_c of the shape in
// the direction -R^T e_z", whatever the shape -- a Sphere's single point d r (geometry.py:415-456), the top-n_query
// vertices of a Polygon (geometry.py:220-252, 162-202), the outputs of a support-function network.  The caller
// evaluates the shape's support points (they are piecewise constant or linear in the shape parameters and carry
// no state gradient) and gets d loss / d p_c back.  Contacts c >= n_c are switched off by a linear term deep in the
// polar cone (zero force, zero curvature) and take no part in the loss.  Same reference spans as above.
// ---------------------------------------------------------------------------
template <typename T> CN_HD T contact_off() { return T(1e30); }

template <typename T>
CN_HD void body_geometry_pts(const CubeParams<T>& P, const T* quat, const T* pts, int n_c, T* R, const CubeProb<T>& S) {
  quat_to_rot(quat, R);
  T A[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const T r0 = R[3 * i], r1 = R[3 * i + 1], r2 = R[3 * i + 2];
    A[3 * i + 0] = r0 * P.Io[0] + r1 * P.Io[3] + r2 * P.Io[4];
    A[3 * i + 1] = r0 * P.Io[3] + r1 * P.Io[1] + r2 * P.Io[5];
    A[3 * i + 2] = r0 * P.Io[4] + r1 * P.Io[5] + r2 * P.Io[2];
  }
  S.IW(0) = A[0] * R[0] + A[1] * R[1] + A[2] * R[2];
  S.IW(1) = A[3] * R[3] + A[4] * R[4] + A[5] * R[5];
  S.IW(2) = A[6] * R[6] + A[7] * R[7] + A[8] * R[8];
  S.IW(3) = A[0] * R[3] + A[1] * R[4] + A[2] * R[5];
  S.IW(4) = A[0] * R[6] + A[1] * R[7] + A[2] * R[8];
  S.IW(5) = A[3] * R[6] + A[4] * R[7] + A[5] * R[8];
  T cW[3];
  rot3(R, P.c, cW);
#pragma unroll
  for (int i = 0; i < 3; ++i) S.mcW(i) = P.m * cW[i];
#pragma unroll
  for (int c = 0; c < CUBE_NC; ++c) {
    T r[3] = {T(0), T(0), T(0)};
    if (c < n_c) rot3(R, pts + 3 * c, r);
#pragma unroll
    for (int i = 0; i < 3; ++i) S.rho(3 * c + i) = r[i];
  }
}

// loss (multibody_learnable_system.py:104-197) with witness points: grad11 += d loss / d [inertia 10 | mu];
// grad_pts (12, written): d loss / d p_c (zero rows for c >= n_c); force_out (nullable, 12): reference order.
template <typename T>
CN_HD T body_loss_sample_pts(const CubeParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, const T* pts,
                             int n_c, T* grad11, T* grad_pts, T* force_out, int* iters_out) {
  T store[CUBE_PROB_FIELDS];
  const CubeProb<T> S{store, 1};
  T R[9], vp[6], acc[6], dv[6];
  body_geometry_pts(P, xp, pts, n_c, R, S);
  const T pos_z = xp[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) vp[i] = xp[7 + i];
  cube_free_accel(P, R, vp, acc, acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) dv[i] = vp[i] - (x[7 + i] + P.dt * acc[i]);
  T dvW[6], vW[6];
  rot3(R, dv, dvW); rot3(R, vp, vW);
#pragma unroll
  for (int i = 0; i < 3; ++i) { dvW[3 + i] = dv[3 + i]; vW[3 + i] = vp[3 + i]; }
  T pen = T(0);
#pragma unroll
  for (int c = 0; c < CUBE_NC; ++c) {
    if (c < n_c) {
      const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
      T ed[3], ev[3];
      cross3(dvW, rho, ed); cross3(vW, rho, ev);
#pragma unroll
      for (int i = 0; i < 3; ++i) { ed[i] += dvW[3 + i]; ev[i] += vW[3 + i]; }
      const T sx = P.mu * ev[0], sy = P.mu * ev[1];
      const T speed2 = sx * sx + sy * sy;
      const T speed = speed2 * t_rsqrt(t_max(speed2, t_tiny<T>()));
      const T phic = rho[2] + pos_z;
      S.q(3 * c) = -P.mu * ed[0] + P.dt * sx;
      S.q(3 * c + 1) = -P.mu * ed[1] + P.dt * sy;
      S.q(3 * c + 2) = -ed[2] + t_abs(phic) + P.dt * speed;
      const T pneg = t_max(-phic, T(0));
      pen += pneg * pneg;
    } else {
      S.q(3 * c) = T(0); S.q(3 * c + 1) = T(0); S.q(3 * c + 2) = contact_off<T>();
    }
  }
  T Mdv[6];
  cube_mass_mul(P, S, dvW, Mdv);
  T e = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) e += dvW[i] * Mdv[i];
  const T konst = T(0.5) * e + pen;
  T u[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  const int it = cube_solve<T, 4>(P, S, cfg, u);
  if (iters_out) *iters_out = it;
  // forces, loss
  T zW[6] = {T(0), T(0), T(0), T(0), T(0), T(0)}, fs[12];
  T qf = T(0), ff = T(0), fmax = T(0);
#pragma unroll
  for (int c = 0; c < CUBE_NC; ++c) {
    T rho[3], r[3], f[3] = {T(0), T(0), T(0)};
    if (c < n_c) {
      cube_contact_residual(P, S, c, u, rho, r);
      cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
      const T ft[3] = {P.mu * f[0], P.mu * f[1], f[2]};
      T tq[3];
      cross3(rho, ft, tq);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        zW[i] += tq[i]; zW[3 + i] += ft[i];
        qf += S.q(3 * c + i) * f[i]; ff += f[i] * f[i];
        const T af = t_abs(f[i]);
        fmax = (af > fmax || af != af) ? af : fmax;
      }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) fs[3 * c + i] = f[i];
    if (force_out) { force_out[c] = f[2]; force_out[4 + 2 * c] = f[0]; force_out[4 + 2 * c + 1] = f[1]; }
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) grad_pts[i] = T(0);
  if (!(fmax <= T(1e3))) {
    if (force_out) for (int i = 0; i < 12; ++i) force_out[i] = T(0);
    return T(0);
  }
  T z[6], y[6];
  rot3t(R, zW, z);
#pragma unroll
  for (int i = 0; i < 3; ++i) z[3 + i] = zW[3 + i];
  cube_minv(P, R, z, z + 3, y, y + 3);
  T zy = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + konst;
  if (!grad11) return loss;
  // envelope backward, as cube_loss_epilogue, with d/d p_c instead of d/d half lengths
  T lam[6], b[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { b[i] = y[i] - dv[i]; lam[i] = P.dt * b[i]; }
  T Kww[9], N[9], trvv = T(0);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Kww[3 * i + j] = T(0.5) * (dv[i] * dv[j] - y[i] * y[j]) - lam[i] * acc[j];
      N[3 * i + j] = (dv[i] * dv[3 + j] - y[i] * y[3 + j]) - lam[i] * acc[3 + j] - lam[3 + j] * acc[i];
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) trvv += T(0.5) * (dv[3 + i] * dv[3 + i] - y[3 + i] * y[3 + i]) - lam[3 + i] * acc[3 + i];
  rigid_body_inertia_adjoint<T>(P.m, P.c, R, vp, P.grav, Kww, N, trvv, lam, grad11);
  T bW[3], wW[3];
  rot3(R, b, bW); rot3(R, vp, wW);
  T gmu = T(0);
#pragma unroll
  for (int c = 0; c < CUBE_NC; ++c) {
    if (c < n_c) {
      const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
      const T ftx = fs[3 * c], fty = fs[3 * c + 1], fn = fs[3 * c + 2];
      T eb[3], ev[3];
      cross3(bW, rho, eb); cross3(wW, rho, ev);
#pragma unroll
      for (int i = 0; i < 3; ++i) { eb[i] += b[3 + i]; ev[i] += vp[3 + i]; }
      const T sx = P.mu * ev[0], sy = P.mu * ev[1];
      const T sinv = t_rsqrt(t_max(sx * sx + sy * sy, t_tiny<T>()));
      const T ux = sx * sinv, uy = sy * sinv;
      const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
      gmu += ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
      const T ft[3] = {P.mu * ftx, P.mu * fty, fn};
      const T gt[3] = {P.mu * gx, P.mu * gy, T(0)};
      T ftB[3], gtB[3], p1[3], p2[3];
      rot3t(R, ft, ftB); rot3t(R, gt, gtB);
      cross3(ftB, b, p1); cross3(gtB, vp, p2);
      const T phic = rho[2] + pos_z;
      const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - T(2) * t_max(-phic, T(0));
#pragma unroll
      for (int k = 0; k < 3; ++k) grad_pts[3 * c + k] = p1[k] + p2[k] + phibar * R[6 + k];
    }
  }
  grad11[10] += gmu;
  return loss;
}

// ---------------------------------------------------------------------------
// Witness-point pieces of the wavefront loss kernel (cube_loss_wf_kernel, PTS instance): the same per-sample
// composition as body_loss_sample_pts -- triage, prologue, feasible-segment start, Newton visits, epilogue -- cut where
// the box pieces above are cut.  pts points at the sample's 12 body-frame point coordinates (read in place: the
// per-contact loops may be rolled, and a rolled loop over a register array would go through local memory).  Contacts
// c >= n_c are switched off as in body_loss_sample_pts: rho_c = 0, q_c = (0, 0, contact_off), zero force, no
// penetration term.  grad_pts (12, nullable, written) receives wpts * d loss / d p_c (zero rows for c >= n_c).
// ---------------------------------------------------------------------------

// Free-flight fast path (the triage phase), as cube_loss_free_flight: true (loss, grad11 += d loss / d [inertia | mu],
// grad_pts written) when every active contact's q lies in the polar cone; false, nothing written, otherwise.
template <typename T>
CN_HD bool body_loss_free_flight_pts(const CubeParams<T>& P, const T* x, const T* xp, const T* pts, int n_c, T wpts,
                                     T* grad11, T* grad_pts, T* loss_out) {
  T R[9], vp[6], acc[6], dv[6];
  quat_to_rot(xp, R);
#pragma unroll
  for (int i = 0; i < 6; ++i) vp[i] = xp[7 + i];
  cube_free_accel(P, R, vp, acc, acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) dv[i] = vp[i] - (x[7 + i] + P.dt * acc[i]);
  T dvW[3], vW[3];
  rot3(R, dv, dvW); rot3(R, vp, vW);
  bool open = true;
  T pen4 = T(0);
#pragma unroll 1
  for (int c = 0; c < n_c; ++c) {
    T rho[3], ed[3], ev[3];
    rot3(R, pts + 3 * c, rho);
    cross3_add(dvW, rho, dv + 3, ed); cross3_add(vW, rho, vp + 3, ev);
    const T tx = P.mu * ev[0], ty = P.mu * ev[1];
    const T speed2 = tx * tx + ty * ty;
    const T speed = speed2 * t_rsqrt0(speed2);
    const T phic = rho[2] + xp[6];
    const T q0 = -P.mu * ed[0] + P.dt * tx, q1 = -P.mu * ed[1] + P.dt * ty;
    const T qn = -ed[2] + t_abs(phic) + P.dt * speed;
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
    const T pneg2 = t_abs(phic) - phic;              // 2 max(-phi_c, 0), exactly
    pen4 += pneg2 * pneg2;
  }
  if (!open) return false;
  const T pen = T(0.25) * pen4;
  // 1/2 dv^T M dv in state coordinates, as cube_loss_free_flight
  T vB[3], Iw[3], cxv[3];
  rot3t(R, dv + 3, vB);
  sym3_mul(P.Io, dv, Iw);
  cross3(P.c, vB, cxv);
  const T e = dot3(dv, Iw) + T(2) * P.m * dot3(dv, cxv) + P.m * dot3(dv + 3, dv + 3);
  *loss_out = T(0.5) * e + pen;
#pragma unroll 1
  for (int c = 0; c < CUBE_NC; ++c) {
    // d loss / d p_c at f = 0: the penetration term only, -2 max(-phi_c, 0) R^T e_z
    const T phic = c < n_c ? R[6] * pts[3 * c] + R[7] * pts[3 * c + 1] + R[8] * pts[3 * c + 2] + xp[6] : T(0);
    const T phibar = (phic - t_abs(phic)) * wpts;
#pragma unroll
    for (int k = 0; k < 3; ++k) if (grad_pts) grad_pts[3 * c + k] = (grad11 && c < n_c) ? phibar * R[6 + k] : T(0);
  }
  if (grad11) {
    T lam[6], Kww[9], N[9], trvv = T(0);
#pragma unroll
    for (int i = 0; i < 6; ++i) lam[i] = -P.dt * dv[i];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        Kww[3 * i + j] = T(0.5) * dv[i] * dv[j] - lam[i] * acc[j];
        N[3 * i + j] = dv[i] * dv[3 + j] - lam[i] * acc[3 + j] - lam[3 + j] * acc[i];
      }
#pragma unroll
    for (int i = 0; i < 3; ++i) trvv += T(0.5) * dv[3 + i] * dv[3 + i] - lam[3 + i] * acc[3 + i];
    rigid_body_inertia_adjoint<T>(P.m, P.c, R, vp, P.grav, Kww, N, trvv, lam, grad11);
  }
  return true;
}

// Prologue: the loss QP at (q+, v+) in the slot S and the sample's auxiliaries A (A.sel unused), as cube_loss_prologue.
// A switched-off contact stays inside the polar cone along the whole start segment, so it takes no part in a_min.
template <typename T, int UNR>
CN_HD void body_loss_prologue_pts(const CubeParams<T>& P, const T* x, const T* xp, const T* pts, int n_c,
                                  const CubeProb<T>& S, CubeLossAux<T>& A) {
  T* R = A.R;
  quat_to_rot(xp, R);
  T Am[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const T r0 = R[3 * i], r1 = R[3 * i + 1], r2 = R[3 * i + 2];
    Am[3 * i + 0] = r0 * P.Io[0] + r1 * P.Io[3] + r2 * P.Io[4];
    Am[3 * i + 1] = r0 * P.Io[3] + r1 * P.Io[1] + r2 * P.Io[5];
    Am[3 * i + 2] = r0 * P.Io[4] + r1 * P.Io[5] + r2 * P.Io[2];
  }
  S.IW(0) = Am[0] * R[0] + Am[1] * R[1] + Am[2] * R[2];
  S.IW(1) = Am[3] * R[3] + Am[4] * R[4] + Am[5] * R[5];
  S.IW(2) = Am[6] * R[6] + Am[7] * R[7] + Am[8] * R[8];
  S.IW(3) = Am[0] * R[3] + Am[1] * R[4] + Am[2] * R[5];
  S.IW(4) = Am[0] * R[6] + Am[1] * R[7] + Am[2] * R[8];
  S.IW(5) = Am[3] * R[6] + Am[4] * R[7] + Am[5] * R[8];
  T cW[3];
  rot3(R, P.c, cW);
#pragma unroll
  for (int i = 0; i < 3; ++i) S.mcW(i) = P.m * cW[i];
  A.sel = 0u;
  A.pos_z = xp[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) A.vp[i] = xp[7 + i];
  cube_free_accel(P, R, A.vp, A.acc, A.acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) A.dv[i] = A.vp[i] - (x[7 + i] + P.dt * A.acc[i]);
  T dvW[6], vW[6];
  rot3(R, A.dv, dvW); rot3(R, A.vp, vW);
#pragma unroll
  for (int i = 0; i < 3; ++i) { dvW[3 + i] = A.dv[3 + i]; vW[3 + i] = A.vp[3 + i]; }
  T pen4 = T(0), a_min = T(2);
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    if (c < n_c) {
      T rho[3];
      rot3(R, pts + 3 * c, rho);
#pragma unroll
      for (int i = 0; i < 3; ++i) S.rho(3 * c + i) = rho[i];
      T ed[3], ev[3];
      cross3_add(dvW, rho, dvW + 3, ed); cross3_add(vW, rho, vW + 3, ev);
      const T sx = P.mu * ev[0], sy = P.mu * ev[1];
      const T speed2 = sx * sx + sy * sy;
      const T speed = speed2 * t_rsqrt0(speed2);
      const T phic = rho[2] + A.pos_z;
      const T s0 = P.dt * sx, s1 = P.dt * sy, s2 = t_abs(phic) + P.dt * speed;
      const T e0 = -P.mu * ed[0], e1 = -P.mu * ed[1], e2 = -ed[2];
      S.q(3 * c) = e0 + s0;
      S.q(3 * c + 1) = e1 + s1;
      S.q(3 * c + 2) = e2 + s2;
      const T pneg2 = t_abs(phic) - phic;
      pen4 += pneg2 * pneg2;
      if (CN_LOSS_START_FACTOR > 0) {             // as cube_loss_prologue
        const T Aq = e0 * e0 + e1 * e1 - e2 * e2, Bh = s0 * e0 + s1 * e1 - s2 * e2;
        const T cs = s0 * s0 + s1 * s1 - s2 * s2;
        const T Cq = T(0.5) * (cs - t_abs(cs));
        const T disc = Bh * Bh - Aq * Cq;
        const T den = Bh + disc * t_rsqrt0(disc);
        const T a_c = den > T(0) ? -Cq * t_rcp(den) : T(2);
        a_min = a_c < a_min ? a_c : a_min;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 3; ++i) S.rho(3 * c + i) = T(0);
      S.q(3 * c) = T(0); S.q(3 * c + 1) = T(0); S.q(3 * c + 2) = contact_off<T>();
    }
  }
  const T pen = T(0.25) * pen4;
  A.a_min = a_min;
#pragma unroll
  for (int i = 0; i < 6; ++i) A.dvW[i] = dvW[i];
  T Mdv[6];
  cube_mass_mul(P, S, dvW, Mdv);
  T e = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) e += dvW[i] * Mdv[i];
  A.konst = T(0.5) * e + pen;
}

// Epilogue: loss at the optimum u; with grad11, grad11 += d loss / d [inertia | mu] and grad_pts = wpts d loss / d p_c
// (the formulas of body_loss_sample_pts); without, grad_pts is zero.  PARK as in cube_loss_epilogue.
template <typename T, int UNR, bool PARK = false>
CN_HD T body_loss_epilogue_pts(const CubeParams<T>& P, const CubeProb<T>& S, const CubeLossAux<T>& A, const T* u, int n_c,
                               T wpts, T* grad11, T* grad_pts, T* force_out) {
  const T* R = A.R;
  T zW[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  T qf = T(0), ff = T(0);
  bool fok = true;
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    T f[3] = {T(0), T(0), T(0)};
    if (c < n_c) {
      T rho[3], r[3];
      cube_contact_residual(P, S, c, u, rho, r);
      cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
      const T ft[3] = {P.mu * f[0], P.mu * f[1], f[2]};
      cross3_add(rho, ft, zW, zW);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        zW[3 + i] += ft[i];
        qf += S.q(3 * c + i) * f[i]; ff += f[i] * f[i];
        fok = fok && t_abs(f[i]) <= T(1e3);
      }
      if (PARK) {
#pragma unroll
        for (int i = 0; i < 3; ++i) S.q(3 * c + i) = f[i];
      }
    }
    if (force_out) { force_out[c] = f[2]; force_out[4 + 2 * c] = f[0]; force_out[4 + 2 * c + 1] = f[1]; }
  }
  if (grad_pts) {
#pragma unroll 1
    for (int i = 0; i < 12; ++i) grad_pts[i] = T(0);
  }
  if (!fok) {
    if (force_out) for (int i = 0; i < 12; ++i) force_out[i] = T(0);
    return T(0);
  }
  T z[6], y[6];
  rot3t(R, zW, z);
#pragma unroll
  for (int i = 0; i < 3; ++i) z[3 + i] = zW[3 + i];
  cube_minv(P, R, z, z + 3, y, y + 3);
  T zy = T(0);
#pragma unroll
  for (int i = 0; i < 6; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + A.konst;
  if (!grad11) return loss;
  const T* dv = A.dv; const T* a = A.acc; const T* w = A.vp;
  T lam[6], b[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { b[i] = y[i] - dv[i]; lam[i] = P.dt * b[i]; }
  T Kww[9], N[9], trvv = T(0);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Kww[3 * i + j] = T(0.5) * (dv[i] * dv[j] - y[i] * y[j]) - lam[i] * a[j];
      N[3 * i + j] = (dv[i] * dv[3 + j] - y[i] * y[3 + j]) - lam[i] * a[3 + j] - lam[3 + j] * a[i];
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) trvv += T(0.5) * (dv[3 + i] * dv[3 + i] - y[3 + i] * y[3 + i]) - lam[3 + i] * a[3 + i];
  rigid_body_inertia_adjoint<T>(P.m, P.c, R, w, P.grav, Kww, N, trvv, lam, grad11);
  T bW[3], wW[3];
  rot3(R, b, bW); rot3(R, w, wW);
  T gmu = T(0);
#pragma unroll UNR
  for (int c = 0; c < CUBE_NC; ++c) {
    if (c < n_c) {
      T rho[3], r[3], f[3];
      if (PARK) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { rho[i] = S.rho(3 * c + i); f[i] = S.q(3 * c + i); }
      } else {
        cube_contact_residual(P, S, c, u, rho, r);
        cone_eval<T, false>(r, P.inv_eps, P.mu, f, (T*)nullptr);
      }
      const T ftx = f[0], fty = f[1], fn = f[2];
      T eb[3], ev[3];
      cross3_add(bW, rho, b + 3, eb); cross3_add(wW, rho, w + 3, ev);
      const T sx = P.mu * ev[0], sy = P.mu * ev[1];
      const T sinv = t_rsqrt0(sx * sx + sy * sy);
      const T ux = sx * sinv, uy = sy * sinv;
      const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
      gmu = gmu + ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
      const T phic = rho[2] + A.pos_z;
      const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - (t_abs(phic) - phic);
      // as cube_loss_epilogue: R^T (ft x bW + gt x wW + phibar e_z)
      const T ft[3] = {P.mu * ftx, P.mu * fty, fn};
      const T gt[3] = {P.mu * gx, P.mu * gy, T(0)};
      T p[3], pB[3];
      cross3(ft, bW, p);
      cross3_add(gt, wW, p, p);
      p[2] += phibar;
      rot3t(R, p, pB);
#pragma unroll
      for (int k = 0; k < 3; ++k) if (grad_pts) grad_pts[3 * c + k] = wpts * pB[k];
    }
  }
  grad11[10] += gmu;
  return loss;
}

// The wavefront kernel's per-sample composition in one thread (host emulation of the PTS instance): triage, then
// prologue, feasible-segment start, Newton visits and epilogue.  Returns the loss; iters_out: Newton directions.
template <typename T>
CN_HD T body_loss_sample_pts_wf(const CubeParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, const T* pts,
                                int n_c, T* grad11, T* grad_pts, int* iters_out) {
  T l = T(0);
  if (body_loss_free_flight_pts<T>(P, x, xp, pts, n_c, T(1), grad11, grad_pts, &l)) {
    if (iters_out) *iters_out = 0;
    return l;
  }
  T store[CUBE_PROB_FIELDS];
  const CubeProb<T> S{store, 1};
  CubeLossAux<T> A;
  body_loss_prologue_pts<T, 1>(P, x, xp, pts, n_c, S, A);
  T u[6];
  cube_loss_start<T>(A, T(CN_LOSS_START_FACTOR), u);
  T d[6], d0 = T(0), best = T(-1);
  CubeTrial<T> tr{T(1), T(0), T(1)};
  int it = 0;
  while (cube_newton_visit<T, 1>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
  if (iters_out) *iters_out = it & 0xff;
  return body_loss_epilogue_pts<T, 1, true>(P, S, A, u, n_c, T(1), grad11, grad_pts, (T*)nullptr);
}

// learnable time step with witness points (forward_dynamics :260-304 + the Lie-group update)
template <typename T>
CN_HD int body_step_sample_pts(const CubeParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* pts, int n_c,
                               T* xn, T* force_out) {
  T store[CUBE_PROB_FIELDS];
  const CubeProb<T> S{store, 1};
  CubeStepAux<T> A;
  A.sel = 0u;
  body_geometry_pts(P, x, pts, n_c, A.R, S);
  T acc[6], vmW[6];
  cube_free_accel(P, A.R, x + 7, acc, acc + 3);
#pragma unroll
  for (int i = 0; i < 6; ++i) A.vm[i] = x[7 + i] + P.dt * acc[i];
  rot3(A.R, A.vm, vmW);
#pragma unroll
  for (int i = 0; i < 3; ++i) vmW[3 + i] = A.vm[3 + i];
  const T inv_dt = T(1) / P.dt;
#pragma unroll
  for (int c = 0; c < CUBE_NC; ++c) {
    if (c < n_c) {
      const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
      T e[3];
      cross3(vmW, rho, e);
      S.q(3 * c) = P.mu * (e[0] + vmW[3]);
      S.q(3 * c + 1) = P.mu * (e[1] + vmW[4]);
      S.q(3 * c + 2) = (e[2] + vmW[5]) + (rho[2] + x[6]) * inv_dt;
    } else {
      S.q(3 * c) = T(0); S.q(3 * c + 1) = T(0); S.q(3 * c + 2) = contact_off<T>();
    }
  }
  T u[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
  const int it = cube_solve<T, 4>(P, S, cfg, u);
  cube_step_epilogue<T, 4>(P, S, A, x, u, xn, force_out);
  return it;
}

// ---------------------------------------------------------------------------
// Dense dynamics terms in the reference's own coordinates and ordering, for callers of
// MultibodyTerms.forward (multibody_terms.py:584-609): M (6x6), J (12x6) = [J_n (4 rows) ; mu J_t
// (x,y interleaved per contact, 8 rows)] (:401-426), phi (4), contact-free acceleration (6) and the
// Delassus operator D = J M^-1 J^T (12x12).  Contacts by ascending box-vertex index.  State
// coordinates: v = [w_body ; v_world], so the point Jacobian of corner p is [-R S(p), I3].
// ---------------------------------------------------------------------------
template <typename T>
CN_HD void cube_terms_sample(const CubeParams<T>& P, const T* q, const T* v, T* M, T* J, T* phi, T* acc, T* D) {
  T R[9], store[33];
  CubeProb<T> S{store, 1};
  uint32_t sel;
  cube_geometry<T, 1>(P, q, R, sel, S);
  cube_free_accel(P, R, v, acc, acc + 3);
  // M = [[Io, m S(c) R^T], [-m R S(c), m I]]
  const T Sc[9] = {T(0), -P.c[2], P.c[1], P.c[2], T(0), -P.c[0], -P.c[1], P.c[0], T(0)};
  for (int i = 0; i < 36; ++i) M[i] = T(0);
  M[0] = P.Io[0]; M[7] = P.Io[1]; M[14] = P.Io[2];
  M[1] = M[6] = P.Io[3]; M[2] = M[12] = P.Io[4]; M[8] = M[13] = P.Io[5];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      T b = T(0);                                   // (S(c) R^T)_{ij} = sum_k Sc[i][k] R[j][k]
      for (int k = 0; k < 3; ++k) b += Sc[3 * i + k] * R[3 * j + k];
      M[6 * i + 3 + j] = P.m * b;
      M[6 * (3 + j) + i] = P.m * b;
    }
  for (int i = 0; i < 3; ++i) M[6 * (3 + i) + 3 + i] = P.m;
  for (int c = 0; c < CUBE_NC; ++c) {
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};   // R p_c
    phi[c] = rho[2] + q[6];
    // -R S(p) = -S(R p) R = -S(rho) R : row i = -(rho x R-columns)...  use (-S(rho) R)_{ij} = -(S(rho) R)_{ij}
    T E[9];
    for (int j = 0; j < 3; ++j) {
      const T col[3] = {R[j], R[3 + j], R[6 + j]};
      T cr[3];
      cross3(rho, col, cr);
      for (int i = 0; i < 3; ++i) E[3 * i + j] = -cr[i];
    }
    for (int j = 0; j < 3; ++j) {
      J[6 * c + j] = E[6 + j];                               // normal row: z
      J[6 * (4 + 2 * c) + j] = P.mu * E[j];                  // tangential x
      J[6 * (4 + 2 * c + 1) + j] = P.mu * E[3 + j];          // tangential y
      J[6 * c + 3 + j] = j == 2 ? T(1) : T(0);
      J[6 * (4 + 2 * c) + 3 + j] = j == 0 ? P.mu : T(0);
      J[6 * (4 + 2 * c + 1) + 3 + j] = j == 1 ? P.mu : T(0);
    }
  }
  if (D) {
    T W[72];                                          // M^-1 J^T, column r = M^-1 (row r of J)
    for (int r = 0; r < 12; ++r) cube_minv(P, R, J + 6 * r, J + 6 * r + 3, W + 6 * r, W + 6 * r + 3);
    for (int a = 0; a < 12; ++a)
      for (int b = 0; b < 12; ++b) {
        T s = T(0);
        for (int k = 0; k < 6; ++k) s += J[6 * a + k] * W[6 * b + k];
        D[12 * a + b] = s;
      }
  }
}

}  // namespace cn
