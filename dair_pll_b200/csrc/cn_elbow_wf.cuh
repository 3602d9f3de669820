// Two-body (elbow) loss path in the form the wavefront kernel needs: closed-form articulated terms, no dense
// 7x7 arrays outside the Newton Hessian, a small per-sample record.
//
// Same reference spans as cn_elbow.cuh (contactnets_loss multibody_learnable_system.py:104-197; ContactTerms /
// LagrangianTerms.forward multibody_terms.py:214-237, 428-521; plane-convex collision geometry.py:553-582); same
// internal coordinates u^ = [w_W1 ; v_W(o1) ; thetadot].  What changes is the algebra:
//   * mass matrix: M^ = [composite rigid body of both links about o1] bordered by ONE hinge column,
//       M^ u = [ I_c u_w + mc_c x u_v + h_w td ;  m_c u_v - mc_c x u_w + h_v td ;  h_w.u_w + h_v.u_v + h_t td ]
//     (17 numbers: I_c 6, mc_c 3, m_c 1, h_w 3, h_v 3, h_t 1) with, for link 2 about o2 (A = R2 Io2 R2^T, k = m2 R2 c2):
//       I_c = I_W1 + A - S(k) S(rJ) - S(rJ) S(k) - m2 S(rJ)^2,  mc_c = m1 R1 c1 + k + m2 rJ,  m_c = m1 + m2,
//       h_w = A a + rJ x (a x k),  h_v = a x k,  h_t = a.A a                       (a = world hinge axis)
//   * M^-1 b: closed form -- the composite body by its 3x3 central inertia (as cube_minv), the hinge by a scalar
//     Schur complement; no 7x7 factorisation in the prologue or the epilogue
//   * envelope backward: Mbar = 1/2 (dv dv^T - y y^T) - lam a^T is a sum of three outer products, so each link's
//     inertia adjoint is formed from the link's own twists of dv, y, lam, a (four 6-vectors) exactly as the cube's
//     epilogue does -- no 7x7 or 6x6 cotangent matrices.
// The Newton Hessian H = M^ + sum_c J_c^T K_c J_c is the one dense object: packed lower triangle (28), Cholesky in
// registers.
#pragma once
#include "cn_elbow.cuh"

namespace cn {

constexpr int EW_REC = 77;       // record: M17 | rho 24 | hc 12 (link-2 contacts) | q 24
constexpr int EW_FIELDS = 96;    // + u 7 | d 7 | best 1 | d0 1 | alpha, lo, hi

// View of the per-sample record: element k at p[k * s] (s = 1: local array; s = #slots: shared-memory pool, field-major)
template <typename T> struct ElbowRec {
  T* p;
  int s;
  CN_HD T& Ic(int i) const { return p[i * s]; }              // composite inertia about o1, world [xx,yy,zz,xy,xz,yz]
  CN_HD T& mc(int i) const { return p[(6 + i) * s]; }        // composite first moment, world
  CN_HD T& mt() const { return p[9 * s]; }                   // total mass
  CN_HD T& hw(int i) const { return p[(10 + i) * s]; }       // hinge column
  CN_HD T& hv(int i) const { return p[(13 + i) * s]; }
  CN_HD T& ht() const { return p[16 * s]; }
  CN_HD T& rho(int k) const { return p[(17 + k) * s]; }      // lever arms from o1, world, 3 per contact
  CN_HD T& hc(int k) const { return p[(41 + k) * s]; }       // hinge columns of the link-2 contacts (k = 3 (c - 4) + i)
  CN_HD T& q(int k) const { return p[(53 + k) * s]; }        // QP linear term, sappy order per contact
};

// kinematics + the closed-form mass terms held in registers while a sample is being set up
template <typename T> struct ElbowSetup {
  T R1[9], R2[9], aW[3], rJ[3];
  T Ic[6], mc[3], mt, hw[3], hv[3], ht;       // M^ (17)
  T A2[6], k2[3];                             // link 2 about o2: world inertia, first moment
  T I1[6], k1[3];                             // link 1 about o1
  // closed-form inverse: central composite inertia inverse, M6^-1 h, 1 / Schur complement
  T Cinv[6], gh[6], sinv;
};

template <typename T> CN_HD void sym_rotate(const T* R, const T* Io, T* out /* [xx,yy,zz,xy,xz,yz] */) {
  T A[9];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const T r0 = R[3 * i], r1 = R[3 * i + 1], r2 = R[3 * i + 2];
    A[3 * i + 0] = r0 * Io[0] + r1 * Io[3] + r2 * Io[4];
    A[3 * i + 1] = r0 * Io[3] + r1 * Io[1] + r2 * Io[5];
    A[3 * i + 2] = r0 * Io[4] + r1 * Io[5] + r2 * Io[2];
  }
  out[0] = A[0] * R[0] + A[1] * R[1] + A[2] * R[2];
  out[1] = A[3] * R[3] + A[4] * R[4] + A[5] * R[5];
  out[2] = A[6] * R[6] + A[7] * R[7] + A[8] * R[8];
  out[3] = A[0] * R[3] + A[1] * R[4] + A[2] * R[5];
  out[4] = A[0] * R[6] + A[1] * R[7] + A[2] * R[8];
  out[5] = A[3] * R[6] + A[4] * R[7] + A[5] * R[8];
}

// -(S(a) S(b) + S(b) S(a)) = 2 (a.b) I - a b^T - b a^T, accumulated with weight w into a symmetric 6-vector
template <typename T> CN_HD void sym_add_cross2(T* S6, const T* a, const T* b, T w) {
  const T ab = dot3(a, b);
  S6[0] += w * (T(2) * ab - T(2) * a[0] * b[0]);
  S6[1] += w * (T(2) * ab - T(2) * a[1] * b[1]);
  S6[2] += w * (T(2) * ab - T(2) * a[2] * b[2]);
  S6[3] += w * (-(a[0] * b[1] + a[1] * b[0]));
  S6[4] += w * (-(a[0] * b[2] + a[2] * b[0]));
  S6[5] += w * (-(a[1] * b[2] + a[2] * b[1]));
}

template <typename T> CN_HD void elbow_setup(const ElbowParams<T>& P, const T* q, ElbowSetup<T>& E) {
  quat_to_rot(q, E.R1);
  T Rj[9];
  axis_angle_rot(P.axis, q[7], Rj);
  mat3_mul(E.R1, Rj, E.R2);
  rot3(E.R1, P.axis, E.aW);
  rot3(E.R1, P.pJ, E.rJ);
  sym_rotate(E.R1, P.body[0].Io, E.I1);
  sym_rotate(E.R2, P.body[1].Io, E.A2);
  T c1[3], c2[3];
  rot3(E.R1, P.body[0].c, c1);
  rot3(E.R2, P.body[1].c, c2);
  const T m1 = P.body[0].m, m2 = P.body[1].m;
#pragma unroll
  for (int i = 0; i < 3; ++i) { E.k1[i] = m1 * c1[i]; E.k2[i] = m2 * c2[i]; }
#pragma unroll
  for (int i = 0; i < 6; ++i) E.Ic[i] = E.I1[i] + E.A2[i];
  sym_add_cross2(E.Ic, E.k2, E.rJ, T(1));             // - S(k) S(rJ) - S(rJ) S(k)
  sym_add_cross2(E.Ic, E.rJ, E.rJ, T(0.5) * m2);      // - m2 S(rJ)^2 = m2 (|rJ|^2 I - rJ rJ^T)
#pragma unroll
  for (int i = 0; i < 3; ++i) E.mc[i] = E.k1[i] + E.k2[i] + m2 * E.rJ[i];
  E.mt = m1 + m2;
  T Aa[3], axk[3], t[3];
  sym3_mul(E.A2, E.aW, Aa);
  cross3(E.aW, E.k2, axk);
  cross3(E.rJ, axk, t);
#pragma unroll
  for (int i = 0; i < 3; ++i) { E.hw[i] = Aa[i] + t[i]; E.hv[i] = axk[i]; }
  E.ht = dot3(E.aW, Aa);
}

// y6 = M6^-1 [tau ; f] for the composite body (world coordinates): I_cen w = tau - mc x f / m,  v = (f + mc x w) / m
template <typename T> CN_HD void elbow_minv6(const ElbowSetup<T>& E, const T* tau, const T* f, T* w, T* v) {
  const T im = T(1) / E.mt;
  T cxf[3], rhs[3], cxw[3];
  cross3(E.mc, f, cxf);
#pragma unroll
  for (int i = 0; i < 3; ++i) rhs[i] = tau[i] - cxf[i] * im;
  sym3_mul(E.Cinv, rhs, w);
  cross3(E.mc, w, cxw);
#pragma unroll
  for (int i = 0; i < 3; ++i) v[i] = (f[i] + cxw[i]) * im;
}

template <typename T> CN_HD void elbow_minv_setup(ElbowSetup<T>& E) {
  // central inertia of the composite: I_c + S(mc)^2 / m = I_c - (|mc|^2 I - mc mc^T) / m
  T C[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) C[i] = E.Ic[i];
  sym_add_cross2(C, E.mc, E.mc, T(-0.5) / E.mt);
  sym3_inv(C, E.Cinv);
  elbow_minv6(E, E.hw, E.hv, E.gh, E.gh + 3);
  E.sinv = T(1) / (E.ht - (dot3(E.hw, E.gh) + dot3(E.hv, E.gh + 3)));
}

// x = M^-1 b (7): bordered system [M6 h; h^T ht]
template <typename T> CN_HD void elbow_minv(const ElbowSetup<T>& E, const T* b, T* x) {
  T y[6];
  elbow_minv6(E, b, b + 3, y, y + 3);
  const T t = (b[6] - (dot3(E.hw, y) + dot3(E.hv, y + 3))) * E.sinv;
#pragma unroll
  for (int i = 0; i < 6; ++i) x[i] = y[i] - E.gh[i] * t;
  x[6] = t;
}

// o = M^ u from the 17 numbers
template <typename T>
CN_HD void elbow_mass_mul17(const T* Ic, const T* mc, T mt, const T* hw, const T* hv, T ht, const T* u, T* o) {
  T b[3], c[3];
  cross3(mc, u + 3, b);
  cross3(mc, u, c);
  o[0] = Ic[0] * u[0] + Ic[3] * u[1] + Ic[4] * u[2] + b[0] + hw[0] * u[6];
  o[1] = Ic[3] * u[0] + Ic[1] * u[1] + Ic[5] * u[2] + b[1] + hw[1] * u[6];
  o[2] = Ic[4] * u[0] + Ic[5] * u[1] + Ic[2] * u[2] + b[2] + hw[2] * u[6];
#pragma unroll
  for (int i = 0; i < 3; ++i) o[3 + i] = mt * u[3 + i] - c[i] + hv[i] * u[6];
  o[6] = dot3(hw, u) + dot3(hv, u + 3) + ht * u[6];
}

// F^ (7) at world twist uW: sum_i T_i^T (F_i - M_i b_i), per link in world coordinates about its own origin,
//   F_i = [-w_i x (I_i w_i) + k_i x g ; -w_i x (w_i x k_i) + m_i g],  b_2 = [(w_1 x a) td ; w_1 x (w_1 x rJ)].
// Also returns b_2 (6) for the backward.
template <typename T>
CN_HD void elbow_force17(const ElbowParams<T>& P, const ElbowSetup<T>& E, const T* uW, T* F, T* b2) {
  const T g[3] = {T(0), T(0), -P.grav};
  // link 1
  T Iw[3], wIw[3], kg[3], wk[3], wwk[3];
  sym3_mul(E.I1, uW, Iw);
  cross3(uW, Iw, wIw);
  cross3(E.k1, g, kg);
  cross3(uW, E.k1, wk); cross3(uW, wk, wwk);
#pragma unroll
  for (int i = 0; i < 3; ++i) { F[i] = -wIw[i] + kg[i]; F[3 + i] = -wwk[i] + P.body[0].m * g[i]; }
  // link 2
  T w2[3], wxa[3], wxr[3], wwr[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) w2[i] = uW[i] + E.aW[i] * uW[6];
  cross3(uW, E.aW, wxa);
  cross3(uW, E.rJ, wxr); cross3(uW, wxr, wwr);
#pragma unroll
  for (int i = 0; i < 3; ++i) { b2[i] = wxa[i] * uW[6]; b2[3 + i] = wwr[i]; }
  T F2[6], Mb[3], kxb[3], kxbw[3];
  sym3_mul(E.A2, w2, Iw);
  cross3(w2, Iw, wIw);
  cross3(E.k2, g, kg);
  cross3(w2, E.k2, wk); cross3(w2, wk, wwk);
  // M_2 b_2 = [A b_w + k x b_v ; m2 b_v - k x b_w]
  sym3_mul(E.A2, b2, Mb);
  cross3(E.k2, b2 + 3, kxb);
  cross3(E.k2, b2, kxbw);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    F2[i] = -wIw[i] + kg[i] - (Mb[i] + kxb[i]);
    F2[3 + i] = -wwk[i] + P.body[1].m * g[i] - (P.body[1].m * b2[3 + i] - kxbw[i]);
  }
  // T2^T F2 = [tau + rJ x f ; f ; a.tau]
  T rxf[3];
  cross3(E.rJ, F2 + 3, rxf);
#pragma unroll
  for (int i = 0; i < 3; ++i) { F[i] += F2[i] + rxf[i]; F[3 + i] += F2[3 + i]; }
  F[6] = dot3(E.aW, F2);
}

// Per-link parameters are selected with value ternaries, and per-contact inputs / outputs (learned witness points,
// forces, witness-point gradients) are read and written in place in global memory: nothing in this file indexes a
// per-thread array dynamically, so the kernels built from it need no local memory.
template <typename T> CN_HD T elbow_mu(const ElbowParams<T>& P, int c) { return (c >> 2) ? P.mu[1] : P.mu[0]; }

// witness point c (0..7) in its geometry frame: box corner (sel bits) or learned support point (pts: this sample's
// 8 x 3 points, storage type IO)
template <typename T, typename IO>
CN_HD void elbow_witness(const ElbowParams<T>& P, uint32_t sel0, uint32_t sel1, const IO* pts, int c, T* p) {
  const int b = c >> 2, cl = c & 3;
  const uint32_t sel = b ? sel1 : sel0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const T off = b ? P.off[1][k] : P.off[0][k];
    const T hk = b ? P.h[1][k] : P.h[0][k];
    p[k] = off + (pts ? T(pts[3 * c + k]) : sgn_bit<T>(sel, cl, k) * hk);
  }
}

// lever arm from o1 and hinge column of contact c
template <typename T>
CN_HD void elbow_contact_geometry(const ElbowSetup<T>& E, int c, const T* p, T* rho, T* hcol) {
  if (c < 4) {
    rot3(E.R1, p, rho);
    hcol[0] = hcol[1] = hcol[2] = T(0);
  } else {
    T r[3];
    rot3(E.R2, p, r);
    cross3(E.aW, r, hcol);
#pragma unroll
    for (int i = 0; i < 3; ++i) rho[i] = E.rJ[i] + r[i];
  }
}

// quantities both the triage and the full prologue produce
template <typename T> struct ElbowLossCore {
  T vp[7], dv[7], acc[7], b2[6];
  T pos_z, konst;
  T a_start;    // start fraction of the Newton solve on the feasible segment u = (1 - a) dv (cube_loss_prologue, cn_cube.cuh)
  uint32_t sel0, sel1;
};

template <typename T>
CN_HD void elbow_loss_core(const ElbowParams<T>& P, const T* x, const T* xp, bool learned, ElbowSetup<T>& E,
                           ElbowLossCore<T>& A) {
  elbow_setup(P, xp, E);
  elbow_minv_setup(E);
  A.pos_z = xp[6];
  T vold[7], F[7];
  elbow_to_world(E.R1, xp + 8, A.vp);
  elbow_to_world(E.R1, x + 8, vold);
  elbow_force17(P, E, A.vp, F, A.b2);
  elbow_minv(E, F, A.acc);
#pragma unroll
  for (int i = 0; i < 7; ++i) A.dv[i] = A.vp[i] - (vold[i] + P.dt * A.acc[i]);
  {
    const T d1[3] = {-E.R1[6], -E.R1[7], -E.R1[8]}, d2[3] = {-E.R2[6], -E.R2[7], -E.R2[8]};
    A.sel0 = learned ? 0u : cube_select_corners(d1, P.h[0]);
    A.sel1 = learned ? 0u : cube_select_corners(d2, P.h[1]);
  }
  T Mdv[7];
  elbow_mass_mul17(E.Ic, E.mc, E.mt, E.hw, E.hv, E.ht, A.dv, Mdv);
  T e = T(0);
#pragma unroll
  for (int i = 0; i < 7; ++i) e += A.dv[i] * Mdv[i];
  A.konst = T(0.5) * e;                            // + penetration term, added by the contact loops
}

// K h for K = [K00,K01,K02,K11,K12,K22]
template <typename T> CN_HD void sym3_mul_k(const T* K, const T* h, T* o) {
  o[0] = K[0] * h[0] + K[1] * h[1] + K[2] * h[2];
  o[1] = K[1] * h[0] + K[3] * h[1] + K[4] * h[2];
  o[2] = K[2] * h[0] + K[4] * h[1] + K[5] * h[2];
}

// contact-point velocity for twist u given (rho, hcol)
template <typename T> CN_HD void point_vel7(const T* rho, const T* hcol, const T* u, T* e) {
  cross3(u, rho, e);
#pragma unroll
  for (int i = 0; i < 3; ++i) e[i] += u[3 + i] + hcol[i] * u[6];
}

// q_c of the loss QP (:158-161) and the contact's penetration term
template <typename T>
CN_HD void elbow_loss_q(const ElbowParams<T>& P, const ElbowLossCore<T>& A, int c, const T* rho, const T* hcol, T* qc,
                        T& pen, T& a_min) {
  const T mu = elbow_mu(P, c);
  T ed[3], ev[3];
  point_vel7(rho, hcol, A.dv, ed);
  point_vel7(rho, hcol, A.vp, ev);
  const T sx = mu * ev[0], sy = mu * ev[1];
  const T speed2 = sx * sx + sy * sy;
  const T speed = speed2 * t_rsqrt(t_max(speed2, t_tiny<T>()));
  const T phic = rho[2] + A.pos_z;
  const T s0 = P.dt * sx, s1 = P.dt * sy, s2 = t_abs(phic) + P.dt * speed;
  const T e0 = -mu * ed[0], e1 = -mu * ed[1], e2 = -ed[2];
  qc[0] = e0 + s0;
  qc[1] = e1 + s1;
  qc[2] = e2 + s2;
  const T pneg = t_max(-phic, T(0));
  pen += pneg * pneg;
  if (CN_LOSS_START_FACTOR > 0) {
    // where this contact leaves the polar cone along u = (1 - a) dv (see cube_loss_prologue)
    const T Aq = e0 * e0 + e1 * e1 - e2 * e2, Bq = T(2) * (s0 * e0 + s1 * e1 - s2 * e2);
    const T Cq = t_min(s0 * s0 + s1 * s1 - s2 * s2, T(0));
    const T disc = Bq * Bq - T(4) * Aq * Cq;
    const T dpos = t_max(disc, T(0));
    const T den = Bq + dpos * t_rsqrt(t_max(dpos, t_tiny<T>()));
    const T a_c = (disc >= T(0) && den > T(0)) ? T(-2) * Cq * t_rcp(den) : T(2);
    a_min = t_min(a_min, a_c);
  }
}

// twist of link BI for world twist v7: [w (link body frame) ; v (world, link origin)]
template <typename T, int BI> CN_HD void elbow_link_twist(const ElbowSetup<T>& E, const T* v7, T* out) {
  T V[6];
  if (BI == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) V[i] = v7[i];
  } else {
    T wxr[3];
    cross3(v7, E.rJ, wxr);
#pragma unroll
    for (int i = 0; i < 3; ++i) { V[i] = v7[i] + E.aW[i] * v7[6]; V[3 + i] = v7[3 + i] + wxr[i]; }
  }
  rot3t(BI ? E.R2 : E.R1, V, out);
#pragma unroll
  for (int i = 0; i < 3; ++i) out[3 + i] = V[3 + i];
}

// Inertia adjoint of link BI from the four world twists (dv, y, lam, a) of the envelope backward:
//   Mbar = 1/2 (dv dv^T - y y^T) - lam a^T  (sum of outer products) and Fbar = lam.
// The link sees the twists T_i (.) (T_1 = [I6 | 0], T_2 = elbow_T2), angular parts in its body frame; link 2's bias term
// F^ -= T_2^T M_2 b_2 adds -lam_2 b_2^T.  grad10[0..9] += d loss / d the link's inertia vector.
template <typename T, int BI>
CN_HD void elbow_inertia_adjoint_link(const ElbowParams<T>& P, const ElbowSetup<T>& E, const ElbowLossCore<T>& A,
                                      const T* y, const T* lam, T* grad10) {
  const T* R = BI ? E.R2 : E.R1;
  T dv[6], yy[6], lm[6], ab[6];
  elbow_link_twist<T, BI>(E, A.dv, dv);
  elbow_link_twist<T, BI>(E, y, yy);
  elbow_link_twist<T, BI>(E, lam, lm);
  elbow_link_twist<T, BI>(E, A.acc, ab);
  if (BI == 1) {
    T bB[3];
    rot3t(R, A.b2, bB);
#pragma unroll
    for (int i = 0; i < 3; ++i) { ab[i] += bB[i]; ab[3 + i] += A.b2[3 + i]; }
  }
  T Kww[9], N[9], trvv = T(0);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Kww[3 * i + j] = T(0.5) * (dv[i] * dv[j] - yy[i] * yy[j]) - lm[i] * ab[j];
      N[3 * i + j] = (dv[i] * dv[3 + j] - yy[i] * yy[3 + j]) - lm[i] * ab[3 + j] - lm[3 + j] * ab[i];
    }
#pragma unroll
  for (int i = 0; i < 3; ++i) trvv += T(0.5) * (dv[3 + i] * dv[3 + i] - yy[3 + i] * yy[3 + i]) - lm[3 + i] * ab[3 + i];
  // body angular velocity at v+: w_i = R_i^T (w_1 [+ a td])
  T wW[3], wB[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wW[i] = A.vp[i] + (BI ? E.aW[i] * A.vp[6] : T(0));
  rot3t(R, wW, wB);
  rigid_body_inertia_adjoint<T>(P.body[BI].m, P.body[BI].c, R, wB, P.grav, Kww, N, trvv, lm, grad10);
}

template <typename T>
CN_HD void elbow_inertia_adjoints(const ElbowParams<T>& P, const ElbowSetup<T>& E, const ElbowLossCore<T>& A,
                                  const T* y, const T* lam, T* grad) {
  elbow_inertia_adjoint_link<T, 0>(P, E, A, y, lam, grad);
  elbow_inertia_adjoint_link<T, 1>(P, E, A, y, lam, grad + 10);
}

// d loss / d (witness point c, geometry frame) given the contact's force and the world twists b = y - dv, v+
template <typename T>
CN_HD void elbow_witness_adjoint(const ElbowParams<T>& P, const ElbowSetup<T>& E, const ElbowLossCore<T>& A, int c,
                                 const T* rho, const T* hcol, const T* f, const T* b, T* pbar, T& gmu) {
  const int bi = c >> 2;
  const T mu = elbow_mu(P, c);
  T eb[3], ev[3];
  point_vel7(rho, hcol, b, eb);
  point_vel7(rho, hcol, A.vp, ev);
  const T ftx = f[0], fty = f[1], fn = f[2];
  const T sx = mu * ev[0], sy = mu * ev[1];
  const T sinv = t_rsqrt(t_max(sx * sx + sy * sy, t_tiny<T>()));
  const T ux = sx * sinv, uy = sy * sinv;
  const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
  gmu += ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
  const T ft[3] = {mu * ftx, mu * fty, fn};
  const T gt[3] = {mu * gx, mu * gy, T(0)};
  T Ob[3], Ov[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Ob[i] = b[i] + (bi ? E.aW[i] * b[6] : T(0));
    Ov[i] = A.vp[i] + (bi ? E.aW[i] * A.vp[6] : T(0));
  }
  // p1 + p2 in world coordinates (rotation commutes with the cross product), then into the link frame
  T w1[3], w2[3], pw[3], pB[3], zrow[3];
  cross3(ft, Ob, w1); cross3(gt, Ov, w2);
#pragma unroll
  for (int i = 0; i < 3; ++i) pw[i] = w1[i] + w2[i];
  if (bi) { rot3t(E.R2, pw, pB); zrow[0] = E.R2[6]; zrow[1] = E.R2[7]; zrow[2] = E.R2[8]; }
  else { rot3t(E.R1, pw, pB); zrow[0] = E.R1[6]; zrow[1] = E.R1[7]; zrow[2] = E.R1[8]; }
  const T phic = rho[2] + A.pos_z;
  const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - T(2) * t_max(-phic, T(0));
#pragma unroll
  for (int k = 0; k < 3; ++k) pbar[k] = pB[k] + phibar * zrow[k];
}

// scatter of one contact's witness-point cotangent: learned geometry -> global grad_pts (scaled by the sample's
// upstream weight), boxes -> the two half-length accumulators
template <typename T, typename IO>
CN_HD void elbow_scatter_pbar(const ElbowLossCore<T>& A, int c, const T* pbar, IO* grad_pts, T weight, T* gh0, T* gh1) {
  const int bi = c >> 2, cl = c & 3;
  if (grad_pts) {
#pragma unroll
    for (int k = 0; k < 3; ++k) grad_pts[3 * c + k] = IO(weight * pbar[k]);
  } else {
    const uint32_t sel = bi ? A.sel1 : A.sel0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const T v = sgn_bit<T>(sel, cl, k) * pbar[k];
      if (bi) gh1[k] += v; else gh0[k] += v;
    }
  }
}

// ---------------------------------------------------------------------------
// Triage: everything in registers, no record.  Returns true (and the sample's loss / gradients) when every
// contact's q lies in the polar cone -- free flight, u = 0, f = 0 --; false (nothing written) when the sample needs
// the solver.  grad: += [inertia1 10 | inertia2 10 | mu 2 | half1 3 | half2 3]; grad_pts (24, nullable): written.
// ---------------------------------------------------------------------------
template <typename T, typename IO>
CN_HD bool elbow_loss_free_flight(const ElbowParams<T>& P, const T* x, const T* xp, const IO* pts, T* grad, IO* grad_pts,
                                  T weight, T* loss_out) {
  ElbowSetup<T> E;
  ElbowLossCore<T> A;
  elbow_loss_core(P, x, xp, pts != nullptr, E, A);
  bool open = true;
  T pen = T(0), a_unused = T(2);
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    T p[3], rho[3], hcol[3], qc[3];
    elbow_witness(P, A.sel0, A.sel1, pts, c, p);
    elbow_contact_geometry(E, c, p, rho, hcol);
    elbow_loss_q(P, A, c, rho, hcol, qc, pen, a_unused);
    open = open && (qc[2] >= T(0)) && (qc[0] * qc[0] + qc[1] * qc[1] <= qc[2] * qc[2]);
  }
  if (!open) return false;
  *loss_out = A.konst + pen;
  if (grad) {
    T y[7], lam[7], b[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) { y[i] = T(0); b[i] = -A.dv[i]; lam[i] = P.dt * b[i]; }
    elbow_inertia_adjoints(P, E, A, y, lam, grad);
    const T f0[3] = {T(0), T(0), T(0)};
    T gh0[3] = {T(0), T(0), T(0)}, gh1[3] = {T(0), T(0), T(0)};
#pragma unroll 1
    for (int c = 0; c < EL_NC; ++c) {
      T p[3], rho[3], hcol[3], pbar[3], gmu = T(0);
      elbow_witness(P, A.sel0, A.sel1, pts, c, p);
      elbow_contact_geometry(E, c, p, rho, hcol);
      elbow_witness_adjoint(P, E, A, c, rho, hcol, f0, b, pbar, gmu);
      elbow_scatter_pbar(A, c, pbar, grad_pts, weight, gh0, gh1);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { grad[22 + k] += gh0[k]; grad[25 + k] += gh1[k]; }
  } else if (grad_pts) {
#pragma unroll 1
    for (int i = 0; i < 24; ++i) grad_pts[i] = IO(0);
  }
  return true;
}

// Full prologue: builds the record (M17, rho, hc, q) at (q+, v+); E and A stay in registers for the epilogue.
template <typename T, typename IO>
CN_HD void elbow_loss_prologue_wf(const ElbowParams<T>& P, const T* x, const T* xp, const IO* pts, const ElbowRec<T>& S,
                                  ElbowSetup<T>& E, ElbowLossCore<T>& A) {
  elbow_loss_core(P, x, xp, pts != nullptr, E, A);
#pragma unroll
  for (int i = 0; i < 6; ++i) S.Ic(i) = E.Ic[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) { S.mc(i) = E.mc[i]; S.hw(i) = E.hw[i]; S.hv(i) = E.hv[i]; }
  S.mt() = E.mt; S.ht() = E.ht;
  T pen = T(0), a_min = T(2);
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    T p[3], rho[3], hcol[3], qc[3];
    elbow_witness(P, A.sel0, A.sel1, pts, c, p);
    elbow_contact_geometry(E, c, p, rho, hcol);
    elbow_loss_q(P, A, c, rho, hcol, qc, pen, a_min);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      S.rho(3 * c + i) = rho[i];
      S.q(3 * c + i) = qc[i];
      if (c >= 4) S.hc(3 * (c - 4) + i) = hcol[i];
    }
  }
  A.konst += pen;
  A.a_start = CN_LOSS_START_FACTOR > 0 ? t_min(T(CN_LOSS_START_FACTOR) * a_min, T(1)) : T(1);
}

template <typename T> CN_HD void elbow_rec_contact(const ElbowRec<T>& S, int c, T* rho, T* hcol) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    rho[i] = S.rho(3 * c + i);
    hcol[i] = c >= 4 ? S.hc(3 * (c - 4) + i) : T(0);
  }
}

// Gradient and packed-lower-triangle Hessian (28: H[i (i + 1) / 2 + j], j <= i) of the primal objective at u
template <typename T, bool WANT_H>
CN_HD void elbow_eval_wf(const ElbowParams<T>& P, const ElbowRec<T>& S, const T* u, T* g, T* H, T& res2, T& scale2) {
  T Mu[7], z[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  {
    const T Ic[6] = {S.Ic(0), S.Ic(1), S.Ic(2), S.Ic(3), S.Ic(4), S.Ic(5)};
    const T mc[3] = {S.mc(0), S.mc(1), S.mc(2)};
    const T hw[3] = {S.hw(0), S.hw(1), S.hw(2)}, hv[3] = {S.hv(0), S.hv(1), S.hv(2)};
    const T mt = S.mt(), ht = S.ht();
    elbow_mass_mul17(Ic, mc, mt, hw, hv, ht, u, Mu);
    if (WANT_H) {
      // rows 0-2 (ww), 3-5 (vw | vv), 6 (hinge)
      H[0] = Ic[0]; H[1] = Ic[3]; H[2] = Ic[1]; H[3] = Ic[4]; H[4] = Ic[5]; H[5] = Ic[2];
      // M_vw = -S(mc): rows 3..5, cols 0..2
      H[6] = T(0);    H[7] = mc[2];   H[8] = -mc[1];  H[9] = mt;
      H[10] = -mc[2]; H[11] = T(0);   H[12] = mc[0];  H[13] = T(0); H[14] = mt;
      H[15] = mc[1];  H[16] = -mc[0]; H[17] = T(0);   H[18] = T(0); H[19] = T(0); H[20] = mt;
      H[21] = hw[0]; H[22] = hw[1]; H[23] = hw[2]; H[24] = hv[0]; H[25] = hv[1]; H[26] = hv[2]; H[27] = ht;
    }
  }
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = elbow_mu(P, c);
    T rho[3], hcol[3], e[3], r[3], f[3], K[6];
    elbow_rec_contact(S, c, rho, hcol);
    point_vel7(rho, hcol, u, e);
    r[0] = mu * e[0] + S.q(3 * c); r[1] = mu * e[1] + S.q(3 * c + 1); r[2] = e[2] + S.q(3 * c + 2);
    cone_eval<T, WANT_H>(r, P.inv_eps, mu, f, K);
    const T ft[3] = {mu * f[0], mu * f[1], f[2]};
    T tq[3];
    cross3(rho, ft, tq);
#pragma unroll
    for (int i = 0; i < 3; ++i) { z[i] += tq[i]; z[3 + i] += ft[i]; }
    z[6] += dot3(hcol, ft);
    if (WANT_H) {
      const T K0[3] = {K[0], K[1], K[2]}, K1[3] = {K[1], K[3], K[4]}, K2[3] = {K[2], K[4], K[5]};
      T P0[3], P1[3], P2[3];                    // Pm = S(rho) K, column j = rho x K_j
      cross3(rho, K0, P0); cross3(rho, K1, P1); cross3(rho, K2, P2);
      // H_vw (rows 3+j, cols i) += Pm^T
#pragma unroll
      for (int i = 0; i < 3; ++i) { H[6 + i] += P0[i]; H[10 + i] += P1[i]; H[15 + i] += P2[i]; }
      // H_ww += -Pm S(rho): row i = rho x (row i of Pm)
      const T r0[3] = {P0[0], P1[0], P2[0]}, r1[3] = {P0[1], P1[1], P2[1]}, r2[3] = {P0[2], P1[2], P2[2]};
      T w0[3], w1[3], w2[3];
      cross3(rho, r0, w0); cross3(rho, r1, w1); cross3(rho, r2, w2);
      H[0] += w0[0]; H[1] += w1[0]; H[2] += w1[1]; H[3] += w2[0]; H[4] += w2[1]; H[5] += w2[2];
      // H_vv += K
      H[9] += K[0]; H[13] += K[1]; H[14] += K[3]; H[18] += K[2]; H[19] += K[4]; H[20] += K[5];
      // hinge row: kh = K h;  H_tw += rho x kh,  H_tv += kh,  H_tt += h.kh   (zero for link-1 contacts)
      T kh[3], rk[3];
      sym3_mul_k(K, hcol, kh);
      cross3(rho, kh, rk);
#pragma unroll
      for (int i = 0; i < 3; ++i) { H[21 + i] += rk[i]; H[24 + i] += kh[i]; }
      H[27] += dot3(hcol, kh);
    }
  }
  res2 = T(0); T a2 = T(0), b2 = T(0);
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    g[i] = Mu[i] - z[i];
    res2 += g[i] * g[i] * P.dscale[i];
    a2 += Mu[i] * Mu[i] * P.dscale[i];
    b2 += z[i] * z[i] * P.dscale[i];
  }
  scale2 = t_max(a2, b2);
}

// packed lower-triangular Cholesky solve H d = -g, fully unrolled (N = 7); H is destroyed
template <typename T> CN_HD void chol7_packed_solve_neg(T* H, const T* g, T* d) {
  T inv_diag[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    T s = H[j * (j + 1) / 2 + j];
#pragma unroll
    for (int m = 0; m < j; ++m) s -= H[j * (j + 1) / 2 + m] * H[j * (j + 1) / 2 + m];
    const T il = t_rsqrt(s);
    inv_diag[j] = il;
#pragma unroll
    for (int i = j + 1; i < 7; ++i) {
      T t = H[i * (i + 1) / 2 + j];
#pragma unroll
      for (int m = 0; m < j; ++m) t -= H[i * (i + 1) / 2 + m] * H[j * (j + 1) / 2 + m];
      H[i * (i + 1) / 2 + j] = t * il;
    }
  }
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    T s = -g[i];
#pragma unroll
    for (int m = 0; m < i; ++m) s -= H[i * (i + 1) / 2 + m] * d[m];
    d[i] = s * inv_diag[i];
  }
#pragma unroll
  for (int i = 6; i >= 0; --i) {
    T s = d[i];
#pragma unroll
    for (int m = i + 1; m < 7; ++m) s -= H[m * (m + 1) / 2 + i] * d[m];
    d[i] = s * inv_diag[i];
  }
}

// phi''(alpha) = d^T H d from the packed lower triangle
template <typename T> CN_HD T quad7_packed(const T* H, const T* d) {
  T s = T(0);
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    T row = T(0);
#pragma unroll
    for (int j = 0; j < i; ++j) row += H[i * (i + 1) / 2 + j] * d[j];
    s += d[i] * (T(2) * row + H[i * (i + 1) / 2 + i] * d[i]);
  }
  return s;
}

// One Newton visit (one gradient/Hessian evaluation, no inner loop): the scheme of cube_newton_visit for n_v = 7.
template <typename T>
CN_HD int elbow_newton_visit(const ElbowParams<T>& P, const ElbowRec<T>& S, const SolverCfg<T>& cfg, T* u, T* d, T& d0,
                             T& best_res2, CubeTrial<T>& tr, int& it) {
  T g[7], H[28], res2, scale2;
  elbow_eval_wf<T, true>(P, S, u, g, H, res2, scale2);
  if (cube_converged(cfg, res2, scale2)) return NEWTON_DONE;
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
    for (int i = 0; i < 7; ++i) d1 += g[i] * d[i];
    const T thresh = -cfg.ls_c * d0;
    const bool accept = trials == 0 ? (d1 <= thresh) : (t_abs(d1) <= thresh);
    if (!accept) {
      if (d1 < T(0)) tr.lo = tr.alpha; else tr.hi = tr.alpha;
      const T d2 = quad7_packed(H, d);
      T an = tr.alpha - d1 * t_rcp(d2);
      if (!(an > tr.lo && an < tr.hi)) an = T(0.5) * (tr.lo + tr.hi);
      int nt = trials + 1;
      if (tr.hi - tr.lo <= T(4) * eps_of<T>() * tr.hi || nt >= 7) {
        an = tr.lo > T(0) ? tr.lo : an;
        nt = 0xff;
      }
      const T step = an - tr.alpha;
#pragma unroll
      for (int i = 0; i < 7; ++i) u[i] += step * d[i];
      tr.alpha = an;
      it = (it & ~0xff00) | (nt << 8);
      return NEWTON_CONTINUE;
    }
  }
  if ((it & 0xff) >= cfg.max_iter) return NEWTON_DONE;
  chol7_packed_solve_neg<T>(H, g, d);
  T dd = T(0);
#pragma unroll
  for (int i = 0; i < 7; ++i) { dd += g[i] * d[i]; u[i] += d[i]; }
  d0 = dd < T(0) ? dd : T(0);
  tr.alpha = T(1); tr.lo = T(0); tr.hi = T(1);
  it = (it & ~0xff00) + 1;
  if (res2 <= cfg.tol_final * cfg.tol_final * scale2) return NEWTON_DONE;
  return NEWTON_CONTINUE;
}

// Loss at the solved u and the envelope backward.  E, A: this sample's setup (rebuilt by the prologue); the forces
// are parked in the record's q between the two contact passes (S is consumed).  grad (nullable): += 28 entries;
// force_out (nullable, this sample's 24 entries in global memory): [n(8); (tx,ty)(8)]; grad_pts (nullable, this
// sample's 24 entries in global memory): weight * d loss / d witness points (written).
template <typename T, typename IO>
CN_HD T elbow_loss_epilogue_wf(const ElbowParams<T>& P, const ElbowRec<T>& S, const ElbowSetup<T>& E,
                               const ElbowLossCore<T>& A, const T* u, T* grad, IO* force_out, IO* grad_pts, T weight) {
  T z[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  T qf = T(0), ff = T(0), fmax = T(0);
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = elbow_mu(P, c);
    T rho[3], hcol[3], e[3], r[3], f[3];
    elbow_rec_contact(S, c, rho, hcol);
    point_vel7(rho, hcol, u, e);
    r[0] = mu * e[0] + S.q(3 * c); r[1] = mu * e[1] + S.q(3 * c + 1); r[2] = e[2] + S.q(3 * c + 2);
    cone_eval<T, false>(r, P.inv_eps, mu, f, (T*)nullptr);
    const T ft[3] = {mu * f[0], mu * f[1], f[2]};
    T tq[3];
    cross3(rho, ft, tq);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      z[i] += tq[i]; z[3 + i] += ft[i];
      qf += S.q(3 * c + i) * f[i]; ff += f[i] * f[i];
      const T af = t_abs(f[i]);
      fmax = (af > fmax || af != af) ? af : fmax;
    }
    z[6] += dot3(hcol, ft);
#pragma unroll
    for (int i = 0; i < 3; ++i) S.q(3 * c + i) = f[i];           // park the force
    if (force_out) { force_out[c] = IO(f[2]); force_out[8 + 2 * c] = IO(f[0]); force_out[8 + 2 * c + 1] = IO(f[1]); }
  }
  if (!(fmax <= T(1e3))) {                    // |f| > 1e3, NaN or Inf: force := 0, constant := 0 (:186-192)
#pragma unroll 1
    for (int i = 0; i < 24; ++i) {
      if (force_out) force_out[i] = IO(0);
      if (grad_pts) grad_pts[i] = IO(0);
    }
    return T(0);
  }
  T y[7];
  elbow_minv(E, z, y);
  T zy = T(0);
#pragma unroll
  for (int i = 0; i < 7; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + A.konst;
  if (!grad) {
    if (grad_pts) {
#pragma unroll 1
      for (int i = 0; i < 24; ++i) grad_pts[i] = IO(0);
    }
    return loss;
  }
  T lam[7], b[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) { b[i] = y[i] - A.dv[i]; lam[i] = P.dt * b[i]; }
  elbow_inertia_adjoints(P, E, A, y, lam, grad);
  T gh0[3] = {T(0), T(0), T(0)}, gh1[3] = {T(0), T(0), T(0)}, gmu0 = T(0), gmu1 = T(0);
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    T rho[3], hcol[3], pbar[3], gmu = T(0);
    elbow_rec_contact(S, c, rho, hcol);
    const T f[3] = {S.q(3 * c), S.q(3 * c + 1), S.q(3 * c + 2)};
    elbow_witness_adjoint(P, E, A, c, rho, hcol, f, b, pbar, gmu);
    if (c >> 2) gmu1 += gmu; else gmu0 += gmu;
    elbow_scatter_pbar(A, c, pbar, grad_pts, weight, gh0, gh1);
  }
  grad[20] += gmu0; grad[21] += gmu1;
#pragma unroll
  for (int k = 0; k < 3; ++k) { grad[22 + k] += gh0[k]; grad[25 + k] += gh1[k]; }
  return loss;
}

// Whole per-sample path on a local record (host emulation / one-sample-per-thread checks of this formulation)
template <typename T>
CN_HD T elbow_loss_sample_wf(const ElbowParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, const T* pts,
                             T* grad, T* force_out, T* grad_pts, int* iters_out) {
  T l = T(0);
  if (elbow_loss_free_flight<T, T>(P, x, xp, pts, grad, grad_pts, T(1), &l)) {
    if (iters_out) *iters_out = 0;
    if (force_out) for (int i = 0; i < 24; ++i) force_out[i] = T(0);
    return l;
  }
  T store[EW_REC];
  const ElbowRec<T> S{store, 1};
  ElbowSetup<T> E;
  ElbowLossCore<T> A;
  elbow_loss_prologue_wf<T, T>(P, x, xp, pts, S, E, A);
  T u[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) u[i] = (T(1) - A.a_start) * A.dv[i];
  int it = 0;
  T d[7], d0 = T(0), best = T(-1);
  CubeTrial<T> tr{T(1), T(0), T(1)};
  while (elbow_newton_visit<T>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
  if (iters_out) *iters_out = it & 0xff;
  return elbow_loss_epilogue_wf<T, T>(P, S, E, A, u, grad, force_out, grad_pts, T(1));
}

// Learnable time step of the two-body system on this file's algebra (closed-form mass terms and inverse, 17-number mass
// record, packed 7x7 Hessian) -- the plain-arithmetic step of the rollout kernels.  Same mathematics as elbow_step_sample
// (cn_elbow.cuh: forward_dynamics multibody_learnable_system.py:199-304 + VelocityIntegrator.step integrator.py:153-162 +
// FloatingBaseSpace.exponential state_space.py:466-486), which stays as the dual-number instance of the backward; the two
// agree to rounding (host-emulation test).  u_out: the QP optimum (v+ = v- + u*), kept for the backward.
template <typename T>
CN_HD int elbow_step_sample_wf(const ElbowParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* pts, T* xn,
                               T* force_out, T* u_out, const T* u_fixed = nullptr) {
  // u_fixed: the optimum is known (kept by the forward rollout) and entered as a constant; ONE Newton step at it then
  // carries, in dual-number arithmetic, the implicit-function derivative of the solve, -H(u*)^-1 dg/d(direction), at the
  // cost of one evaluation instead of a whole dual-number solve (in plain arithmetic the step changes nothing)
  T store[EW_REC];
  const ElbowRec<T> S{store, 1};
  ElbowSetup<T> E;
  elbow_setup(P, x, E);
  elbow_minv_setup(E);
  T vW[7], F[7], b2[6], acc[7], vm[7];
  elbow_to_world(E.R1, x + 8, vW);
  elbow_force17(P, E, vW, F, b2);
  elbow_minv(E, F, acc);
#pragma unroll
  for (int i = 0; i < 7; ++i) vm[i] = vW[i] + P.dt * acc[i];
#pragma unroll
  for (int i = 0; i < 6; ++i) S.Ic(i) = E.Ic[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) { S.mc(i) = E.mc[i]; S.hw(i) = E.hw[i]; S.hv(i) = E.hv[i]; }
  S.mt() = E.mt; S.ht() = E.ht;
  uint32_t sel0 = 0u, sel1 = 0u;
  if (!pts) {
    const T d1[3] = {-E.R1[6], -E.R1[7], -E.R1[8]}, d2[3] = {-E.R2[6], -E.R2[7], -E.R2[8]};
    sel0 = cube_select_corners(d1, P.h[0]);
    sel1 = cube_select_corners(d2, P.h[1]);
  }
  const T inv_dt = T(1) / P.dt;
  bool open = true;
#pragma unroll 1
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = elbow_mu(P, c);
    T p[3], rho[3], hcol[3], e[3];
    elbow_witness<T, T>(P, sel0, sel1, pts, c, p);
    elbow_contact_geometry(E, c, p, rho, hcol);
    point_vel7(rho, hcol, vm, e);
    const T q0 = mu * e[0], q1 = mu * e[1], qn = e[2] + (rho[2] + x[6]) * inv_dt;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      S.rho(3 * c + i) = rho[i];
      if (c >= 4) S.hc(3 * (c - 4) + i) = hcol[i];
    }
    S.q(3 * c) = q0; S.q(3 * c + 1) = q1; S.q(3 * c + 2) = qn;
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
  }
  T u[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  int it = 0;
  if (u_fixed) {
#pragma unroll
    for (int i = 0; i < 7; ++i) u[i] = u_fixed[i];
    if (!open) {
      T g[7], H[28], d[7], res2, scale2;
      elbow_eval_wf<T, true>(P, S, u, g, H, res2, scale2);
      chol7_packed_solve_neg<T>(H, g, d);
#pragma unroll
      for (int i = 0; i < 7; ++i) u[i] += d[i];
    }
  } else if (!open) {
    T d[7], d0 = T(0), best = T(-1);
    CubeTrial<T> tr{T(1), T(0), T(1)};
    while (elbow_newton_visit<T>(P, S, cfg, u, d, d0, best, tr, it) != NEWTON_DONE) {}
  }
  if (u_out) {
#pragma unroll
    for (int i = 0; i < 7; ++i) u_out[i] = u[i];
  }
  if (force_out) {
#pragma unroll 1
    for (int c = 0; c < EL_NC; ++c) {
      const T mu = elbow_mu(P, c);
      T rho[3], hcol[3], e[3], f[3];
      elbow_rec_contact(S, c, rho, hcol);
      point_vel7(rho, hcol, u, e);
      const T r[3] = {mu * e[0] + S.q(3 * c), mu * e[1] + S.q(3 * c + 1), e[2] + S.q(3 * c + 2)};
      cone_eval<T, false>(r, P.inv_eps, mu, f, (T*)nullptr);
      force_out[c] = f[2]; force_out[8 + 2 * c] = f[0]; force_out[8 + 2 * c + 1] = f[1];
    }
  }
  // v+ = v- + u (world twist) -> state coordinates, then q+ = q (+) v+ dt
  T vnW[7], vn[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) vnW[i] = vm[i] + u[i];
  rot3t(E.R1, vnW, vn);
#pragma unroll
  for (int i = 3; i < 7; ++i) vn[i] = vnW[i];
  const T rx = vn[0] * P.dt, ry = vn[1] * P.dt, rz = vn[2] * P.dt;
  const T ang = t_sqrt(rx * rx + ry * ry + rz * rz);
  const T half = T(0.5) * ang;
  using ::sin;          // (cn_dual.cuh's overloads for dual numbers would otherwise hide the scalar ones in this namespace)
  using ::cos;
  const T sinc = half > T(0) ? sin(half) / half : T(1);
  const T dw = cos(half), k = T(0.5) * sinc;
  const T dx = rx * k, dy = ry * k, dz = rz * k;
  const T qw = x[0], qx = x[1], qy = x[2], qz = x[3];
  xn[0] = qw * dw - (qx * dx + qy * dy + qz * dz);
  xn[1] = qw * dx + dw * qx + (qy * dz - qz * dy);
  xn[2] = qw * dy + dw * qy + (qz * dx - qx * dz);
  xn[3] = qw * dz + dw * qz + (qx * dy - qy * dx);
#pragma unroll
  for (int i = 0; i < 3; ++i) xn[4 + i] = x[4 + i] + vn[3 + i] * P.dt;
  xn[7] = x[7] + vn[6] * P.dt;
#pragma unroll
  for (int i = 0; i < 7; ++i) xn[8 + i] = vn[i];
  return it & 0xff;
}

}  // namespace cn
