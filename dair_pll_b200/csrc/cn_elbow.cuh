// Floating base + one revolute child, two box geometries against the ground plane
// (assets/contactnets_elbow.urdf): n_q = 8, n_v = 7, 2 x 4 contacts, k = 24.
//
// Same reference spans as cn_cube.cuh (contactnets_loss multibody_learnable_system.py:104-197,
// forward_dynamics :199-304, ContactTerms.forward multibody_terms.py:428-521, top-k support
// geometry.py:162-202, plane-convex collision :553-582), for the articulated asset; the five
// symbolic callables are restated here in closed form (oracle/callables.py derives the same
// quantities generically and tests/ ties them to physics).
//
// Internal velocity coordinates: world twist of body 1 plus the hinge rate,
//   u^ = [w_W1 ; v_W(origin 1) ; thetadot] = blkdiag(R1, I3, 1) v_state.
// Body twists: V1 = [I6 | 0] u^,  V2 = T2 u^ with T2 = [[I, 0, a_W], [-S(r_J), I, 0]]
// (a_W world hinge axis, r_J = R1 p_J).  Per body, in world coordinates about its own origin,
//   M_i = [[R_i Io_i R_i^T, m_i S(c_Wi)], [-m_i S(c_Wi), m_i I]],
//   F_i = [-w_i x (I_Wi w_i) + m_i c_Wi x g ; -m_i w_i x (w_i x c_Wi) + m_i g],
// and M^ = sum T_i^T M_i T_i,  F^ = sum T_i^T (F_i - M_i b_i),  b_2 = [(w_1 x a_W) thetadot ;
// w_1 x (w_1 x r_J)]  (b_1 = 0).  A contact on body i has J_c = [-S(rho_c), I3, h_c] with
// rho_c the lever arm from origin 1 and h_c = a_W x (x_c - o_2) for body 2 (0 for body 1).
//
// This first version keeps the per-sample problem in thread-local arrays (one sample per
// thread); it is the correctness baseline for the articulated asset, not yet wavefront-scheduled.
#pragma once
#include "cn_cube.cuh"

namespace cn {

constexpr int EL_NQ = 8, EL_NV = 7, EL_NX = 15, EL_NC = 8, EL_K = 24;
constexpr int EL_NPARAM = 28;   // [inertia body1 10 | inertia body2 10 | mu_pair 2 | half1 3 | half2 3]
constexpr int EL_NKIN = 12;     // [joint origin 3 | joint axis 3 | box-1 offset 3 | box-2 offset 3] (URDF constants)

template <typename T> struct ElbowBody {
  T m, c[3], Isym[6], Io[6];
};

template <typename T> struct ElbowParams {
  ElbowBody<T> body[2];
  T mu[2], h[2][3];
  T pJ[3], axis[3], off[2][3];
  T dt, eps, inv_eps, grav;
  T dscale[7];
};

template <typename T>
CN_HD void elbow_params_init(ElbowParams<T>& P, const T* inertia /*20*/, const T* mu /*2*/, const T* half /*6*/,
                             const T* kin /*12*/, T dt, T eps) {
  for (int b = 0; b < 2; ++b) {
    ElbowBody<T>& B = P.body[b];
    const T* in = inertia + 10 * b;
    B.m = in[0];
    for (int i = 0; i < 3; ++i) B.c[i] = in[1 + i];
    for (int i = 0; i < 6; ++i) B.Isym[i] = in[4 + i];
    const T cx = B.c[0], cy = B.c[1], cz = B.c[2], m = B.m;
    B.Io[0] = B.Isym[0] + m * (cy * cy + cz * cz);
    B.Io[1] = B.Isym[1] + m * (cx * cx + cz * cz);
    B.Io[2] = B.Isym[2] + m * (cx * cx + cy * cy);
    B.Io[3] = B.Isym[3] - m * cx * cy;
    B.Io[4] = B.Isym[4] - m * cx * cz;
    B.Io[5] = B.Isym[5] - m * cy * cz;
    P.mu[b] = mu[b];
    for (int i = 0; i < 3; ++i) P.h[b][i] = half[3 * b + i];
  }
  for (int i = 0; i < 3; ++i) { P.pJ[i] = kin[i]; P.axis[i] = kin[3 + i]; P.off[0][i] = kin[6 + i]; P.off[1][i] = kin[9 + i]; }
  P.dt = dt; P.eps = eps; P.inv_eps = T(1) / eps; P.grav = T(9.81);
  // fixed positive scales for the stopping test (rough diagonal of M)
  const T mt = P.body[0].m + P.body[1].m;
  for (int i = 0; i < 3; ++i) { P.dscale[i] = T(1) / (P.body[0].Io[i] + P.body[1].Io[i]); P.dscale[3 + i] = T(1) / mt; }
  P.dscale[6] = T(1) / P.body[1].Io[1];
}

// per-sample kinematics at a configuration
template <typename T> struct ElbowKin {
  T R[2][9];     // world rotations of the two bodies
  T aW[3];       // hinge axis, world
  T rJ[3];       // R1 p_J
  uint32_t sel[2];
};

// View of the per-sample quantities that stay fixed during the Newton solve: element k of the 121-field record
// at p[k * s].  Every user holds the record in a per-thread local array (s = 1).
constexpr int ELBOW_PROB_FIELDS = 121;
template <typename T> struct ElbowProb {
  T* p;
  int s;
  CN_HD T& M(int i) const { return p[i * s]; }            // world-twist mass matrix (7x7, full, symmetric)
  CN_HD T& rho(int k) const { return p[(49 + k) * s]; }   // lever arms from origin 1, world, 3 per contact
  CN_HD T& hc(int k) const { return p[(73 + k) * s]; }    // hinge columns (0 for body-1 contacts)
  CN_HD T& q(int k) const { return p[(97 + k) * s]; }     // QP linear term, sappy order per contact
};

// rotation about a unit axis by angle th (Rodrigues), row-major
template <typename T> CN_HD void axis_angle_rot(const T* a, T th, T* R) {
  const T s = sin(th), c = cos(th), v = T(1) - c;
  R[0] = c + a[0] * a[0] * v;        R[1] = a[0] * a[1] * v - a[2] * s; R[2] = a[0] * a[2] * v + a[1] * s;
  R[3] = a[1] * a[0] * v + a[2] * s; R[4] = c + a[1] * a[1] * v;        R[5] = a[1] * a[2] * v - a[0] * s;
  R[6] = a[2] * a[0] * v - a[1] * s; R[7] = a[2] * a[1] * v + a[0] * s; R[8] = c + a[2] * a[2] * v;
}
template <typename T> CN_HD void mat3_mul(const T* A, const T* B, T* C) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
// I_W = R Io R^T as full 3x3 (Io stored [xx,yy,zz,xy,xz,yz])
template <typename T> CN_HD void rotate_inertia(const T* R, const T* Io, T* IW) {
  T A[9];
  for (int i = 0; i < 3; ++i) {
    const T r0 = R[3 * i], r1 = R[3 * i + 1], r2 = R[3 * i + 2];
    A[3 * i + 0] = r0 * Io[0] + r1 * Io[3] + r2 * Io[4];
    A[3 * i + 1] = r0 * Io[3] + r1 * Io[1] + r2 * Io[5];
    A[3 * i + 2] = r0 * Io[4] + r1 * Io[5] + r2 * Io[2];
  }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) IW[3 * i + j] = A[3 * i] * R[3 * j] + A[3 * i + 1] * R[3 * j + 1] + A[3 * i + 2] * R[3 * j + 2];
}

template <typename T> CN_HD void elbow_kinematics(const ElbowParams<T>& P, const T* q, ElbowKin<T>& K) {
  quat_to_rot(q, K.R[0]);
  T Rj[9];
  axis_angle_rot(P.axis, q[7], Rj);
  mat3_mul(K.R[0], Rj, K.R[1]);
  rot3(K.R[0], P.axis, K.aW);
  rot3(K.R[0], P.pJ, K.rJ);
}

// T2 (6x7) applied to a world twist u (7): body-2 twist
template <typename T> CN_HD void elbow_T2(const ElbowKin<T>& K, const T* u, T* V) {
  T wxr[3];
  cross3(u, K.rJ, wxr);
  for (int i = 0; i < 3; ++i) { V[i] = u[i] + K.aW[i] * u[6]; V[3 + i] = u[3 + i] + wxr[i]; }
}
// T2^T applied to a body-2 wrench W (6): generalized force (7)
template <typename T> CN_HD void elbow_T2t(const ElbowKin<T>& K, const T* W, T* o) {
  T rxf[3];
  cross3(K.rJ, W + 3, rxf);                   // (-S(rJ))^T f = rJ x f
  for (int i = 0; i < 3; ++i) { o[i] = W[i] + rxf[i]; o[3 + i] = W[3 + i]; }
  o[6] = dot3(K.aW, W);
}

// body mass matrix in world coordinates about its own origin (6x6 full)
template <typename T> CN_HD void body_mass_world(const ElbowBody<T>& B, const T* R, T* Mi, T* cW) {
  T IW[9];
  rotate_inertia(R, B.Io, IW);
  rot3(R, B.c, cW);
  const T mc[3] = {B.m * cW[0], B.m * cW[1], B.m * cW[2]};
  for (int i = 0; i < 36; ++i) Mi[i] = T(0);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Mi[6 * i + j] = IW[3 * i + j];
  // M_wv = m S(cW); M_vw = -m S(cW)
  Mi[0 * 6 + 4] = -mc[2]; Mi[0 * 6 + 5] = mc[1];
  Mi[1 * 6 + 3] = mc[2];  Mi[1 * 6 + 5] = -mc[0];
  Mi[2 * 6 + 3] = -mc[1]; Mi[2 * 6 + 4] = mc[0];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Mi[6 * (3 + i) + j] = Mi[6 * j + 3 + i];
  for (int i = 0; i < 3; ++i) Mi[6 * (3 + i) + 3 + i] = B.m;
}

// M^ (7x7) and F^ (7) at (kinematics, world twist of the state velocity)
template <typename T>
CN_HD void elbow_mass_force(const ElbowParams<T>& P, const ElbowKin<T>& K, const T* uW, T* M, T* F, T* b2_out) {
  for (int i = 0; i < 49; ++i) M[i] = T(0);
  for (int i = 0; i < 7; ++i) F[i] = T(0);
  const T g[3] = {T(0), T(0), -P.grav};
  for (int b = 0; b < 2; ++b) {
    const ElbowBody<T>& B = P.body[b];
    T Mi[36], cW[3], V[6], bias[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
    body_mass_world(B, K.R[b], Mi, cW);
    if (b == 0) { for (int i = 0; i < 6; ++i) V[i] = uW[i]; }
    else {
      elbow_T2(K, uW, V);
      T wxa[3], wxr[3], wwr[3];
      cross3(uW, K.aW, wxa);
      cross3(uW, K.rJ, wxr); cross3(uW, wxr, wwr);
      for (int i = 0; i < 3; ++i) { bias[i] = wxa[i] * uW[6]; bias[3 + i] = wwr[i]; }
      if (b2_out) for (int i = 0; i < 6; ++i) b2_out[i] = bias[i];
    }
    // F_i = [-w x (I_W w) + m cW x g ; -m w x (w x cW) + m g]
    T Iw[3], wIw[3], cg[3], wc[3], wwc[3], Fi[6];
    for (int i = 0; i < 3; ++i) Iw[i] = Mi[6 * i] * V[0] + Mi[6 * i + 1] * V[1] + Mi[6 * i + 2] * V[2];
    cross3(V, Iw, wIw);
    cross3(cW, g, cg);
    cross3(V, cW, wc); cross3(V, wc, wwc);
    for (int i = 0; i < 3; ++i) { Fi[i] = -wIw[i] + B.m * cg[i]; Fi[3 + i] = -B.m * wwc[i] + B.m * g[i]; }
    if (b == 0) {
      for (int i = 0; i < 6; ++i) {
        F[i] += Fi[i];
        for (int j = 0; j < 6; ++j) M[7 * i + j] += Mi[6 * i + j];
      }
    } else {
      // subtract M_2 b_2, then project with T2^T
      for (int i = 0; i < 6; ++i) {
        T s = T(0);
        for (int j = 0; j < 6; ++j) s += Mi[6 * i + j] * bias[j];
        Fi[i] -= s;
      }
      T f7[7];
      elbow_T2t(K, Fi, f7);
      for (int i = 0; i < 7; ++i) F[i] += f7[i];
      // M += T2^T M_2 T2 : column j of (M_2 T2) = M_2 (T2 e_j), then T2^T of it
      for (int j = 0; j < 7; ++j) {
        T ej[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)}, Vj[6], MV[6], col[7];
        ej[j] = T(1);
        elbow_T2(K, ej, Vj);
        for (int i = 0; i < 6; ++i) {
          T s = T(0);
          for (int m = 0; m < 6; ++m) s += Mi[6 * i + m] * Vj[m];
          MV[i] = s;
        }
        elbow_T2t(K, MV, col);
        for (int i = 0; i < 7; ++i) M[7 * i + j] += col[i];
      }
    }
  }
}

// witness points of both geometries: lever arms, hinge columns.  pts == nullptr: box corners (top-4 of
// 8, geometry.py:162-202); otherwise pts[24] holds the 4 + 4 witness points in the geometry frames, as
// produced by the learned support function (DeepSupportConvex.get_vertices, geometry.py:309-325).
template <typename T>
CN_HD void elbow_contacts(const ElbowParams<T>& P, ElbowKin<T>& K, const ElbowProb<T>& S, const T* pts) {
  for (int b = 0; b < 2; ++b) {
    const T* R = K.R[b];
    const T d[3] = {-R[6], -R[7], -R[8]};
    K.sel[b] = pts ? 0u : cube_select_corners(d, P.h[b]);
    for (int c = 0; c < 4; ++c) {
      T p[3], r[3];
      for (int k = 0; k < 3; ++k)
        p[k] = P.off[b][k] + (pts ? pts[3 * (4 * b + c) + k] : sgn_bit<T>(K.sel[b], c, k) * P.h[b][k]);
      rot3(R, p, r);
      const int cc = 4 * b + c;
      if (b == 0) {
        for (int i = 0; i < 3; ++i) { S.rho(3 * cc + i) = r[i]; S.hc(3 * cc + i) = T(0); }
      } else {
        T ar[3];
        cross3(K.aW, r, ar);
        for (int i = 0; i < 3; ++i) { S.rho(3 * cc + i) = K.rJ[i] + r[i]; S.hc(3 * cc + i) = ar[i]; }
      }
    }
  }
}

// contact-point velocity of contact c for world twist u (7): e = u_w x rho + u_v + h thetadot
template <typename T> CN_HD void elbow_point_vel(const ElbowProb<T>& S, int c, const T* u, T* e) {
  const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
  cross3(u, rho, e);
  for (int i = 0; i < 3; ++i) e[i] += u[3 + i] + S.hc(3 * c + i) * u[6];
}

template <typename T> CN_HD void elbow_residual(const ElbowParams<T>& P, const ElbowProb<T>& S, int c, const T* u, T* r) {
  T e[3];
  elbow_point_vel(S, c, u, e);
  const T mu = P.mu[c >> 2];
  r[0] = mu * e[0] + S.q(3 * c); r[1] = mu * e[1] + S.q(3 * c + 1); r[2] = e[2] + S.q(3 * c + 2);
}

template <typename T, bool WANT_H>
CN_HD void elbow_eval(const ElbowParams<T>& P, const ElbowProb<T>& S, const T* u, T* g, T* H, T& res2, T& scale2) {
  T Mu[7], z[7];
  for (int i = 0; i < 7; ++i) {
    T s = T(0);
    for (int j = 0; j < 7; ++j) s += S.M(7 * i + j) * u[j];
    Mu[i] = s; z[i] = T(0);
  }
  if (WANT_H) for (int i = 0; i < 49; ++i) H[i] = S.M(i);
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = P.mu[c >> 2];
    T r[3], f[3], K[6];
    elbow_residual(P, S, c, u, r);
    cone_eval<T, WANT_H>(r, P.inv_eps, mu, f, K);
    const T ft[3] = {mu * f[0], mu * f[1], f[2]};
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
    const T hc[3] = {S.hc(3 * c), S.hc(3 * c + 1), S.hc(3 * c + 2)};
    T tq[3];
    cross3(rho, ft, tq);
    for (int i = 0; i < 3; ++i) { z[i] += tq[i]; z[3 + i] += ft[i]; }
    z[6] += dot3(hc, ft);
    if (WANT_H) {
      // dense J_c (3x7) = [-S(rho), I, h]
      T J[21];
      J[0] = T(0);     J[1] = rho[2];   J[2] = -rho[1];  J[3] = T(1); J[4] = T(0); J[5] = T(0); J[6] = hc[0];
      J[7] = -rho[2];  J[8] = T(0);     J[9] = rho[0];   J[10] = T(0); J[11] = T(1); J[12] = T(0); J[13] = hc[1];
      J[14] = rho[1];  J[15] = -rho[0]; J[16] = T(0);    J[17] = T(0); J[18] = T(0); J[19] = T(1); J[20] = hc[2];
      T KJ[21];
      for (int j = 0; j < 7; ++j) {
        KJ[j] = K[0] * J[j] + K[1] * J[7 + j] + K[2] * J[14 + j];
        KJ[7 + j] = K[1] * J[j] + K[3] * J[7 + j] + K[4] * J[14 + j];
        KJ[14 + j] = K[2] * J[j] + K[4] * J[7 + j] + K[5] * J[14 + j];
      }
      for (int i = 0; i < 7; ++i)
        for (int j = 0; j <= i; ++j) H[7 * i + j] += J[i] * KJ[j] + J[7 + i] * KJ[7 + j] + J[14 + i] * KJ[14 + j];
    }
  }
  res2 = T(0); T a2 = T(0), b2 = T(0);
  for (int i = 0; i < 7; ++i) {
    g[i] = Mu[i] - z[i];
    res2 += g[i] * g[i] * P.dscale[i];
    a2 += Mu[i] * Mu[i] * P.dscale[i];
    b2 += z[i] * z[i] * P.dscale[i];
  }
  scale2 = t_max(a2, b2);
}

template <typename T> CN_HD bool elbow_trivially_solved(const ElbowProb<T>& S) {
  bool open = true;
  for (int c = 0; c < EL_NC; ++c) {
    const T q0 = S.q(3 * c), q1 = S.q(3 * c + 1), qn = S.q(3 * c + 2);
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
  }
  return open;
}

// Newton solve: the same visit scheme as cube_newton_visit (one gradient/Hessian evaluation per
// visit; rejected steps are searched by safeguarded Newton trials on phi'(alpha) that reuse the full
// evaluation), n_v = 7, Cholesky solve.
template <typename T>
CN_HD int elbow_solve(const ElbowParams<T>& P, const ElbowProb<T>& S, const SolverCfg<T>& cfg, T* u) {
  int it = 0;
  if (elbow_trivially_solved(S)) return 0;
  T d[7], d0 = T(0), best = T(-1);
  T alpha = T(1), lo = T(0), hi = T(1);
  while (true) {
    T g[7], H[49], res2, scale2;
    elbow_eval<T, true>(P, S, u, g, H, res2, scale2);
    if (cube_converged(cfg, res2, scale2)) {
      if (cfg.polish && res2 == res2) {             // dual arithmetic: the step at u* carries the implicit derivative
        T inv_diag[7], ng[7];
        chol_factor<T, 7>(H, inv_diag);
        for (int i = 0; i < 7; ++i) ng[i] = -g[i];
        chol_solve<T, 7>(H, inv_diag, ng, d);
        for (int i = 0; i < 7; ++i) u[i] += d[i];
      }
      break;
    }
    if (res2 <= cfg.tol_stall * cfg.tol_stall * scale2 && !(res2 < T(0.25) * best)) {
      it += 1 << 16;
      if ((it >> 16) >= 3) break;
    } else if (res2 < best || best < T(0)) {
      it &= 0xffff;
    }
    if (res2 < best || best < T(0)) best = res2;
    const int trials = (it >> 8) & 0xff;
    if (d0 < T(0) && trials != 0xff) {
      T d1 = T(0);
      for (int i = 0; i < 7; ++i) d1 += g[i] * d[i];
      const T thresh = -cfg.ls_c * d0;
      const bool accept = trials == 0 ? (d1 <= thresh) : (t_abs(d1) <= thresh);
      if (!accept) {
        if (d1 < T(0)) lo = alpha; else hi = alpha;
        T d2 = T(0);
        for (int i = 0; i < 7; ++i) {
          T row = T(0);
          for (int j = 0; j < 7; ++j) row += H[j <= i ? 7 * i + j : 7 * j + i] * d[j];
          d2 += d[i] * row;
        }
        T an = alpha - d1 / d2;
        if (!(an > lo && an < hi)) an = T(0.5) * (lo + hi);
        int nt = trials + 1;
        if (hi - lo <= T(4) * eps_of<T>() * hi || nt >= 7) {
          an = lo > T(0) ? lo : an;
          nt = 0xff;
        }
        const T step = an - alpha;
        for (int i = 0; i < 7; ++i) u[i] += step * d[i];
        alpha = an;
        it = (it & ~0xff00) | (nt << 8);
        continue;
      }
    }
    if ((it & 0xff) >= cfg.max_iter) break;
    T inv_diag[7], ng[7];
    chol_factor<T, 7>(H, inv_diag);
    for (int i = 0; i < 7; ++i) ng[i] = -g[i];
    chol_solve<T, 7>(H, inv_diag, ng, d);
    T dd = T(0);
    for (int i = 0; i < 7; ++i) { dd += g[i] * d[i]; u[i] += d[i]; }
    d0 = dd < T(0) ? dd : T(0);
    alpha = T(1); lo = T(0); hi = T(1);
    it = (it & ~0xff00) + 1;
    if (res2 <= cfg.tol_final * cfg.tol_final * scale2) break;
  }
  return it & 0xff;
}

// ---------------------------------------------------------------------------
// ContactNets loss + envelope backward
// ---------------------------------------------------------------------------
template <typename T> struct ElbowLossAux {
  ElbowKin<T> K;
  T LM[49], LMinv[7];  // Cholesky factor of M^
  T dv[7], acc[7], vp[7];   // world-twist coordinates
  T b2[6];
  T pos_z, konst;
};

template <typename T>
CN_HD void elbow_to_world(const T* R1, const T* v, T* u) {   // state velocity -> world twist
  rot3(R1, v, u);
  for (int i = 3; i < 7; ++i) u[i] = v[i];
}

template <typename T>
CN_HD void elbow_loss_prologue(const ElbowParams<T>& P, const T* x, const T* xp, const T* pts, const ElbowProb<T>& S,
                               ElbowLossAux<T>& A) {
  elbow_kinematics(P, xp, A.K);
  A.pos_z = xp[6];
  T vold[7];
  elbow_to_world(A.K.R[0], xp + 8, A.vp);
  elbow_to_world(A.K.R[0], x + 8, vold);           // same frame map as the reference: v and v+ are both state coordinates
  T F[7];
  elbow_mass_force(P, A.K, A.vp, A.LM, F, A.b2);       // M into LM, copied to the record before LM is factorised
  for (int i = 0; i < 49; ++i) S.M(i) = A.LM[i];
  chol_factor<T, 7>(A.LM, A.LMinv);
  chol_solve<T, 7>(A.LM, A.LMinv, F, A.acc);
  for (int i = 0; i < 7; ++i) A.dv[i] = A.vp[i] - (vold[i] + P.dt * A.acc[i]);
  elbow_contacts(P, A.K, S, pts);
  T pen = T(0);
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = P.mu[c >> 2];
    T ed[3], ev[3];
    elbow_point_vel(S, c, A.dv, ed);
    elbow_point_vel(S, c, A.vp, ev);
    const T sx = mu * ev[0], sy = mu * ev[1];
    const T speed2 = sx * sx + sy * sy;
    const T speed = speed2 * t_rsqrt(t_max(speed2, t_tiny<T>()));
    const T phic = S.rho(3 * c + 2) + A.pos_z;
    S.q(3 * c) = -mu * ed[0] + P.dt * sx;
    S.q(3 * c + 1) = -mu * ed[1] + P.dt * sy;
    S.q(3 * c + 2) = -ed[2] + t_abs(phic) + P.dt * speed;
    const T pneg = t_max(-phic, T(0));
    pen += pneg * pneg;
  }
  T e = T(0);
  for (int i = 0; i < 7; ++i) {
    T s = T(0);
    for (int j = 0; j < 7; ++j) s += S.M(7 * i + j) * A.dv[j];
    e += A.dv[i] * s;
  }
  A.konst = T(0.5) * e + pen;
}

// grad layout: [inertia1 10 | inertia2 10 | mu 2 | half1 3 | half2 3]; force_out: [n(8); (tx,ty)(8)]
template <typename T>
CN_HD T elbow_loss_epilogue(const ElbowParams<T>& P, const ElbowProb<T>& S, const ElbowLossAux<T>& A, const T* u,
                            T* grad, T* force_out, T* grad_pts) {
  T f[24], z[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  T qf = T(0), ff = T(0), fmax = T(0);
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = P.mu[c >> 2];
    T r[3];
    elbow_residual(P, S, c, u, r);
    cone_eval<T, false>(r, P.inv_eps, mu, f + 3 * c, (T*)nullptr);
    const T ft[3] = {mu * f[3 * c], mu * f[3 * c + 1], f[3 * c + 2]};
    T tq[3];
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
    cross3(rho, ft, tq);
    for (int i = 0; i < 3; ++i) {
      z[i] += tq[i]; z[3 + i] += ft[i];
      qf += S.q(3 * c + i) * f[3 * c + i]; ff += f[3 * c + i] * f[3 * c + i];
      const T af = t_abs(f[3 * c + i]);
      fmax = (af > fmax || af != af) ? af : fmax;
    }
    const T hc[3] = {S.hc(3 * c), S.hc(3 * c + 1), S.hc(3 * c + 2)};
    z[6] += dot3(hc, ft);
  }
  if (!(fmax <= T(1e3))) {
    if (force_out) for (int i = 0; i < 24; ++i) force_out[i] = T(0);
    if (grad_pts) for (int i = 0; i < 24; ++i) grad_pts[i] = T(0);
    return T(0);
  }
  if (force_out)
    for (int c = 0; c < EL_NC; ++c) {
      force_out[c] = f[3 * c + 2]; force_out[8 + 2 * c] = f[3 * c]; force_out[8 + 2 * c + 1] = f[3 * c + 1];
    }
  T y[7];
  chol_solve<T, 7>(A.LM, A.LMinv, z, y);
  T zy = T(0);
  for (int i = 0; i < 7; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + A.konst;
  if (!grad) return loss;

  // ---- envelope backward in world-twist coordinates ----
  T lam[7], b[7];
  for (int i = 0; i < 7; ++i) { b[i] = y[i] - A.dv[i]; lam[i] = P.dt * b[i]; }
  // Mbar = -1/2 y y^T + 1/2 dv dv^T - lam a^T   (7x7, as autograd gives for an unconstrained M)
  T Mbar[49];
  for (int i = 0; i < 7; ++i)
    for (int j = 0; j < 7; ++j) Mbar[7 * i + j] = T(0.5) * (A.dv[i] * A.dv[j] - y[i] * y[j]) - lam[i] * A.acc[j];
  for (int bi = 0; bi < 2; ++bi) {
    // Mbar_i = T_i Mbar T_i^T (6x6), lam_i = T_i lam;  T_1 = [I6 | 0]
    T Mi[36], li[6], wW[3];
    if (bi == 0) {
      for (int i = 0; i < 6; ++i) {
        li[i] = lam[i];
        for (int j = 0; j < 6; ++j) Mi[6 * i + j] = Mbar[7 * i + j];
      }
      for (int i = 0; i < 3; ++i) wW[i] = A.vp[i];
    } else {
      T tmp[42];   // (Mbar T2^T): 7 x 6, row i = T2 applied to row i of Mbar
      for (int i = 0; i < 7; ++i) elbow_T2(A.K, Mbar + 7 * i, tmp + 6 * i);
      for (int j = 0; j < 6; ++j) {
        T col[7], V[6];
        for (int i = 0; i < 7; ++i) col[i] = tmp[6 * i + j];
        elbow_T2(A.K, col, V);
        for (int i = 0; i < 6; ++i) Mi[6 * i + j] = V[i];
      }
      elbow_T2(A.K, lam, li);
      // F = ... - T2^T M_2 b_2  =>  Mbar_2 += -lam_2 b_2^T
      for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) Mi[6 * i + j] -= li[i] * A.b2[j];
      for (int i = 0; i < 3; ++i) wW[i] = A.vp[i] + A.K.aW[i] * A.vp[6];
    }
    // to body-i coordinates: angular parts rotated by R_i^T
    const T* R = A.K.R[bi];
    T Kww[9], N[9], trvv = T(0), lamB[6], wB[3];
    // Kww = R^T Mi_ww R ;  Mwv_B = R^T Mi_wv ;  Mvw_B = Mi_vw R
    T t1[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) t1[3 * i + j] = Mi[6 * i] * R[j] + Mi[6 * i + 1] * R[3 + j] + Mi[6 * i + 2] * R[6 + j];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) Kww[3 * i + j] = R[i] * t1[j] + R[3 + i] * t1[3 + j] + R[6 + i] * t1[6 + j];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        const T wv = R[i] * Mi[3 + j] + R[3 + i] * Mi[6 + 3 + j] + R[6 + i] * Mi[12 + 3 + j];          // (R^T Mi_wv)_{ij}
        const T vw = Mi[6 * (3 + j)] * R[i] + Mi[6 * (3 + j) + 1] * R[3 + i] + Mi[6 * (3 + j) + 2] * R[6 + i];  // (Mi_vw R)_{ji}
        N[3 * i + j] = wv + vw;
      }
    for (int i = 0; i < 3; ++i) trvv += Mi[6 * (3 + i) + 3 + i];
    rot3t(R, li, lamB);
    for (int i = 0; i < 3; ++i) lamB[3 + i] = li[3 + i];
    rot3t(R, wW, wB);
    rigid_body_inertia_adjoint<T>(P.body[bi].m, P.body[bi].c, R, wB, P.grav, Kww, N, trvv, lamB, grad + 10 * bi);
  }
  // contacts: mu per pair, half lengths per box
  for (int c = 0; c < EL_NC; ++c) {
    const int bi = c >> 2, cl = c & 3;
    const T mu = P.mu[bi];
    const T* R = A.K.R[bi];
    T eb[3], ev[3];
    elbow_point_vel(S, c, b, eb);
    elbow_point_vel(S, c, A.vp, ev);
    const T ftx = f[3 * c], fty = f[3 * c + 1], fn = f[3 * c + 2];
    const T sx = mu * ev[0], sy = mu * ev[1];
    const T sinv = t_rsqrt(t_max(sx * sx + sy * sy, t_tiny<T>()));
    const T ux = sx * sinv, uy = sy * sinv;
    const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
    grad[20 + bi] += ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
    const T ft[3] = {mu * ftx, mu * fty, fn};
    const T gt[3] = {mu * gx, mu * gy, T(0)};
    // angular velocities of body bi induced by b and by v+ (world), then body frame
    T Ob[3], Ov[3];
    for (int i = 0; i < 3; ++i) {
      Ob[i] = b[i] + (bi ? A.K.aW[i] * b[6] : T(0));
      Ov[i] = A.vp[i] + (bi ? A.K.aW[i] * A.vp[6] : T(0));
    }
    T ftB[3], gtB[3], ObB[3], OvB[3], p1[3], p2[3];
    rot3t(R, ft, ftB); rot3t(R, gt, gtB); rot3t(R, Ob, ObB); rot3t(R, Ov, OvB);
    cross3(ftB, ObB, p1); cross3(gtB, OvB, p2);
    const T phic = S.rho(3 * c + 2) + A.pos_z;
    const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - T(2) * t_max(-phic, T(0));
    for (int k = 0; k < 3; ++k) {
      const T pbar = p1[k] + p2[k] + phibar * R[6 + k];      // d loss / d (witness point, geometry frame)
      if (grad_pts) grad_pts[3 * c + k] = pbar;
      else grad[22 + 3 * bi + k] += sgn_bit<T>(A.K.sel[bi], cl, k) * pbar;
    }
  }
  return loss;
}

template <typename T>
CN_HD T elbow_loss_sample(const ElbowParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, const T* pts,
                          T* grad, T* force_out, T* grad_pts, int* iters_out) {
  T store[ELBOW_PROB_FIELDS];
  const ElbowProb<T> S{store, 1};
  ElbowLossAux<T> A;
  elbow_loss_prologue(P, x, xp, pts, S, A);
  T u[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  const int it = elbow_solve(P, S, cfg, u);
  if (iters_out) *iters_out = it;
  if (!grad && grad_pts) for (int i = 0; i < 24; ++i) grad_pts[i] = T(0);
  return elbow_loss_epilogue(P, S, A, u, grad, force_out, grad ? grad_pts : (T*)nullptr);
}

// ---------------------------------------------------------------------------
// learnable time step
// ---------------------------------------------------------------------------
template <typename T>
CN_HD int elbow_step_sample(const ElbowParams<T>& P, const SolverCfg<T>& cfg, const T* x, const T* pts, T* xn,
                            T* force_out, T* u_out = nullptr) {
  // u_out: receives the QP optimum u* (world twist + hinge rate; v+ = v- + u*).
  T store[ELBOW_PROB_FIELDS];
  const ElbowProb<T> S{store, 1};
  ElbowKin<T> K;
  elbow_kinematics(P, x, K);
  T vW[7], F[7], LM[49], LMinv[7], acc[7], vm[7];
  elbow_to_world(K.R[0], x + 8, vW);
  elbow_mass_force(P, K, vW, LM, F, (T*)nullptr);
  for (int i = 0; i < 49; ++i) S.M(i) = LM[i];
  chol_factor<T, 7>(LM, LMinv);
  chol_solve<T, 7>(LM, LMinv, F, acc);
  for (int i = 0; i < 7; ++i) vm[i] = vW[i] + P.dt * acc[i];
  elbow_contacts(P, K, S, pts);
  const T inv_dt = T(1) / P.dt;
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = P.mu[c >> 2];
    T e[3];
    elbow_point_vel(S, c, vm, e);
    S.q(3 * c) = mu * e[0];
    S.q(3 * c + 1) = mu * e[1];
    S.q(3 * c + 2) = e[2] + (S.rho(3 * c + 2) + x[6]) * inv_dt;
  }
  T u[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
  const int it = elbow_solve(P, S, cfg, u);
  if (u_out) for (int i = 0; i < 7; ++i) u_out[i] = u[i];
  if (force_out)
    for (int c = 0; c < EL_NC; ++c) {
      T r[3], f[3];
      elbow_residual(P, S, c, u, r);
      cone_eval<T, false>(r, P.inv_eps, P.mu[c >> 2], f, (T*)nullptr);
      force_out[c] = f[2]; force_out[8 + 2 * c] = f[0]; force_out[8 + 2 * c + 1] = f[1];
    }
  // v+ = v- + u (world twist) -> state coordinates
  T vnW[7], vn[7];
  for (int i = 0; i < 7; ++i) vnW[i] = vm[i] + u[i];
  rot3t(K.R[0], vnW, vn);
  for (int i = 3; i < 7; ++i) vn[i] = vnW[i];
  const T rx = vn[0] * P.dt, ry = vn[1] * P.dt, rz = vn[2] * P.dt;
  const T ang = t_sqrt(rx * rx + ry * ry + rz * rz);
  const T half = T(0.5) * ang;
  const T sinc = half > T(0) ? sin(half) / half : T(1);
  const T dw = cos(half), k = T(0.5) * sinc;
  const T dx = rx * k, dy = ry * k, dz = rz * k;
  const T qw = x[0], qx = x[1], qy = x[2], qz = x[3];
  xn[0] = qw * dw - (qx * dx + qy * dy + qz * dz);
  xn[1] = qw * dx + dw * qx + (qy * dz - qz * dy);
  xn[2] = qw * dy + dw * qy + (qz * dx - qx * dz);
  xn[3] = qw * dz + dw * qz + (qx * dy - qy * dx);
  for (int i = 0; i < 3; ++i) xn[4 + i] = x[4 + i] + vn[3 + i] * P.dt;
  xn[7] = x[7] + vn[6] * P.dt;
  for (int i = 0; i < 7; ++i) xn[8 + i] = vn[i];
  return it;
}

// ---------------------------------------------------------------------------
// Dense dynamics terms of the two-body system in the reference's own coordinates and ordering, for callers of
// MultibodyTerms.forward (multibody_terms.py:584-609): M (7x7), J (24x7) = [J_n (8 rows) ; mu J_t (x,y interleaved
// per contact, 16 rows)] (:401-426), phi (8), contact-free acceleration (7), Delassus operator D = J M^-1 J^T
// (24x24).  Contacts: box 1 then box 2, each by ascending vertex index.  State velocity v = [w_body1 ; v_world ;
// hinge rate] = T^T u^ with T = blkdiag(R1, I3, 1) (orthogonal), so M = T^T M^ T, J = J^ T, a = T^T a^.
// ---------------------------------------------------------------------------
template <typename T>
CN_HD void elbow_terms_sample(const ElbowParams<T>& P, const T* q, const T* v, T* M, T* J, T* phi, T* acc, T* D) {
  T store[ELBOW_PROB_FIELDS];
  const ElbowProb<T> S{store, 1};
  ElbowKin<T> K;
  elbow_kinematics(P, q, K);
  T vW[7], F[7], MW[49], LM[49], LMinv[7], aW[7];
  elbow_to_world(K.R[0], v, vW);
  elbow_mass_force(P, K, vW, MW, F, (T*)nullptr);
  for (int i = 0; i < 49; ++i) LM[i] = MW[i];
  chol_factor<T, 7>(LM, LMinv);
  chol_solve<T, 7>(LM, LMinv, F, aW);
  const T* R = K.R[0];
  rot3t(R, aW, acc);
  for (int i = 3; i < 7; ++i) acc[i] = aW[i];
  // M = T^T M^ T: rotate the angular rows and columns into body-1 coordinates
  T tmp[49];
  for (int i = 0; i < 7; ++i) {                       // tmp = M^ T  (columns 0..2 rotated)
    const T* row = MW + 7 * i;
    for (int j = 0; j < 3; ++j) tmp[7 * i + j] = row[0] * R[j] + row[1] * R[3 + j] + row[2] * R[6 + j];
    for (int j = 3; j < 7; ++j) tmp[7 * i + j] = row[j];
  }
  for (int j = 0; j < 7; ++j) {                       // M = T^T tmp  (rows 0..2 rotated)
    for (int i = 0; i < 3; ++i) M[7 * i + j] = R[i] * tmp[j] + R[3 + i] * tmp[7 + j] + R[6 + i] * tmp[14 + j];
    for (int i = 3; i < 7; ++i) M[7 * i + j] = tmp[7 * i + j];
  }
  elbow_contacts(P, K, S, (const T*)nullptr);
  for (int c = 0; c < EL_NC; ++c) {
    const T mu = P.mu[c >> 2];
    const T rho[3] = {S.rho(3 * c), S.rho(3 * c + 1), S.rho(3 * c + 2)};
    phi[c] = rho[2] + q[6];
    // world rows of J^_c = [-S(rho), I3, h]; angular block in state coordinates: (-S(rho)) R1
    T E[9];
    for (int j = 0; j < 3; ++j) {
      const T col[3] = {R[j], R[3 + j], R[6 + j]};
      T cr[3];
      cross3(rho, col, cr);
      for (int i = 0; i < 3; ++i) E[3 * i + j] = -cr[i];
    }
    T* jn = J + 7 * c;
    T* jx = J + 7 * (EL_NC + 2 * c);
    T* jy = J + 7 * (EL_NC + 2 * c + 1);
    for (int j = 0; j < 3; ++j) {
      jn[j] = E[6 + j]; jx[j] = mu * E[j]; jy[j] = mu * E[3 + j];
      jn[3 + j] = j == 2 ? T(1) : T(0);
      jx[3 + j] = j == 0 ? mu : T(0);
      jy[3 + j] = j == 1 ? mu : T(0);
    }
    jn[6] = S.hc(3 * c + 2); jx[6] = mu * S.hc(3 * c); jy[6] = mu * S.hc(3 * c + 1);
  }
  if (D) {
    // D = J M^-1 J^T with M = L L^T (Cholesky of the state-coordinate M): W = L^-1 J^T, D = W^T W
    T LS[49], LSinv[7], W[7 * EL_K];
    for (int i = 0; i < 49; ++i) LS[i] = M[i];
    chol_factor<T, 7>(LS, LSinv);
    for (int r = 0; r < EL_K; ++r)
      for (int i = 0; i < 7; ++i) {
        T s = J[7 * r + i];
        for (int m = 0; m < i; ++m) s -= LS[7 * i + m] * W[EL_K * m + r];
        W[EL_K * i + r] = s * LSinv[i];
      }
    for (int a = 0; a < EL_K; ++a)
      for (int b = 0; b <= a; ++b) {
        T s = T(0);
        for (int k = 0; k < 7; ++k) s += W[EL_K * k + a] * W[EL_K * k + b];
        D[EL_K * a + b] = s;
        D[EL_K * b + a] = s;
      }
  }
}

}  // namespace cn
