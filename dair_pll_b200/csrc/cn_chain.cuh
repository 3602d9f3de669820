// Generic floating-base kinematic TREE of N rigid links joined by N-1 revolute joints (a serial chain or a branching tree:
// link b > 0 hangs off link par(b) < b), one box geometry per link against the ground plane: n_q = 7 + (N-1),
// n_v = 6 + (N-1), 4 N contacts.  SURVEY.md section 8(f) N2, first slice: what the
// reference derives symbolically for ANY plant (multibody_terms.py:114-157 mass matrix / bias forces, :267-319 geometry
// rotations / translations / spatial Jacobians) evaluated here by recursion over the links instead of per-asset closed
// forms -- joint frames may be rotated against their parent link (URDF <origin rpy>), inertial frames are rotated on
// the host.  The hand-derived two-body kernels are the N = 2 instance and this code reproduces their goldens.
//
// Same reference spans as cn_elbow.cuh for everything downstream of the terms (contactnets_loss
// multibody_learnable_system.py:104-197, forward_dynamics :199-304, top-k support geometry.py:162-202, plane-convex
// collision :553-582, the cone QP of sappy); same internal coordinates, world twist of link 0 plus the joint rates:
//   u^ = [w_W0 ; v_W(o_0) ; td_1 .. td_{N-1}] = blkdiag(R_0, I3, I) v_state.
// Link i with parent p = par(i) (serial chain: p = i - 1) and ancestor joints anc(i) = the joints on the path root -> i:
//   R_i = R_p Rfix_i Rot(axis_i, theta_i),  o_i = o_p + R_p pJ_i,  a_i = R_p Rfix_i axis_i,
//   twist   w_i = w_0 + sum_{j in anc(i)} a_j td_j,   v_i = v_0 + w_0 x o_i + sum_{j in anc(i)} td_j a_j x (o_i - o_j)   (= T_i u^)
//   bias    al_i = al_p + (w_p x a_i) td_i,   be_i = be_p + al_p x r_i + w_p x (w_p x r_i),   r_i = o_i - o_p
//   M^ = sum_i T_i^T M_i T_i,   F^ = sum_i T_i^T (F_i - M_i [al_i ; be_i])      (M_i, F_i as in cn_elbow.cuh)
// Contact c on link i:  J_c = [-S(rho_c), I3, a_j x (rho_c - o_j) for j in anc(i), 0 otherwise].
// A PRISMATIC joint i (URDF type="prismatic") keeps the joint frame's orientation and slides the child along a_i:
//   R_i = R_p Rfix_i,  o_i = o_p + R_p pJ_i + a_i q_i;  its column of T and of J_c is [0 ; a_i] (no lever arm);
//   al_i = al_p,  be_i = be_p + al_p x r_i + w_p x (w_p x r_i) + 2 (w_p x a_i) td_i.
// Plain per-thread arrays and loops: this is the general path (one sample per thread), not a tuned one.
#pragma once
#include "cn_elbow.cuh"

namespace cn {

constexpr double CH_OFF = 1e6;  // normal entry of the QP vector of an empty box slot's contacts (m/s; deep in the polar cone)
constexpr int CH_NKIN = 31;     // row b = link b: [joint origin 3 | joint rpy as rotation matrix 9 | axis 3 | . | parent link | . |
                                //   joint type: 0 revolute, 1 prismatic] and box SLOT b: [box offset 3 (entries 15-17) | rotation
                                //   link <- collision frame 9 (19-27) | link the box sits on (29) | slot in use (30)]

template <typename T, int N> struct ChainParams {
  static constexpr int NV = 6 + N - 1, NC = 4 * N, K = 3 * NC;
  ElbowBody<T> body[N];
  T mu[N], h[N][3], off[N][3];
  T pJ[N][3], Rfix[N][9], axis[N][3];      // entry 0 unused
  T Rg[N][9];                              // rotation link frame <- collision (box) frame (URDF <collision><origin rpy>)
  int par[N];                              // parent link (par[b] < b; entry 0 unused)
  unsigned anc[N];                         // bit j set: joint j (1..N-1) lies on the path from the root to link b
  unsigned pris;                           // bit j set: joint j slides along its axis (prismatic) instead of turning
  int glink[N];                            // box slot g sits on link glink[g] (any distribution of <= N boxes over the links)
  unsigned gon;                            // bit g set: slot g holds a box (its four contacts exist)
  T dt, eps, inv_eps, grav;
  T dscale[6 + N - 1];
};

// inertia: N x 10, mu: N, half: N x 3 (nullable: witness-point entry points), kin: N x CH_NKIN
template <typename T, int N>
CN_HD void chain_params_init(ChainParams<T, N>& P, const T* inertia, const T* mu, const T* half, const T* kin, T dt, T eps) {
  T msum = T(0), Isum[3] = {T(0), T(0), T(0)};
  P.pris = 0u; P.gon = 0u;
  for (int b = 0; b < N; ++b) {
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
    const T* kn = kin + CH_NKIN * b;
    for (int i = 0; i < 3; ++i) { P.h[b][i] = half ? half[3 * b + i] : T(0); P.pJ[b][i] = kn[i]; P.axis[b][i] = kn[12 + i]; P.off[b][i] = kn[15 + i]; }
    for (int i = 0; i < 9; ++i) { P.Rfix[b][i] = kn[3 + i]; P.Rg[b][i] = kn[19 + i]; }
    // parent index travels as a number in the table; clamped to [0, b - 1] so that a bad table cannot index out of range
    int pb = b > 0 ? (int)to_double(kn[18]) : 0;
    pb = pb < 0 ? 0 : (pb > b - 1 ? (b > 0 ? b - 1 : 0) : pb);
    P.par[b] = pb;
    P.anc[b] = b > 0 ? (P.anc[pb] | (1u << b)) : 0u;
    if (b > 0 && to_double(kn[28]) > 0.5) P.pris |= 1u << b;
    int gl = (int)to_double(kn[29]);
    P.glink[b] = gl < 0 ? 0 : (gl > N - 1 ? N - 1 : gl);
    if (to_double(kn[30]) > 0.5) P.gon |= 1u << b;
    msum += B.m;
    for (int i = 0; i < 3; ++i) Isum[i] += B.Io[i];
  }
  P.dt = dt; P.eps = eps; P.inv_eps = T(1) / eps; P.grav = T(9.81);
  for (int i = 0; i < 3; ++i) { P.dscale[i] = T(1) / Isum[i]; P.dscale[3 + i] = T(1) / msum; }
  for (int j = 1; j < N; ++j) P.dscale[5 + j] = ((P.pris >> j) & 1u) ? T(1) / P.body[j].m : T(1) / P.body[j].Io[1];
}

template <typename T, int N> struct ChainKin {
  T R[N][9], o[N][3], a[N][3];      // world rotations, origins relative to o_0, joint axes (a[0] unused)
  uint32_t sel[N];
  unsigned anc[N], pris;            // copies of ChainParams::anc / pris (the twist maps below take only the kinematics)
};

template <typename T, int N> CN_HD void chain_kinematics(const ChainParams<T, N>& P, const T* q, ChainKin<T, N>& K) {
  quat_to_rot(q, K.R[0]);
  for (int i = 0; i < 3; ++i) { K.o[0][i] = T(0); K.a[0][i] = T(0); }
  for (int b = 0; b < N; ++b) K.anc[b] = P.anc[b];
  K.pris = P.pris;
  for (int b = 1; b < N; ++b) {
    T Rjf[9], Rj[9], r[3];
    const int p = P.par[b];
    mat3_mul(K.R[p], P.Rfix[b], Rjf);
    rot3(Rjf, P.axis[b], K.a[b]);
    rot3(K.R[p], P.pJ[b], r);
    if ((P.pris >> b) & 1u) {
      for (int i = 0; i < 9; ++i) K.R[b][i] = Rjf[i];
      for (int i = 0; i < 3; ++i) K.o[b][i] = K.o[p][i] + r[i] + K.a[b][i] * q[6 + b];
    } else {
      axis_angle_rot(P.axis[b], q[6 + b], Rj);
      mat3_mul(Rjf, Rj, K.R[b]);
      for (int i = 0; i < 3; ++i) K.o[b][i] = K.o[p][i] + r[i];
    }
  }
}

// V = T_b u (6) for world twist u (NV)
template <typename T, int N> CN_HD void chain_T(const ChainKin<T, N>& K, int b, const T* u, T* V) {
  T wxo[3];
  cross3(u, K.o[b], wxo);
  for (int i = 0; i < 3; ++i) { V[i] = u[i]; V[3 + i] = u[3 + i] + wxo[i]; }
  for (int j = 1; j <= b; ++j) {
    if (!((K.anc[b] >> j) & 1u)) continue;
    if ((K.pris >> j) & 1u) {
      for (int i = 0; i < 3; ++i) V[3 + i] += K.a[j][i] * u[5 + j];
      continue;
    }
    T d[3], axd[3];
    for (int i = 0; i < 3; ++i) d[i] = K.o[b][i] - K.o[j][i];
    cross3(K.a[j], d, axd);
    for (int i = 0; i < 3; ++i) { V[i] += K.a[j][i] * u[5 + j]; V[3 + i] += axd[i] * u[5 + j]; }
  }
}

// o (NV) = T_b^T W for a wrench W = [tau ; f] about o_b
template <typename T, int N> CN_HD void chain_Tt(const ChainKin<T, N>& K, int b, const T* W, T* o) {
  T oxf[3];
  cross3(K.o[b], W + 3, oxf);
  for (int i = 0; i < 3; ++i) { o[i] = W[i] + oxf[i]; o[3 + i] = W[3 + i]; }
  for (int j = 1; j < N; ++j) {
    if (((K.anc[b] >> j) & 1u) && ((K.pris >> j) & 1u)) {
      o[5 + j] = dot3(K.a[j], W + 3);
    } else if ((K.anc[b] >> j) & 1u) {
      T d[3], axd[3];
      for (int i = 0; i < 3; ++i) d[i] = K.o[b][i] - K.o[j][i];
      cross3(K.a[j], d, axd);
      o[5 + j] = dot3(K.a[j], W) + dot3(axd, W + 3);
    } else {
      o[5 + j] = T(0);
    }
  }
}

// M^ (NV x NV, full) and F^ (NV) at world twist uW; bias (N x 6, nullable): the links' velocity-product accelerations
template <typename T, int N>
CN_HD void chain_mass_force(const ChainParams<T, N>& P, const ChainKin<T, N>& K, const T* uW, T* M, T* F, T* bias_out) {
  constexpr int NV = 6 + N - 1;
  for (int i = 0; i < NV * NV; ++i) M[i] = T(0);
  for (int i = 0; i < NV; ++i) F[i] = T(0);
  const T g[3] = {T(0), T(0), -P.grav};
  T wl[N][3], all[N][3], bel[N][3];       // per link: angular velocity, velocity-product accelerations
  for (int b = 0; b < N; ++b) {
    const ElbowBody<T>& B = P.body[b];
    T Mi[36], cW[3], V[6], bias[6];
    body_mass_world(B, K.R[b], Mi, cW);
    chain_T<T, N>(K, b, uW, V);
    if (b > 0) {
      // al_b = al_p + (w_p x a_b) td_b ;  be_b = be_p + al_p x r_b + w_p x (w_p x r_b),  p = parent of b
      const int p = P.par[b];
      T r[3], wxa[3], alxr[3], wxr[3], wwr[3];
      for (int i = 0; i < 3; ++i) r[i] = K.o[b][i] - K.o[p][i];
      cross3(wl[p], K.a[b], wxa);
      cross3(all[p], r, alxr);
      cross3(wl[p], r, wxr); cross3(wl[p], wxr, wwr);
      if ((P.pris >> b) & 1u) {
        for (int i = 0; i < 3; ++i) { bel[b][i] = bel[p][i] + alxr[i] + wwr[i] + T(2) * wxa[i] * uW[5 + b]; }
        for (int i = 0; i < 3; ++i) { all[b][i] = all[p][i]; }
      } else {
        for (int i = 0; i < 3; ++i) { bel[b][i] = bel[p][i] + alxr[i] + wwr[i]; }
        for (int i = 0; i < 3; ++i) { all[b][i] = all[p][i] + wxa[i] * uW[5 + b]; }
      }
    } else {
      for (int i = 0; i < 3; ++i) { all[0][i] = T(0); bel[0][i] = T(0); }
    }
    for (int i = 0; i < 3; ++i) { bias[i] = all[b][i]; bias[3 + i] = bel[b][i]; wl[b][i] = V[i]; }
    if (bias_out) for (int i = 0; i < 6; ++i) bias_out[6 * b + i] = bias[i];
    T Iw[3], wIw[3], cg[3], wc[3], wwc[3], Fi[6];
    for (int i = 0; i < 3; ++i) Iw[i] = Mi[6 * i] * V[0] + Mi[6 * i + 1] * V[1] + Mi[6 * i + 2] * V[2];
    cross3(V, Iw, wIw);
    cross3(cW, g, cg);
    cross3(V, cW, wc); cross3(V, wc, wwc);
    for (int i = 0; i < 3; ++i) { Fi[i] = -wIw[i] + B.m * cg[i]; Fi[3 + i] = -B.m * wwc[i] + B.m * g[i]; }
    for (int i = 0; i < 6; ++i) {
      T s = T(0);
      for (int j = 0; j < 6; ++j) s += Mi[6 * i + j] * bias[j];
      Fi[i] -= s;
    }
    T f7[NV];
    chain_Tt<T, N>(K, b, Fi, f7);
    for (int i = 0; i < NV; ++i) F[i] += f7[i];
    for (int j = 0; j < NV; ++j) {
      T ej[NV], Vj[6], MV[6], col[NV];
      for (int i = 0; i < NV; ++i) ej[i] = T(0);
      ej[j] = T(1);
      chain_T<T, N>(K, b, ej, Vj);
      for (int i = 0; i < 6; ++i) {
        T s = T(0);
        for (int m = 0; m < 6; ++m) s += Mi[6 * i + m] * Vj[m];
        MV[i] = s;
      }
      chain_Tt<T, N>(K, b, MV, col);
      for (int i = 0; i < NV; ++i) M[NV * i + j] += col[i];
    }
  }
}

// per-sample record (local array): M (NV^2) | rho (3 NC) | hc (3 NC (N-1)) | q (3 NC)
template <typename T, int N> struct ChainProb {
  static constexpr int NV = 6 + N - 1, NC = 4 * N;
  T M[NV * NV], rho[3 * NC], hc[3 * NC * (N - 1) + 1], q[3 * NC];
  unsigned con;     // bit c set: contact c exists (box slots in use: all four corners; witness points: the first n of a slot)
};

// pts (nullable, 12 N): WITNESS POINTS instead of box corners -- contact c of slot b is the point pts[3 (4 b + c) ..] given in
// the frame of the slot's link (the caller evaluates the shapes' support points in the direction -R_link^T e_z and places them:
// a sphere's single point, a polygon's top vertices, a network's outputs, box corners in any collision frame); npts packs
// the number of points of slot b in bits 3 b .. 3 b + 2 (0 .. 4).  Same contact machinery downstream.
template <typename T, int N>
CN_HD void chain_contacts(const ChainParams<T, N>& P, ChainKin<T, N>& K, ChainProb<T, N>& S, const T* pts = nullptr,
                          unsigned npts = 0u) {
  S.con = 0u;
  for (int b = 0; b < N; ++b) {             // b: box slot; l: the link it sits on
    const int l = P.glink[b];
    if (pts) {
      const int np = (int)((npts >> (3 * b)) & 7u);
      K.sel[b] = 0u;
      for (int c = 0; c < 4; ++c) {
        const int cc = 4 * b + c;
        const bool on = ((P.gon >> b) & 1u) && c < np;
        T r[3] = {T(0), T(0), T(0)};
        if (on) { rot3(K.R[l], pts + 3 * cc, r); S.con |= 1u << cc; }
        for (int i = 0; i < 3; ++i) S.rho[3 * cc + i] = on ? K.o[l][i] + r[i] : T(0);
        for (int j = 1; j < N; ++j) {
          T hcol[3] = {T(0), T(0), T(0)};
          if (on && ((K.anc[l] >> j) & 1u) && ((K.pris >> j) & 1u)) {
            for (int i = 0; i < 3; ++i) hcol[i] = K.a[j][i];
          } else if (on && ((K.anc[l] >> j) & 1u)) {
            T dd[3];
            for (int i = 0; i < 3; ++i) dd[i] = S.rho[3 * cc + i] - K.o[j][i];
            cross3(K.a[j], dd, hcol);
          }
          for (int i = 0; i < 3; ++i) S.hc[3 * (cc * (N - 1) + (j - 1)) + i] = hcol[i];
        }
      }
      continue;
    }
    if (!((P.gon >> b) & 1u)) {
      // empty slot: its four contacts get a zero Jacobian here and a residual deep in the polar cone where the QP vector is
      // built (zero force, zero curvature), and take no part in the loss
      K.sel[b] = 0u;
      for (int c = 0; c < 4; ++c) {
        const int cc = 4 * b + c;
        for (int i = 0; i < 3; ++i) S.rho[3 * cc + i] = T(0);
        for (int j = 1; j < N; ++j)
          for (int i = 0; i < 3; ++i) S.hc[3 * (cc * (N - 1) + (j - 1)) + i] = T(0);
      }
      continue;
    }
    const T* R = K.R[l];
    // support direction -R_WG^T e_z in the box's own frame, R_WG = R_link Rg  (geometry.py:560-567)
    const T dl[3] = {-R[6], -R[7], -R[8]};
    T d[3];
    rot3t(P.Rg[b], dl, d);
    K.sel[b] = cube_select_corners(d, P.h[b]);
    S.con |= 15u << (4 * b);
    for (int c = 0; c < 4; ++c) {
      T pg[3], p[3], r[3];
      for (int k = 0; k < 3; ++k) pg[k] = sgn_bit<T>(K.sel[b], c, k) * P.h[b][k];
      rot3(P.Rg[b], pg, p);
      for (int k = 0; k < 3; ++k) p[k] += P.off[b][k];
      rot3(R, p, r);
      const int cc = 4 * b + c;
      for (int i = 0; i < 3; ++i) S.rho[3 * cc + i] = K.o[l][i] + r[i];
      for (int j = 1; j < N; ++j) {
        T hcol[3] = {T(0), T(0), T(0)};
        if (((K.anc[l] >> j) & 1u) && ((K.pris >> j) & 1u)) {
          for (int i = 0; i < 3; ++i) hcol[i] = K.a[j][i];
        } else if ((K.anc[l] >> j) & 1u) {
          T dd[3];
          for (int i = 0; i < 3; ++i) dd[i] = S.rho[3 * cc + i] - K.o[j][i];
          cross3(K.a[j], dd, hcol);
        }
        for (int i = 0; i < 3; ++i) S.hc[3 * (cc * (N - 1) + (j - 1)) + i] = hcol[i];
      }
    }
  }
}

template <typename T, int N> CN_HD void chain_point_vel(const ChainProb<T, N>& S, int c, const T* u, T* e) {
  const T rho[3] = {S.rho[3 * c], S.rho[3 * c + 1], S.rho[3 * c + 2]};
  cross3(u, rho, e);
  for (int i = 0; i < 3; ++i) e[i] += u[3 + i];
  for (int j = 1; j < N; ++j)
    for (int i = 0; i < 3; ++i) e[i] += S.hc[3 * (c * (N - 1) + (j - 1)) + i] * u[5 + j];
}

template <typename T, int N, bool WANT_H>
CN_HD void chain_eval(const ChainParams<T, N>& P, const ChainProb<T, N>& S, const T* u, T* g, T* H, T& res2, T& scale2) {
  constexpr int NV = 6 + N - 1, NC = 4 * N;
  T Mu[NV], z[NV];
  for (int i = 0; i < NV; ++i) {
    T s = T(0);
    for (int j = 0; j < NV; ++j) s += S.M[NV * i + j] * u[j];
    Mu[i] = s; z[i] = T(0);
  }
  if (WANT_H) for (int i = 0; i < NV * NV; ++i) H[i] = S.M[i];
  for (int c = 0; c < NC; ++c) {
    const T mu = P.mu[c >> 2];
    T e[3], r[3], f[3], Kc[6];
    chain_point_vel<T, N>(S, c, u, e);
    r[0] = mu * e[0] + S.q[3 * c]; r[1] = mu * e[1] + S.q[3 * c + 1]; r[2] = e[2] + S.q[3 * c + 2];
    cone_eval<T, WANT_H>(r, P.inv_eps, mu, f, Kc);
    const T ft[3] = {mu * f[0], mu * f[1], f[2]};
    // dense J_c (3 x NV)
    T J[3 * NV];
    const T rho[3] = {S.rho[3 * c], S.rho[3 * c + 1], S.rho[3 * c + 2]};
    J[0] = T(0);    J[1] = rho[2];  J[2] = -rho[1];
    J[NV] = -rho[2]; J[NV + 1] = T(0); J[NV + 2] = rho[0];
    J[2 * NV] = rho[1]; J[2 * NV + 1] = -rho[0]; J[2 * NV + 2] = T(0);
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k) J[NV * i + 3 + k] = i == k ? T(1) : T(0);
    for (int j = 1; j < N; ++j)
      for (int i = 0; i < 3; ++i) J[NV * i + 5 + j] = S.hc[3 * (c * (N - 1) + (j - 1)) + i];
    for (int i = 0; i < NV; ++i) z[i] += J[i] * ft[0] + J[NV + i] * ft[1] + J[2 * NV + i] * ft[2];
    if (WANT_H) {
      T KJ[3 * NV];
      for (int j = 0; j < NV; ++j) {
        KJ[j] = Kc[0] * J[j] + Kc[1] * J[NV + j] + Kc[2] * J[2 * NV + j];
        KJ[NV + j] = Kc[1] * J[j] + Kc[3] * J[NV + j] + Kc[4] * J[2 * NV + j];
        KJ[2 * NV + j] = Kc[2] * J[j] + Kc[4] * J[NV + j] + Kc[5] * J[2 * NV + j];
      }
      for (int i = 0; i < NV; ++i)
        for (int j = 0; j <= i; ++j) H[NV * i + j] += J[i] * KJ[j] + J[NV + i] * KJ[NV + j] + J[2 * NV + i] * KJ[2 * NV + j];
    }
  }
  res2 = T(0); T a2 = T(0), b2 = T(0);
  for (int i = 0; i < NV; ++i) {
    g[i] = Mu[i] - z[i];
    res2 += g[i] * g[i] * P.dscale[i];
    a2 += Mu[i] * Mu[i] * P.dscale[i];
    b2 += z[i] * z[i] * P.dscale[i];
  }
  scale2 = t_max(a2, b2);
}

// every contact's q in the polar cone: u = 0 is the exact optimum (free flight)
template <typename T, int N> CN_HD bool chain_open(const ChainProb<T, N>& S) {
  constexpr int NC = 4 * N;
  bool open = true;
  for (int c = 0; c < NC; ++c) {
    const T q0 = S.q[3 * c], q1 = S.q[3 * c + 1], qn = S.q[3 * c + 2];
    open = open && (qn >= T(0)) && (q0 * q0 + q1 * q1 <= qn * qn);
  }
  return open;
}

// the visit scheme of cube_newton_visit / elbow_solve, dimension NV, dense Cholesky.  Free flight returns at once and
// leaves u as it is.
template <typename T, int N>
CN_HD int chain_solve(const ChainParams<T, N>& P, const ChainProb<T, N>& S, const SolverCfg<T>& cfg, T* u) {
  constexpr int NV = 6 + N - 1;
  if (chain_open<T, N>(S)) return 0;
  int it = 0;
  T d[NV], d0 = T(0), best = T(-1);
  T alpha = T(1), lo = T(0), hi = T(1);
  while (true) {
    T g[NV], H[NV * NV], res2, scale2;
    chain_eval<T, N, true>(P, S, u, g, H, res2, scale2);
    if (cube_converged(cfg, res2, scale2)) {
      if (cfg.polish && res2 == res2) {
        T inv_diag[NV], ng[NV];
        chol_factor<T, NV>(H, inv_diag);
        for (int i = 0; i < NV; ++i) ng[i] = -g[i];
        chol_solve<T, NV>(H, inv_diag, ng, d);
        for (int i = 0; i < NV; ++i) u[i] += d[i];
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
      for (int i = 0; i < NV; ++i) d1 += g[i] * d[i];
      const T thresh = -cfg.ls_c * d0;
      const bool accept = trials == 0 ? (d1 <= thresh) : (t_abs(d1) <= thresh);
      if (!accept) {
        if (d1 < T(0)) lo = alpha; else hi = alpha;
        T d2 = T(0);
        for (int i = 0; i < NV; ++i) {
          T row = T(0);
          for (int j = 0; j < NV; ++j) row += H[j <= i ? NV * i + j : NV * j + i] * d[j];
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
        for (int i = 0; i < NV; ++i) u[i] += step * d[i];
        alpha = an;
        it = (it & ~0xff00) | (nt << 8);
        continue;
      }
    }
    if ((it & 0xff) >= cfg.max_iter) break;
    T inv_diag[NV], ng[NV];
    chol_factor<T, NV>(H, inv_diag);
    for (int i = 0; i < NV; ++i) ng[i] = -g[i];
    chol_solve<T, NV>(H, inv_diag, ng, d);
    T dd = T(0);
    for (int i = 0; i < NV; ++i) { dd += g[i] * d[i]; u[i] += d[i]; }
    d0 = dd < T(0) ? dd : T(0);
    alpha = T(1); lo = T(0); hi = T(1);
    it = (it & ~0xff00) + 1;
    if (res2 <= cfg.tol_final * cfg.tol_final * scale2) break;
  }
  return it & 0xff;
}

template <typename T, int N> CN_HD void chain_to_world(const T* R0, const T* v, T* u) {
  constexpr int NV = 6 + N - 1;
  rot3(R0, v, u);
  for (int i = 3; i < NV; ++i) u[i] = v[i];
}

// ContactNets loss + envelope backward.  grad layout (14 N): [inertia N x 10 | mu N | half N x 3]; force_out (3 NC,
// nullable): [n (NC); (tx, ty) (NC)].  u0 (NV, nullable): start point of the solve instead of u = 0 (a warm start);
// u_opt (NV, nullable): the optimum, 0 for free flight and for a sample whose forces are clipped (loss 0).
template <typename T, int N>
CN_HD T chain_loss_sample(const ChainParams<T, N>& P, const SolverCfg<T>& cfg, const T* x, const T* xp, T* grad,
                          T* force_out, int* iters_out, const T* pts = nullptr, unsigned npts = 0u, T* grad_pts = nullptr,
                          const T* u0 = nullptr, T* u_opt = nullptr) {
  constexpr int NV = 6 + N - 1, NC = 4 * N, NQ = 7 + N - 1;
  ChainKin<T, N> K;
  ChainProb<T, N> S;
  chain_kinematics<T, N>(P, xp, K);
  const T pos_z = xp[6];
  T vp[NV], vold[NV], F[NV], LM[NV * NV], LMinv[NV], acc[NV], dv[NV], bias[6 * N];
  chain_to_world<T, N>(K.R[0], xp + NQ, vp);
  chain_to_world<T, N>(K.R[0], x + NQ, vold);
  chain_mass_force<T, N>(P, K, vp, LM, F, bias);
  for (int i = 0; i < NV * NV; ++i) S.M[i] = LM[i];
  chol_factor<T, NV>(LM, LMinv);
  chol_solve<T, NV>(LM, LMinv, F, acc);
  for (int i = 0; i < NV; ++i) dv[i] = vp[i] - (vold[i] + P.dt * acc[i]);
  chain_contacts<T, N>(P, K, S, pts, npts);
  T pen = T(0);
  for (int c = 0; c < NC; ++c) {
    const T mu = P.mu[c >> 2];
    T ed[3], ev[3];
    chain_point_vel<T, N>(S, c, dv, ed);
    chain_point_vel<T, N>(S, c, vp, ev);
    const T sx = mu * ev[0], sy = mu * ev[1];
    const T speed2 = sx * sx + sy * sy;
    const T speed = speed2 * t_rsqrt(t_max(speed2, t_tiny<T>()));
    if (!((S.con >> c) & 1u)) {                   // no such contact: deep in the polar cone, no penetration term
      S.q[3 * c] = T(0); S.q[3 * c + 1] = T(0); S.q[3 * c + 2] = T(CH_OFF);
      continue;
    }
    const T phic = S.rho[3 * c + 2] + pos_z;
    S.q[3 * c] = -mu * ed[0] + P.dt * sx;
    S.q[3 * c + 1] = -mu * ed[1] + P.dt * sy;
    S.q[3 * c + 2] = -ed[2] + t_abs(phic) + P.dt * speed;
    const T pneg = t_max(-phic, T(0));
    pen += pneg * pneg;
  }
  T e = T(0);
  for (int i = 0; i < NV; ++i) {
    T s = T(0);
    for (int j = 0; j < NV; ++j) s += S.M[NV * i + j] * dv[j];
    e += dv[i] * s;
  }
  const T konst = T(0.5) * e + pen;
  T u[NV];
  for (int i = 0; i < NV; ++i) u[i] = T(0);
  // a start point counts only where there is something to solve: in free flight chain_solve leaves u as it is
  if (u0 && !chain_open<T, N>(S))
    for (int i = 0; i < NV; ++i) u[i] = u0[i];
  const int it = chain_solve<T, N>(P, S, cfg, u);
  if (iters_out) *iters_out = it;
  // forces, loss
  T f[3 * NC], z[NV];
  for (int i = 0; i < NV; ++i) z[i] = T(0);
  T qf = T(0), ff = T(0), fmax = T(0);
  for (int c = 0; c < NC; ++c) {
    const T mu = P.mu[c >> 2];
    T ev[3], r[3];
    chain_point_vel<T, N>(S, c, u, ev);
    r[0] = mu * ev[0] + S.q[3 * c]; r[1] = mu * ev[1] + S.q[3 * c + 1]; r[2] = ev[2] + S.q[3 * c + 2];
    cone_eval<T, false>(r, P.inv_eps, mu, f + 3 * c, (T*)nullptr);
    const T ft[3] = {mu * f[3 * c], mu * f[3 * c + 1], f[3 * c + 2]};
    const T rho[3] = {S.rho[3 * c], S.rho[3 * c + 1], S.rho[3 * c + 2]};
    T tq[3];
    cross3(rho, ft, tq);
    for (int i = 0; i < 3; ++i) {
      z[i] += tq[i]; z[3 + i] += ft[i];
      qf += S.q[3 * c + i] * f[3 * c + i]; ff += f[3 * c + i] * f[3 * c + i];
      const T af = t_abs(f[3 * c + i]);
      fmax = (af > fmax || af != af) ? af : fmax;
    }
    for (int j = 1; j < N; ++j) {
      const T* hcol = S.hc + 3 * (c * (N - 1) + (j - 1));
      z[5 + j] += hcol[0] * ft[0] + hcol[1] * ft[1] + hcol[2] * ft[2];
    }
  }
  if (!(fmax <= T(1e3))) {
    if (force_out) for (int i = 0; i < 3 * NC; ++i) force_out[i] = T(0);
    if (u_opt) for (int i = 0; i < NV; ++i) u_opt[i] = T(0);     // its next solve starts cold
    return T(0);
  }
  if (u_opt) for (int i = 0; i < NV; ++i) u_opt[i] = u[i];
  if (force_out)
    for (int c = 0; c < NC; ++c) {
      force_out[c] = f[3 * c + 2]; force_out[NC + 2 * c] = f[3 * c]; force_out[NC + 2 * c + 1] = f[3 * c + 1];
    }
  T y[NV];
  chol_solve<T, NV>(LM, LMinv, z, y);
  T zy = T(0);
  for (int i = 0; i < NV; ++i) zy += z[i] * y[i];
  const T loss = T(0.5) * zy + T(0.5) * P.eps * ff + qf + konst;
  if (!grad) return loss;
  // ---- envelope backward: Mbar = 1/2 (dv dv^T - y y^T) - lam a^T as outer products of the links' own twists ----
  T lam[NV], b[NV];
  for (int i = 0; i < NV; ++i) { b[i] = y[i] - dv[i]; lam[i] = P.dt * b[i]; }
  for (int bi = 0; bi < N; ++bi) {
    const T* R = K.R[bi];
    T tw[4][6];
    const T* src[4] = {dv, y, lam, acc};
    for (int k = 0; k < 4; ++k) {
      T V[6];
      chain_T<T, N>(K, bi, src[k], V);
      rot3t(R, V, tw[k]);
      for (int i = 0; i < 3; ++i) tw[k][3 + i] = V[3 + i];
    }
    T ab[6], bB[3];
    rot3t(R, bias + 6 * bi, bB);
    for (int i = 0; i < 3; ++i) { ab[i] = tw[3][i] + bB[i]; ab[3 + i] = tw[3][3 + i] + bias[6 * bi + 3 + i]; }
    const T* dvl = tw[0]; const T* yl = tw[1]; const T* lm = tw[2];
    T Kww[9], Nm[9], trvv = T(0);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        Kww[3 * i + j] = T(0.5) * (dvl[i] * dvl[j] - yl[i] * yl[j]) - lm[i] * ab[j];
        Nm[3 * i + j] = (dvl[i] * dvl[3 + j] - yl[i] * yl[3 + j]) - lm[i] * ab[3 + j] - lm[3 + j] * ab[i];
      }
    for (int i = 0; i < 3; ++i) trvv += T(0.5) * (dvl[3 + i] * dvl[3 + i] - yl[3 + i] * yl[3 + i]) - lm[3 + i] * ab[3 + i];
    T Vp[6], wB[3];
    chain_T<T, N>(K, bi, vp, Vp);
    rot3t(R, Vp, wB);
    rigid_body_inertia_adjoint<T>(P.body[bi].m, P.body[bi].c, R, wB, P.grav, Kww, Nm, trvv, lm, grad + 10 * bi);
  }
  for (int c = 0; c < NC; ++c) {
    const int bi = c >> 2, cl = c & 3;           // bi: box slot (mu, half lengths); li: its link (kinematics)
    if (!((S.con >> c) & 1u)) {
      if (grad_pts) for (int k = 0; k < 3; ++k) grad_pts[3 * c + k] = T(0);
      continue;
    }
    const int li = P.glink[bi];
    const T mu = P.mu[bi];
    const T* R = K.R[li];
    T eb[3], ev[3];
    chain_point_vel<T, N>(S, c, b, eb);
    chain_point_vel<T, N>(S, c, vp, ev);
    const T ftx = f[3 * c], fty = f[3 * c + 1], fn = f[3 * c + 2];
    const T sx = mu * ev[0], sy = mu * ev[1];
    const T sinv = t_rsqrt(t_max(sx * sx + sy * sy, t_tiny<T>()));
    const T ux = sx * sinv, uy = sy * sinv;
    const T gx = P.dt * (fn * ux + ftx), gy = P.dt * (fn * uy + fty);
    grad[10 * N + bi] += ftx * eb[0] + fty * eb[1] + gx * ev[0] + gy * ev[1];
    const T ft[3] = {mu * ftx, mu * fty, fn};
    const T gt[3] = {mu * gx, mu * gy, T(0)};
    T Vb[6], Vv[6], w1[3], w2[3], pw[3], pB[3];
    chain_T<T, N>(K, li, b, Vb);
    chain_T<T, N>(K, li, vp, Vv);
    cross3(ft, Vb, w1); cross3(gt, Vv, w2);           // angular parts of the link's twists (world)
    for (int i = 0; i < 3; ++i) pw[i] = w1[i] + w2[i];
    rot3t(R, pw, pB);
    const T phic = S.rho[3 * c + 2] + pos_z;
    const T phibar = (phic > T(0) ? fn : (phic < T(0) ? -fn : T(0))) - T(2) * t_max(-phic, T(0));
    // d loss / d (corner in the link frame), taken back into the box frame: d corner / d h_k = Rg[:, k] sgn_k
    T gl[3], gg[3];
    for (int k = 0; k < 3; ++k) gl[k] = pB[k] + phibar * R[6 + k];
    if (pts) {                                    // witness points: d loss / d (point in its link's frame) goes to the caller
      if (grad_pts) for (int k = 0; k < 3; ++k) grad_pts[3 * c + k] = gl[k];
      continue;
    }
    rot3t(P.Rg[bi], gl, gg);
    for (int k = 0; k < 3; ++k) grad[11 * N + 3 * bi + k] += sgn_bit<T>(K.sel[bi], cl, k) * gg[k];
  }
  return loss;
}

// learnable time step (forward_dynamics :260-304 + the Lie-group update): x (NQ + NV) -> xn
template <typename T, int N>
CN_HD int chain_step_sample(const ChainParams<T, N>& P, const SolverCfg<T>& cfg, const T* x, T* xn, const T* pts = nullptr,
                            unsigned npts = 0u) {
  constexpr int NV = 6 + N - 1, NC = 4 * N, NQ = 7 + N - 1;
  ChainKin<T, N> K;
  ChainProb<T, N> S;
  chain_kinematics<T, N>(P, x, K);
  T vW[NV], F[NV], LM[NV * NV], LMinv[NV], acc[NV], vm[NV];
  chain_to_world<T, N>(K.R[0], x + NQ, vW);
  chain_mass_force<T, N>(P, K, vW, LM, F, (T*)nullptr);
  for (int i = 0; i < NV * NV; ++i) S.M[i] = LM[i];
  chol_factor<T, NV>(LM, LMinv);
  chol_solve<T, NV>(LM, LMinv, F, acc);
  for (int i = 0; i < NV; ++i) vm[i] = vW[i] + P.dt * acc[i];
  chain_contacts<T, N>(P, K, S, pts, npts);
  const T inv_dt = T(1) / P.dt;
  for (int c = 0; c < NC; ++c) {
    const T mu = P.mu[c >> 2];
    T e[3];
    chain_point_vel<T, N>(S, c, vm, e);
    const bool on = (S.con >> c) & 1u;             // (a contact that does not exist: deep in the polar cone, as in the loss)
    S.q[3 * c] = on ? mu * e[0] : T(0);
    S.q[3 * c + 1] = on ? mu * e[1] : T(0);
    S.q[3 * c + 2] = on ? e[2] + (S.rho[3 * c + 2] + x[6]) * inv_dt : T(CH_OFF);
  }
  T u[NV];
  for (int i = 0; i < NV; ++i) u[i] = T(0);
  const int it = chain_solve<T, N>(P, S, cfg, u);
  T vnW[NV], vn[NV];
  for (int i = 0; i < NV; ++i) vnW[i] = vm[i] + u[i];
  rot3t(K.R[0], vnW, vn);
  for (int i = 3; i < NV; ++i) vn[i] = vnW[i];
  const T rx = vn[0] * P.dt, ry = vn[1] * P.dt, rz = vn[2] * P.dt;
  const T ang = t_sqrt(rx * rx + ry * ry + rz * rz);
  const T half = T(0.5) * ang;
  using std::cos;
  using std::sin;
  const T sinc = half > T(0) ? sin(half) / half : T(1);
  const T dw = cos(half), k = T(0.5) * sinc;
  const T dx = rx * k, dy = ry * k, dz = rz * k;
  const T qw = x[0], qx = x[1], qy = x[2], qz = x[3];
  xn[0] = qw * dw - (qx * dx + qy * dy + qz * dz);
  xn[1] = qw * dx + dw * qx + (qy * dz - qz * dy);
  xn[2] = qw * dy + dw * qy + (qz * dx - qx * dz);
  xn[3] = qw * dz + dw * qz + (qx * dy - qy * dx);
  for (int i = 0; i < 3; ++i) xn[4 + i] = x[4 + i] + vn[3 + i] * P.dt;
  for (int j = 1; j < N; ++j) xn[6 + j] = x[6 + j] + vn[5 + j] * P.dt;
  for (int i = 0; i < NV; ++i) xn[NQ + i] = vn[i];
  return it;
}

// ---------------------------------------------------------------------------
// Dense dynamics terms of a tree in the reference's own coordinates and ordering, for callers of MultibodyTerms.forward
// (multibody_terms.py:584-609): M (NV x NV), J (3 nc x NV) = [J_n (nc rows) ; mu J_t (x, y interleaved per contact,
// 2 nc rows)] (:401-426), phi (nc), contact-free acceleration (NV), Delassus operator D = J M^-1 J^T (3 nc x 3 nc, nullable),
// nc = 4 n_boxes: the contacts of the first n_boxes box slots (the system's boxes in their order), each box by ascending
// vertex index.  State velocity v = [w_body0 ; v_world ; joint rates] = T^T u^ with T = blkdiag(R_0, I3, I) (orthogonal), so
// M = T^T M^ T, J = J^ T, a = T^T a^  (as elbow_terms_sample does for the two-body system).
// ---------------------------------------------------------------------------
template <typename T, int N>
CN_HD void chain_terms_sample(const ChainParams<T, N>& P, const T* q, const T* v, int n_boxes, T* M, T* J, T* phi, T* acc, T* D) {
  constexpr int NV = 6 + N - 1, NC = 4 * N;
  const int nc = 4 * n_boxes, kk = 3 * nc;
  ChainKin<T, N> K;
  ChainProb<T, N> S;
  chain_kinematics<T, N>(P, q, K);
  T vW[NV], F[NV], MW[NV * NV], LM[NV * NV], LMinv[NV], aW[NV];
  chain_to_world<T, N>(K.R[0], v, vW);
  chain_mass_force<T, N>(P, K, vW, MW, F, (T*)nullptr);
  for (int i = 0; i < NV * NV; ++i) LM[i] = MW[i];
  chol_factor<T, NV>(LM, LMinv);
  chol_solve<T, NV>(LM, LMinv, F, aW);
  const T* R = K.R[0];
  rot3t(R, aW, acc);
  for (int i = 3; i < NV; ++i) acc[i] = aW[i];
  T tmp[NV * NV];
  for (int i = 0; i < NV; ++i) {                      // tmp = M^ T  (columns 0..2 rotated)
    const T* row = MW + NV * i;
    for (int j = 0; j < 3; ++j) tmp[NV * i + j] = row[0] * R[j] + row[1] * R[3 + j] + row[2] * R[6 + j];
    for (int j = 3; j < NV; ++j) tmp[NV * i + j] = row[j];
  }
  for (int j = 0; j < NV; ++j) {                      // M = T^T tmp  (rows 0..2 rotated)
    for (int i = 0; i < 3; ++i) M[NV * i + j] = R[i] * tmp[j] + R[3 + i] * tmp[NV + j] + R[6 + i] * tmp[2 * NV + j];
    for (int i = 3; i < NV; ++i) M[NV * i + j] = tmp[NV * i + j];
  }
  chain_contacts<T, N>(P, K, S);
  for (int c = 0; c < nc && c < NC; ++c) {
    const T mu = P.mu[c >> 2];
    const T rho[3] = {S.rho[3 * c], S.rho[3 * c + 1], S.rho[3 * c + 2]};
    phi[c] = rho[2] + q[6];
    T E[9];                                            // (-S(rho)) R_0: the angular block in state coordinates
    for (int j = 0; j < 3; ++j) {
      const T col[3] = {R[j], R[3 + j], R[6 + j]};
      T cr[3];
      cross3(rho, col, cr);
      for (int i = 0; i < 3; ++i) E[3 * i + j] = -cr[i];
    }
    T* jn = J + NV * c;
    T* jx = J + NV * (nc + 2 * c);
    T* jy = J + NV * (nc + 2 * c + 1);
    for (int j = 0; j < 3; ++j) {
      jn[j] = E[6 + j]; jx[j] = mu * E[j]; jy[j] = mu * E[3 + j];
      jn[3 + j] = j == 2 ? T(1) : T(0);
      jx[3 + j] = j == 0 ? mu : T(0);
      jy[3 + j] = j == 1 ? mu : T(0);
    }
    for (int j = 1; j < N; ++j) {
      const T* hcol = S.hc + 3 * (c * (N - 1) + (j - 1));
      jn[5 + j] = hcol[2]; jx[5 + j] = mu * hcol[0]; jy[5 + j] = mu * hcol[1];
    }
  }
  if (D) {
    // D = J M^-1 J^T with M = L L^T (Cholesky of the state-coordinate M): D_ab = W_a . W_b with W_r = L^-1 J_r^T.  The
    // W_r are recomputed per pair instead of being kept (3 nc x NV doubles per thread): this is an export, not a hot loop.
    T LS[NV * NV], LSinv[NV];
    for (int i = 0; i < NV * NV; ++i) LS[i] = M[i];
    chol_factor<T, NV>(LS, LSinv);
    for (int a = 0; a < kk; ++a) {
      T Wa[NV];
      for (int i = 0; i < NV; ++i) {
        T sa = J[NV * a + i];
        for (int m = 0; m < i; ++m) sa -= LS[NV * i + m] * Wa[m];
        Wa[i] = sa * LSinv[i];
      }
      for (int b = 0; b <= a; ++b) {
        T Wb[NV];
        for (int i = 0; i < NV; ++i) {
          T sb = J[NV * b + i];
          for (int m = 0; m < i; ++m) sb -= LS[NV * i + m] * Wb[m];
          Wb[i] = sb * LSinv[i];
        }
        T sdot = T(0);
        for (int k = 0; k < NV; ++k) sdot += Wa[k] * Wb[k];
        D[kk * a + b] = sdot;
        D[kk * b + a] = sdot;
      }
    }
  }
}

}  // namespace cn
