// Tile-cooperative 3-D rigid-body step for free-base tree robots (cassie3d_stiff.xml; BASELINE.json configs[3]).
//
// Restates mj_step for the reference's 3-D model (model/cassie3d_stiff.xml:5: dt 5e-4, PGS, 50 iterations, elliptic
// cones, Euler with implicit joint damping) -- the same pipeline the planar engine restates for cassie2d_stiff.xml
// (Cassie2d.cpp:62,81,92) -- for a general kinematic tree: free joint with quaternion integration, 3-D hinges, 3-row
// connects, joint limits, condim-3 elliptic contacts (plane-sphere, plane-capsule, capsule-capsule).
//
// Mapping (north_star: "each env maps to one warp or sub-warp using shuffle reductions"): one env per TILE of LANES
// lanes (8, 16 or 32), all per-env scratch in shared memory, every loop strided over the lanes of the tile, reductions by
// xor shuffles inside the tile.  Control flow is uniform per tile, tiles of one warp may diverge.  With LANES = 1 the
// same code is plain serial C++: tests/host_harness/tree_harness.cpp runs it on the CPU against the oracle.
//
// Formulation (deliberately not the oracle's): spatial vectors [angular; linear] in world axes about the BASE position
// (so fp32 never sees the distance walked), composite-rigid-body mass matrix, recursive Newton-Euler bias with the
// children pulled level by level, dense Cholesky M = L L^T, one forward substitution per constraint row
// (Y = L^-1 J^T in place of J, A = Y^T Y + R packed in shared memory, qacc and J^T f recovered from Y f), and a "publish" Gauss-Seidel sweep: every row owns its residual, a new force is broadcast and folded into all
// residuals with one FMA per row.
#pragma once
#include <math.h>
#include "tree_model.h"

#if defined(__CUDACC__)
#define TREE_UNROLL4 _Pragma("unroll 4")
#define TREE_FN __device__ __forceinline__
#define TREE_HD __host__ __device__ __forceinline__
#else
#define TREE_UNROLL4
#define TREE_FN inline
#define TREE_HD inline
#endif

namespace cassie {
namespace tree {

constexpr int kLD = kMaxDof + 1;       // row stride of [row][dof] arrays: odd, so lanes walking rows hit distinct banks
TREE_HD int tri(int r, int c) { return r >= c ? r * (r + 1) / 2 + c : c * (c + 1) / 2 + r; }

// ---------------------------------------------------------------------------------------------- tile runtime
template <int LANES>
struct Tile {
#if defined(__CUDACC__)
  int lane;
  unsigned mask;
  __device__ __forceinline__ static Tile make() {
    Tile t;
    const unsigned l = threadIdx.x & 31u;
    t.lane = (int)(l & (unsigned)(LANES - 1));
    t.mask = LANES == 32 ? 0xffffffffu : (((1u << (LANES & 31)) - 1u) << (l & ~(unsigned)(LANES - 1)));
    return t;
  }
  __device__ __forceinline__ void sync() const { __syncwarp(mask); }
  template <typename V> __device__ __forceinline__ V sum(V v) const {
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, LANES);
    return v;
  }
#else
  int lane;
  static Tile make() { Tile t; t.lane = 0; return t; }
  void sync() const {}
  template <typename V> V sum(V v) const { return v; }
#endif
};

// ---------------------------------------------------------------------------------------------- per-env scratch
// ROWS / CON: constraint-row and contact capacity of this instantiation (njmax / nconmax).  The kernels run a small
// capacity first (kFastRows rows: one register slot per lane, 11.5 KB per env) and hand the rare env that needs more to the
// full-capacity instantiation (tree_kernels.cuh), so capacity never changes a result.
template <typename T, int ROWS = kMaxRows, int CON = kMaxCon>
struct Scratch {
  static constexpr int kRows = ROWS, kCon = CON, kPackedA = ROWS * (ROWS + 1) / 2;
  // state (q: base position, quaternion w x y z, hinge angles)
  T q[kMaxDof + 1], qd[kMaxDof], warm[kMaxDof], ctrl[kMaxAct];
  // kinematics about the base position, world axes
  T xpos[kMaxLinks][3], xmat[kMaxLinks][9];
  T S[kMaxDof][6];
  // link velocities, velocity-product accelerations and RNE forces are dead once the bias is formed; the per-row vectors
  // of the constraint solve are born later: they share storage
  union {
    struct { T V[kMaxLinks][6], A[kMaxLinks][6], F[kMaxLinks][6]; };
    struct { T r_pos[ROWS], r_R[ROWS], r_aref[ROWS], r_b[ROWS], r_f[ROWS]; };
  };
  T r_acc[ROWS];
  T Ic[kMaxLinks][10];                 // mass, h = m c (3), inertia about the origin xx yy zz xy xz yz
  T gw[kMaxGeoms][6];                  // geom points in the world frame (relative to the base)
  // ONE square array for the mass matrix and its factor: strict upper triangle = M (symmetric), lower triangle incl. the
  // diagonal = L of the current Cholesky factorisation, Mdiag = diagonal of M
  T L[kMaxDof * kLD], Mdiag[kMaxDof], dinv[kMaxDof];
  T qfrc[kMaxDof], qacc_s[kMaxDof], qacc[kMaxDof], qfc[kMaxDof], tmp[kMaxDof], wk[kMaxDof];
  // contacts
  int ncon, nefc, n_dropped, sweeps, overflow;   // overflow: this step needed more rows / contacts than ROWS / CON
  unsigned char slot_on[2 * kMaxPairs];
  int c_pair[CON], c_end[CON], c_dim[CON];
  T c_dist[CON], c_pos[CON][3], c_frame[CON][9];
  // constraint rows
  signed char r_type[ROWS], r_sub[ROWS];
  short r_id[ROWS];
  T J[ROWS * kLD];                 // constraint Jacobian, overwritten by Y = L^-1 J^T (row r = y_r^T) before the solve
  T Am[kPackedA];
  static_assert(5 * ROWS <= 3 * kMaxLinks * 6, "the row vectors must fit in the storage of V, A, F");
  static_assert(ROWS <= 64, "row kinds are kept in 64-bit masks");
};
constexpr int kFastRows = 32, kFastCon = 9;   // the common-case capacity (6 connect rows + 8 condim-3 contacts + 2 limits)

enum RowType { kRowEq = 0, kRowLimit = 1, kRowContact = 2 };
constexpr double kMinVal = 1e-15;

// ---------------------------------------------------------------------------------------------- small algebra
template <typename T> TREE_HD void cross3(T* r, const T* a, const T* b) {
  const T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename T> TREE_HD T dot3(const T* a, const T* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename T> TREE_HD void mulv(T* r, const T* M, const T* v) {
  const T x = M[0] * v[0] + M[1] * v[1] + M[2] * v[2], y = M[3] * v[0] + M[4] * v[1] + M[5] * v[2], z = M[6] * v[0] + M[7] * v[1] + M[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename T> TREE_HD void mulm(T* R, const T* A, const T* B) {
  T t[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) t[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
  for (int i = 0; i < 9; i++) R[i] = t[i];
}
template <typename T> TREE_HD T dot6(const T* a, const T* b) {
  return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
}
// spatial inertia (m, h, I about the origin) times a motion vector [w; v] -> force [n; f]
template <typename T> TREE_HD void inertia_mul(T* r, const T* I, const T* mv) {
  const T* h = I + 1;
  const T* w = mv;
  const T* v = mv + 3;
  T hv[3], hw[3];
  cross3(hv, h, v);
  cross3(hw, h, w);
  r[0] = I[4] * w[0] + I[7] * w[1] + I[8] * w[2] + hv[0];
  r[1] = I[7] * w[0] + I[5] * w[1] + I[9] * w[2] + hv[1];
  r[2] = I[8] * w[0] + I[9] * w[1] + I[6] * w[2] + hv[2];
  r[3] = I[0] * v[0] - hw[0];
  r[4] = I[0] * v[1] - hw[1];
  r[5] = I[0] * v[2] - hw[2];
}
// motion cross product v x s and force cross product v x* f
template <typename T> TREE_HD void crm(T* r, const T* v, const T* s) {
  T a[3], b[3], c[3];
  cross3(a, v, s);
  cross3(b, v, s + 3);
  cross3(c, v + 3, s);
  r[0] = a[0]; r[1] = a[1]; r[2] = a[2];
  r[3] = b[0] + c[0]; r[4] = b[1] + c[1]; r[5] = b[2] + c[2];
}
template <typename T> TREE_HD void crf(T* r, const T* v, const T* f) {
  T a[3], b[3], c[3];
  cross3(a, v, f);
  cross3(b, v + 3, f + 3);
  cross3(c, v, f + 3);
  r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2];
  r[3] = c[0]; r[4] = c[1]; r[5] = c[2];
}
// mju_makeFrame: f[0..2] = normal (made unit), f[3..5] = optional y hint
template <typename T> TREE_HD void make_frame(T* f) {
  T* x = f; T* y = f + 3; T* z = f + 6;
  T n = (T)1 / sqrt(dot3(x, x));
  for (int i = 0; i < 3; i++) x[i] *= n;
  if (sqrt(dot3(y, y)) < (T)0.5) {
    y[0] = y[1] = y[2] = 0;
    if (x[1] < (T)0.5 && x[1] > (T)-0.5) y[1] = 1; else y[2] = 1;
  }
  const T t = dot3(x, y);
  for (int i = 0; i < 3; i++) y[i] -= t * x[i];
  n = (T)1 / sqrt(dot3(y, y));
  for (int i = 0; i < 3; i++) y[i] *= n;
  cross3(z, x, y);
}
// getimpedance (5-parameter solimp)
template <typename T> TREE_HD T impedance(const T* si, T pos, T margin) {
  if (si[0] == si[1] || si[2] <= (T)kMinVal) return (T)0.5 * (si[0] + si[1]);
  T x = (pos - margin) / si[2];
  if (x < 0) x = -x;
  if (x >= 1) return si[1];
  if (x <= 0) return si[0];
  T y;
  if (si[4] == (T)1) y = x;
  else if (x <= si[3]) y = pow(x, si[4]) / pow(si[3], si[4] - 1);
  else y = 1 - pow(1 - x, si[4]) / pow(1 - si[3], si[4] - 1);
  return si[0] + y * (si[1] - si[0]);
}
// point Jacobian column of dof d for a world point P on a link moved by d
template <typename T> TREE_HD void jac_col(T* r, const T* S, const T* P) {
  T t[3];
  cross3(t, S, P);
  r[0] = S[3] + t[0]; r[1] = S[4] + t[1]; r[2] = S[5] + t[2];
}

// ---------------------------------------------------------------------------------------------- kinematics + dynamics
// One link's frame (orientation, position about the base position): the frame part of link_pass below, the same
// arithmetic, for the env's frame pass (tree_env.cuh).  A hinge link also returns its joint's anchor `an` and axis `ax`
// in world axes.  Needs the parent's frame.
template <typename T, typename SC>
TREE_FN void link_frame(const TreeModel<T>& m, SC& s, int l, T* an, T* ax) {
  T* pos = s.xpos[l];
  T* mat = s.xmat[l];
  if (l == 0) {
    T w = s.q[3], x = s.q[4], y = s.q[5], z = s.q[6];
    const T nq = (T)1 / sqrt(w * w + x * x + y * y + z * z);   // mj_normalizeQuat
    w *= nq; x *= nq; y *= nq; z *= nq;
    mat[0] = 1 - 2 * (y * y + z * z); mat[1] = 2 * (x * y - w * z); mat[2] = 2 * (x * z + w * y);
    mat[3] = 2 * (x * y + w * z); mat[4] = 1 - 2 * (x * x + z * z); mat[5] = 2 * (y * z - w * x);
    mat[6] = 2 * (x * z - w * y); mat[7] = 2 * (y * z + w * x); mat[8] = 1 - 2 * (x * x + y * y);
    pos[0] = pos[1] = pos[2] = 0;
  } else {
    const int p = m.parent[l];
    T R0[9], t[3];
    mulm(R0, s.xmat[p], m.lmat[l]);
    mulv(t, s.xmat[p], m.lpos[l]);
    mulv(an, R0, m.jpos[l]);
    for (int i = 0; i < 3; i++) an[i] += s.xpos[p][i] + t[i];
    mulv(ax, R0, m.axis[l]);
    // rotation about the hinge axis, in the link frame (Rodrigues)
    const T th = s.q[6 + l] - m.ref[l];
    const T sn = sin(th), cs = cos(th), vc = 1 - cs;
    const T* a = m.axis[l];
    T Rl[9] = {cs + a[0] * a[0] * vc, a[0] * a[1] * vc - a[2] * sn, a[0] * a[2] * vc + a[1] * sn,
               a[1] * a[0] * vc + a[2] * sn, cs + a[1] * a[1] * vc, a[1] * a[2] * vc - a[0] * sn,
               a[2] * a[0] * vc - a[1] * sn, a[2] * a[1] * vc + a[0] * sn, cs + a[2] * a[2] * vc};
    mulm(mat, R0, Rl);
    mulv(t, mat, m.jpos[l]);
    for (int i = 0; i < 3; i++) pos[i] = an[i] - t[i];
  }
}

// One link: frame, motion subspace, velocity, velocity-product acceleration, own spatial inertia and RNE force.
template <typename T, typename SC>
TREE_FN void link_pass(const TreeModel<T>& m, SC& s, int l) {
  T* pos = s.xpos[l];
  T* mat = s.xmat[l];
  T Vl[6], Al[6];
  if (l == 0) {
    T w = s.q[3], x = s.q[4], y = s.q[5], z = s.q[6];
    const T nq = (T)1 / sqrt(w * w + x * x + y * y + z * z);   // mj_normalizeQuat
    w *= nq; x *= nq; y *= nq; z *= nq;
    mat[0] = 1 - 2 * (y * y + z * z); mat[1] = 2 * (x * y - w * z); mat[2] = 2 * (x * z + w * y);
    mat[3] = 2 * (x * y + w * z); mat[4] = 1 - 2 * (x * x + z * z); mat[5] = 2 * (y * z - w * x);
    mat[6] = 2 * (x * z - w * y); mat[7] = 2 * (y * z + w * x); mat[8] = 1 - 2 * (x * x + y * y);
    pos[0] = pos[1] = pos[2] = 0;
    for (int k = 0; k < 3; k++) {
      T* St = s.S[k];
      T* Sr = s.S[3 + k];
      for (int i = 0; i < 6; i++) { St[i] = 0; Sr[i] = 0; }
      St[3 + k] = 1;
      Sr[0] = mat[k]; Sr[1] = mat[3 + k]; Sr[2] = mat[6 + k];
    }
    T ww[3];
    mulv(ww, mat, s.qd + 3);                       // angular velocity in world axes
    Vl[0] = ww[0]; Vl[1] = ww[1]; Vl[2] = ww[2]; Vl[3] = s.qd[0]; Vl[4] = s.qd[1]; Vl[5] = s.qd[2];
    Al[0] = Al[1] = Al[2] = 0;
    cross3(Al + 3, s.qd, ww);                      // the three rotational cdof_dot use the velocity before them (mj_comVel)
  } else {
    const int p = m.parent[l], d = 5 + l;
    T R0[9], t[3], an[3], ax[3];
    mulm(R0, s.xmat[p], m.lmat[l]);
    mulv(t, s.xmat[p], m.lpos[l]);
    mulv(an, R0, m.jpos[l]);
    for (int i = 0; i < 3; i++) an[i] += s.xpos[p][i] + t[i];
    mulv(ax, R0, m.axis[l]);
    // rotation about the hinge axis, in the link frame (Rodrigues)
    const T th = s.q[6 + l] - m.ref[l];
    const T sn = sin(th), cs = cos(th), vc = 1 - cs;
    const T* a = m.axis[l];
    T Rl[9] = {cs + a[0] * a[0] * vc, a[0] * a[1] * vc - a[2] * sn, a[0] * a[2] * vc + a[1] * sn,
               a[1] * a[0] * vc + a[2] * sn, cs + a[1] * a[1] * vc, a[1] * a[2] * vc - a[0] * sn,
               a[2] * a[0] * vc - a[1] * sn, a[2] * a[1] * vc + a[0] * sn, cs + a[2] * a[2] * vc};
    mulm(mat, R0, Rl);
    mulv(t, mat, m.jpos[l]);
    for (int i = 0; i < 3; i++) pos[i] = an[i] - t[i];
    T* S = s.S[d];
    S[0] = ax[0]; S[1] = ax[1]; S[2] = ax[2];
    cross3(S + 3, an, ax);
    T Sd[6];
    crm(Sd, s.V[p], S);
    const T qd = s.qd[d];
    for (int i = 0; i < 6; i++) { Vl[i] = s.V[p][i] + S[i] * qd; Al[i] = s.A[p][i] + Sd[i] * qd; }
  }
  for (int i = 0; i < 6; i++) { s.V[l][i] = Vl[i]; s.A[l][i] = Al[i]; }
  // own spatial inertia about the origin
  T c[3], RI[9], Iw[9];
  mulv(c, mat, m.com[l]);
  for (int i = 0; i < 3; i++) c[i] += pos[i];
  const T* I6 = m.inertia[l];
  const T If[9] = {I6[0], I6[3], I6[4], I6[3], I6[1], I6[5], I6[4], I6[5], I6[2]};
  mulm(RI, mat, If);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) Iw[3 * i + j] = RI[3 * i] * mat[3 * j] + RI[3 * i + 1] * mat[3 * j + 1] + RI[3 * i + 2] * mat[3 * j + 2];
  const T ms = m.mass[l], c2 = dot3(c, c);
  T* I = s.Ic[l];
  I[0] = ms; I[1] = ms * c[0]; I[2] = ms * c[1]; I[3] = ms * c[2];
  I[4] = Iw[0] + ms * (c2 - c[0] * c[0]); I[5] = Iw[4] + ms * (c2 - c[1] * c[1]); I[6] = Iw[8] + ms * (c2 - c[2] * c[2]);
  I[7] = Iw[1] - ms * c[0] * c[1]; I[8] = Iw[2] - ms * c[0] * c[2]; I[9] = Iw[5] - ms * c[1] * c[2];
  // RNE force with gravity as a base acceleration -g: F = I (A - [0; g]) + V x* (I V)
  T Ag[6] = {Al[0], Al[1], Al[2], Al[3] - m.gravity[0], Al[4] - m.gravity[1], Al[5] - m.gravity[2]};
  T IA[6], IV[6], VIV[6];
  inertia_mul(IA, I, Ag);
  inertia_mul(IV, I, Vl);
  crf(VIV, Vl, IV);
  for (int i = 0; i < 6; i++) s.F[l][i] = IA[i] + VIV[i];
}

// mj_kinematics + mj_comVel + mj_crb + mj_rne: frames, M (with armature), bias in s.tmp
template <int LANES, typename T, typename SC>
TREE_FN void dynamics(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s) {
  for (int lev = 0; lev < m.nlevels; lev++) {
    for (int i = m.level_off[lev] + tl.lane; i < m.level_off[lev + 1]; i += LANES) link_pass(m, s, i);
    tl.sync();
  }
  // composite inertias and subtree forces: every link pulls its (finished) children, deepest level first
  for (int lev = m.nlevels - 2; lev >= 0; lev--) {
    for (int l = m.level_off[lev] + tl.lane; l < m.level_off[lev + 1]; l += LANES)
      for (int k = m.child_off[l]; k < m.child_off[l + 1]; k++) {
        const int c = m.child[k];
        for (int i = 0; i < 10; i++) s.Ic[l][i] += s.Ic[c][i];
        for (int i = 0; i < 6; i++) s.F[l][i] += s.F[c][i];
      }
    tl.sync();
  }
  const int nv = m.nv;
  for (int d = tl.lane; d < nv; d += LANES) {
    const int l = d < 6 ? 0 : d - 5;
    T f6[6];
    inertia_mul(f6, s.Ic[l], s.S[d]);
    const unsigned anc = m.anc[l];
    for (int a = 0; a < d; a++) {
      const T v = ((anc >> a) & 1u) ? dot6(s.S[a], f6) : (T)0;
      s.L[a * kLD + d] = v;                      // M lives in the strict upper triangle (a < d)
    }
    s.Mdiag[d] = dot6(s.S[d], f6) + m.armature[d];
    s.tmp[d] = dot6(s.S[d], s.F[l]);
  }
  tl.sync();
}

// dense Cholesky of (M + diag(add)) into s.L (lower triangle) and s.dinv = 1 / L_kk.  Left-looking, rows owned by fixed
// lanes, ONE tile barrier per column: the running diagonal wk[i] = M_ii - sum_{j<k} L_ij^2 is kept by the owner of row i,
// so the pivot of column k is one shared-memory read; L[i][k] = (M[i][k] - sum_j L[i][j] L[k][j]) / L[k][k].
template <int LANES, typename T, typename SC>
TREE_FN void cholesky(const Tile<LANES>& tl, int n, SC& s, const T* add, T scale) {
  for (int i = tl.lane; i < n; i += LANES) s.wk[i] = s.Mdiag[i] + (add ? scale * add[i] : (T)0);
  tl.sync();
  for (int k = 0; k < n; k++) {
    const T d = s.wk[k];
    const T inv = (T)1 / sqrt(d);
    if (tl.lane == 0) { s.dinv[k] = inv; s.L[k * kLD + k] = d * inv; }   // L_kk = sqrt(d): read by J^T f = L z only
    for (int i = tl.lane; i < n; i += LANES) {
      if (i <= k) continue;
      T v = s.L[k * kLD + i];                      // M[i][k] = M[k][i], upper triangle
      TREE_UNROLL4
      for (int j = 0; j < k; j++) v -= s.L[i * kLD + j] * s.L[k * kLD + j];
      v *= inv;
      s.L[i * kLD + k] = v;
      s.wk[i] -= v * v;
    }
    tl.sync();
  }
}

// x <- L^-T x for one vector in shared memory, cooperative: the finished entries go to `out` (a different array), so a
// column needs ONE barrier
template <int LANES, typename T, typename SC>
TREE_FN void backward_one(const Tile<LANES>& tl, int n, const SC& s, T* x, T* out) {
  for (int k = n - 1; k >= 0; k--) {
    const T xk = x[k] * s.dinv[k];
    if (tl.lane == 0) out[k] = xk;
    for (int j = tl.lane; j < k; j += LANES) x[j] -= s.L[k * kLD + j] * xk;
    tl.sync();
  }
}

// x <- (L L^T)^-1 x for one vector in shared memory, cooperative (column sweeps, one FMA per lane and step); s.wk is scratch
template <int LANES, typename T, typename SC>
TREE_FN void solve_one(const Tile<LANES>& tl, int n, SC& s, T* x) {
  for (int k = 0; k < n; k++) {
    const T xk = x[k] * s.dinv[k];
    if (tl.lane == 0) s.wk[k] = xk;
    for (int i = k + 1 + tl.lane; i < n; i += LANES) x[i] -= s.L[i * kLD + k] * xk;
    tl.sync();
  }
  backward_one(tl, n, s, s.wk, x);
}

// one lane, one right-hand side: x <- L^-1 x (forward substitution, serial)
template <typename T, typename SC>
TREE_FN void forward_row(int n, const SC& s, T* x) {
  for (int i = 0; i < n; i++) {
    T v = x[i];
    TREE_UNROLL4
    for (int j = 0; j < i; j++) v -= s.L[i * kLD + j] * x[j];
    x[i] = v * s.dinv[i];
  }
}

// ---------------------------------------------------------------------------------------------- collision
// signed distance of the sphere of radius r at c to the world plane (base-relative coordinates)
template <typename T, typename SC>
TREE_FN T plane_dist(const TreeModel<T>& m, const SC& s, const T* c, T r) {
  T d[3] = {c[0] - (m.plane_pos[0] - s.q[0]), c[1] - (m.plane_pos[1] - s.q[1]), c[2] - (m.plane_pos[2] - s.q[2])};
  return dot3(d, m.plane_n) - r;
}
// closest points of two segments (a0,a1), (b0,b1); returns the distance
template <typename T>
TREE_FN T seg_seg(const T* a0, const T* a1, const T* b0, const T* b1, T* pa, T* pb) {
  T d1[3], d2[3], r[3];
  for (int i = 0; i < 3; i++) { d1[i] = a1[i] - a0[i]; d2[i] = b1[i] - b0[i]; r[i] = a0[i] - b0[i]; }
  const T a = dot3(d1, d1), e = dot3(d2, d2), f = dot3(d2, r), c = dot3(d1, r), b = dot3(d1, d2), den = a * e - b * b;
  T sp = den > (T)1e-14 ? (b * f - c * e) / den : (T)0;
  sp = sp < 0 ? (T)0 : (sp > 1 ? (T)1 : sp);
  T tp = (b * sp + f) / e;
  if (tp < 0) { tp = 0; sp = -c / a; sp = sp < 0 ? (T)0 : (sp > 1 ? (T)1 : sp); }
  else if (tp > 1) { tp = 1; sp = (b - c) / a; sp = sp < 0 ? (T)0 : (sp > 1 ? (T)1 : sp); }
  T dd[3];
  for (int i = 0; i < 3; i++) { pa[i] = a0[i] + sp * d1[i]; pb[i] = b0[i] + tp * d2[i]; dd[i] = pa[i] - pb[i]; }
  return sqrt(dot3(dd, dd));
}

// mj_collision: geoms to the world frame, narrow phase per pair in MuJoCo's pair order, contacts compacted in that order
template <int LANES, typename T, typename SC>
TREE_FN void collide(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s) {
  for (int g = tl.lane; g < m.ng; g += LANES) {
    const int l = m.g_link[g];
    T t[3];
    mulv(t, s.xmat[l], m.g_p0[g]);
    for (int i = 0; i < 3; i++) s.gw[g][i] = s.xpos[l][i] + t[i];
    mulv(t, s.xmat[l], m.g_p1[g]);
    for (int i = 0; i < 3; i++) s.gw[g][3 + i] = s.xpos[l][i] + t[i];
  }
  tl.sync();
  for (int p = tl.lane; p < m.npair; p += LANES) {
    const int a = m.pair_a[p], b = m.pair_b[p];
    int on0 = 0, on1 = 0;
    if (a < 0) {
      on0 = plane_dist(m, s, s.gw[b], m.g_radius[b]) <= 0;
      if (m.g_type[b] == kCapsule) on1 = plane_dist(m, s, s.gw[b] + 3, m.g_radius[b]) <= 0;
    } else {
      T pa[3], pb[3];
      // segments run from the 'from' end (p1) to the 'to' end (p0), like the oracle's
      const T cd = seg_seg(s.gw[a] + 3, s.gw[a], s.gw[b] + 3, s.gw[b], pa, pb);
      on0 = (cd - m.g_radius[a] - m.g_radius[b] <= 0) && cd >= (T)1e-12;
    }
    s.slot_on[2 * p] = on0;
    s.slot_on[2 * p + 1] = on1;
  }
  tl.sync();
  // ordered compaction (every lane runs the same scan; lane 0 writes)
  int n = 0, dropped = 0, rows = 3 * m.neq;
  for (int sl = 0; sl < 2 * m.npair; sl++) {
    if (!s.slot_on[sl]) continue;
    const int dim = m.pair_condim[sl >> 1];
    if (n < SC::kCon && rows + dim <= SC::kRows) {
      if (tl.lane == 0) { s.c_pair[n] = sl >> 1; s.c_end[n] = sl & 1; s.c_dim[n] = dim; }
      n++;
      rows += dim;
    } else
      dropped++;
  }
  if (tl.lane == 0) { s.ncon = n; s.n_dropped = dropped; s.overflow = dropped > 0; }
  tl.sync();
  for (int c = tl.lane; c < n; c += LANES) {
    const int p = s.c_pair[c], a = m.pair_a[p], b = m.pair_b[p];
    T* fr = s.c_frame[c];
    if (a < 0) {
      const T* ctr = s.gw[b] + 3 * s.c_end[c];
      const T r = m.g_radius[b], dist = plane_dist(m, s, ctr, r);
      s.c_dist[c] = dist;
      for (int i = 0; i < 3; i++) {
        s.c_pos[c][i] = ctr[i] - m.plane_n[i] * (r + (T)0.5 * dist);
        fr[i] = m.plane_n[i];
        fr[3 + i] = 0;
      }
      if (m.g_type[b] == kCapsule) {
        // frame y hint = capsule axis ('from' -> 'to'), mjc_PlaneCapsule
        T ax[3] = {s.gw[b][0] - s.gw[b][3], s.gw[b][1] - s.gw[b][4], s.gw[b][2] - s.gw[b][5]};
        const T n1 = (T)1 / sqrt(dot3(ax, ax));
        for (int i = 0; i < 3; i++) fr[3 + i] = ax[i] * n1;
      }
    } else {
      T pa[3], pb[3];
      const T cd = seg_seg(s.gw[a] + 3, s.gw[a], s.gw[b] + 3, s.gw[b], pa, pb);
      const T gap = cd - m.g_radius[a] - m.g_radius[b];
      s.c_dist[c] = gap;
      for (int i = 0; i < 3; i++) {
        const T nrm = (pb[i] - pa[i]) / cd;
        fr[i] = nrm;
        fr[3 + i] = 0;
        s.c_pos[c][i] = pa[i] + nrm * (m.g_radius[a] + (T)0.5 * gap);
      }
    }
    make_frame(fr);
  }
  tl.sync();
}

// ---------------------------------------------------------------------------------------------- constraints
// mj_makeConstraint + mj_makeImpedance: row table (connects, joint limits, contacts), Jacobians, R, aref
template <int LANES, typename T, typename SC>
TREE_FN void make_rows(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s) {
  if (tl.lane == 0) {
    int n = 0, crows = 0;
    for (int c = 0; c < s.ncon; c++) crows += s.c_dim[c];
    for (int e = 0; e < m.neq; e++)
      for (int k = 0; k < 3; k++) { s.r_type[n] = kRowEq; s.r_id[n] = e; s.r_sub[n] = k; n++; }
    for (int ud = 6; ud < m.nv; ud++) {       // MuJoCo's joint order: it fixes the Gauss-Seidel order of the limit rows
      const int d = m.dof_of_user[ud];
      if (!m.limited[d]) continue;
      const T qv = s.q[d + 1];
      // lower side first (mj_instantiateLimit); the rows left after the contacts' reservation bound the count
      if (qv - m.range[d][0] < 0) { if (n + crows < SC::kRows) { s.r_type[n] = kRowLimit; s.r_id[n] = d; s.r_sub[n] = 0; n++; } else s.overflow = 1; }
      if (m.range[d][1] - qv < 0) { if (n + crows < SC::kRows) { s.r_type[n] = kRowLimit; s.r_id[n] = d; s.r_sub[n] = 1; n++; } else s.overflow = 1; }
    }
    for (int c = 0; c < s.ncon; c++)
      for (int k = 0; k < s.c_dim[c]; k++) { s.r_type[n] = kRowContact; s.r_id[n] = c; s.r_sub[n] = k; n++; }
    s.nefc = n;
  }
  tl.sync();
  const int nv = m.nv, nefc = s.nefc;
  const T h2 = 2 * m.timestep;
  for (int r = tl.lane; r < nefc; r += LANES) {
    T* Jr = s.J + r * kLD;
    const int type = s.r_type[r], id = s.r_id[r], sub = s.r_sub[r];
    T pos = 0, diag = 0, imp = 0, K = 0, B = 0;
    if (type == kRowEq) {
      const int l1 = m.eq_l1[id], l2 = m.eq_l2[id];
      T P1[3], P2[3], t[3];
      mulv(t, s.xmat[l1], m.eq_a1[id]);
      for (int i = 0; i < 3; i++) P1[i] = s.xpos[l1][i] + t[i];
      mulv(t, s.xmat[l2], m.eq_a2[id]);
      for (int i = 0; i < 3; i++) P2[i] = s.xpos[l2][i] + t[i];
      const unsigned a1 = m.anc[l1], a2 = m.anc[l2];
      for (int d = 0; d < nv; d++) {
        T v = 0, c3[3];
        if ((a1 >> d) & 1u) { jac_col(c3, s.S[d], P1); v += c3[sub]; }
        if ((a2 >> d) & 1u) { jac_col(c3, s.S[d], P2); v -= c3[sub]; }
        Jr[d] = v;
      }
      const T dv[3] = {P1[0] - P2[0], P1[1] - P2[1], P1[2] - P2[2]};
      pos = dv[sub];
      diag = m.eq_invweight[id];
      const T* sr = m.eq_solref[id];
      const T* si = m.eq_solimp[id];
      imp = impedance(si, sqrt(dot3(dv, dv)), (T)0);
      const T sr0 = (sr[0] > 0 && sr[0] < h2) ? h2 : sr[0];
      K = (T)1 / fmax((T)kMinVal, si[1] * si[1] * sr0 * sr0 * sr[1] * sr[1]);
      B = (T)2 / fmax((T)kMinVal, si[1] * sr0);
    } else if (type == kRowLimit) {
      for (int d = 0; d < nv; d++) Jr[d] = 0;
      Jr[id] = sub == 0 ? (T)1 : (T)-1;
      pos = sub == 0 ? s.q[id + 1] - m.range[id][0] : m.range[id][1] - s.q[id + 1];
      diag = m.dof_invweight[id];
      const T* sr = m.lim_solref[id];
      const T* si = m.lim_solimp[id];
      imp = impedance(si, pos, (T)0);
      const T sr0 = (sr[0] > 0 && sr[0] < h2) ? h2 : sr[0];
      K = (T)1 / fmax((T)kMinVal, si[1] * si[1] * sr0 * sr0 * sr[1] * sr[1]);
      B = (T)2 / fmax((T)kMinVal, si[1] * sr0);
    } else {
      const int p = s.c_pair[id], ga = m.pair_a[p], gb = m.pair_b[p];
      const T* dir = s.c_frame[id] + 3 * sub;
      const T* P = s.c_pos[id];
      const unsigned ab = m.anc[m.g_link[gb]], aa = ga < 0 ? 0u : m.anc[m.g_link[ga]];
      for (int d = 0; d < nv; d++) {
        T v = 0, c3[3];
        if (((ab ^ aa) >> d) & 1u) {     // a dof that moves both bodies alike contributes nothing
          jac_col(c3, s.S[d], P);
          v = dot3(dir, c3);
          if (!((ab >> d) & 1u)) v = -v;
        }
        Jr[d] = v;
      }
      pos = sub == 0 ? s.c_dist[id] : (T)0;
      diag = m.pair_invweight[p];
      const T* sr = m.pair_solref[p];
      const T* si = m.pair_solimp[p];
      imp = impedance(si, s.c_dist[id], (T)0);
      const T sr0 = (sr[0] > 0 && sr[0] < h2) ? h2 : sr[0];
      K = sub == 0 ? (T)1 / fmax((T)kMinVal, si[1] * si[1] * sr0 * sr0 * sr[1] * sr[1]) : (T)0;
      B = (T)2 / fmax((T)kMinVal, si[1] * sr0);
    }
    T R = (1 - imp) * diag / imp;
    if (R < (T)kMinVal) R = (T)kMinVal;
    if (type == kRowContact && sub > 0) R = R / fmax((T)kMinVal, m.impratio);   // tangent rows (friction[0] == friction[1])
    T vel = 0;
    TREE_UNROLL4
    for (int d = 0; d < nv; d++) vel += Jr[d] * s.qd[d];
    s.r_pos[r] = pos;
    s.r_R[r] = R;
    s.r_aref[r] = -B * vel - K * imp * pos;
  }
  tl.sync();
}

// mju_QCQP2
template <typename T>
TREE_FN int qcqp2(T* res, const T* Ain, const T* bin, const T* dd, T r) {
  const T b1 = bin[0] * dd[0], b2 = bin[1] * dd[1];
  const T A11 = Ain[0] * dd[0] * dd[0], A22 = Ain[3] * dd[1] * dd[1], A12 = Ain[1] * dd[0] * dd[1];
  T la = 0, v1 = 0, v2 = 0;
  for (int it = 0; it < 20; it++) {
    const T det = (A11 + la) * (A22 + la) - A12 * A12;
    if (det < (T)1e-10) { res[0] = 0; res[1] = 0; return 0; }
    const T di = 1 / det;
    const T P11 = (A22 + la) * di, P22 = (A11 + la) * di, P12 = -A12 * di;
    v1 = -P11 * b1 - P12 * b2; v2 = -P12 * b1 - P22 * b2;
    const T val = v1 * v1 + v2 * v2 - r * r;
    if (val < (T)1e-10) break;
    const T deriv = -2 * (P11 * v1 * v1 + 2 * P12 * v1 * v2 + P22 * v2 * v2);
    const T delta = -val / deriv;
    if (delta < (T)1e-10) break;
    la += delta;
  }
  res[0] = v1 * dd[0]; res[1] = v2 * dd[1];
  return la != 0;
}

// mj_fwdConstraint: b, A = J M^-1 J^T + R, warm start, PGS (mj_solPGS), qacc, constraint force
template <int LANES, typename T, typename SC>
TREE_FN void solve_constraints(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s) {
  const int nv = m.nv, nefc = s.nefc;
  if (nefc == 0) {
    for (int d = tl.lane; d < nv; d += LANES) { s.qacc[d] = s.qacc_s[d]; s.qfc[d] = 0; }
    if (tl.lane == 0) s.sweeps = 0;
    tl.sync();
    return;
  }
  // b = J qacc_smooth - aref, jar = J qacc_warmstart - aref (kept in r_pos, which make_rows is done with), then
  // Y = L^-1 J^T in place of J, one right-hand side per lane
  for (int r = tl.lane; r < nefc; r += LANES) {
    T* Jr = s.J + r * kLD;
    T bsum = 0, wsum = 0;
    TREE_UNROLL4
    for (int d = 0; d < nv; d++) { bsum += Jr[d] * s.qacc_s[d]; wsum += Jr[d] * s.warm[d]; }
    s.r_b[r] = bsum - s.r_aref[r];
    s.r_pos[r] = wsum - s.r_aref[r];
    forward_row(nv, s, Jr);
  }
  tl.sync();
  for (int r = tl.lane; r < nefc; r += LANES) {
    const T* Yr = s.J + r * kLD;
    T* Ar = s.Am + r * (r + 1) / 2;
    for (int c = 0; c <= r; c++) {
      const T* Yc = s.J + c * kLD;
      T v = 0;
      TREE_UNROLL4
      for (int d = 0; d < nv; d++) v += Yr[d] * Yc[d];
      if (c == r) v += s.r_R[r];
      Ar[c] = v;
    }
  }
  tl.sync();
  // warm start: forces of mj_constraintUpdate at qacc_warmstart, kept only if their dual cost is negative
  for (int r = tl.lane; r < nefc; r += LANES) {
    if (s.r_type[r] == kRowContact && s.r_sub[r] != 0) continue;   // a contact's rows are set by its normal row
    const int type = s.r_type[r];
    const int dim = type == kRowContact ? s.c_dim[s.r_id[r]] : 1;
    T jar[3];
    for (int j = 0; j < dim; j++) jar[j] = s.r_pos[r + j];
    if (type == kRowEq) s.r_f[r] = -jar[0] / s.r_R[r];
    else if (dim == 1) s.r_f[r] = jar[0] < 0 ? -jar[0] / s.r_R[r] : (T)0;    // joint limit, frictionless contact
    else {
      const T* fr = m.pair_friction[s.c_pair[s.r_id[r]]];
      const T mu = fr[0] / sqrt(fmax((T)kMinVal, m.impratio));
      const T U0 = jar[0] * mu, U1 = jar[1] * fr[0], U2 = jar[2] * fr[0];
      const T N = U0, Tn = sqrt(U1 * U1 + U2 * U2);
      if (N >= mu * Tn || (Tn <= 0 && N >= 0)) { s.r_f[r] = s.r_f[r + 1] = s.r_f[r + 2] = 0; }
      else if (mu * N + Tn <= 0 || (Tn <= 0 && N < 0)) {
        for (int j = 0; j < 3; j++) s.r_f[r + j] = -jar[j] / s.r_R[r + j];
      } else {
        const T Dm = ((T)1 / s.r_R[r]) / fmax((T)kMinVal, mu * mu * (1 + mu * mu));
        const T f0 = -Dm * (N - mu * Tn) * mu;
        s.r_f[r] = f0;
        s.r_f[r + 1] = -f0 / Tn * U1 * fr[0];
        s.r_f[r + 2] = -f0 / Tn * U2 * fr[0];
      }
    }
  }
  tl.sync();
  T cost = 0;
  for (int r = tl.lane; r < nefc; r += LANES) {
    s.r_pos[r] = (T)1 / s.Am[r * (r + 1) / 2 + r];        // 1 / A_rr for the scalar-row updates (jar is consumed)
    T v = 0;
    TREE_UNROLL4
    for (int c = 0; c < nefc; c++) v += s.Am[tri(r, c)] * s.r_f[c];
    s.r_acc[r] = v;
    cost += s.r_f[r] * ((T)0.5 * v + s.r_b[r]);
  }
  cost = tl.sum(cost);
  tl.sync();
  for (int r = tl.lane; r < nefc; r += LANES) {
    if (cost > 0) { s.r_f[r] = 0; s.r_acc[r] = s.r_b[r]; }
    else s.r_acc[r] += s.r_b[r];
  }
  tl.sync();
  // PGS: r_acc[r] = b[r] + sum_c A[r][c] f[c] is kept current; a block reads its residual, updates its forces
  // (identically in every lane) and publishes the change to all rows
  const T scale = (T)1 / (m.meaninertia * (T)(nv > 1 ? nv : 1));
  int iter = 0;
#if defined(__CUDACC__)
  if constexpr (LANES >= 8) {
    // The residuals and forces live in REGISTERS of the lanes that own the rows (lane l of the tile owns rows l, l + LANES,
    // ...: K slots), a block's residual / old force is a tile shuffle from its owner, the publish is one FMA per owned row
    // on registers -- no shared-memory traffic for acc / f and no barrier inside the sweep.  Same arithmetic as the general
    // path below (tests/test_gpu_tree.py runs the fp64 parity cases on 8, 16 and 32 lanes; the CPU harness runs the
    // general path).
    constexpr int K = (SC::kRows + LANES - 1) / LANES;
    T acc[K], fr[K];
    int rb[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
      const int q = tl.lane + k * LANES;
      rb[k] = q * (q + 1) / 2;
      acc[k] = q < nefc ? s.r_acc[q] : (T)0;
      fr[k] = q < nefc ? s.r_f[q] : (T)0;
    }
    // value of row `row` from its owner
    auto bcast = [&](const T (&a)[K], int row) -> T {
      T sel = a[0];
#pragma unroll
      for (int k = 1; k < K; k++) sel = row >= k * LANES ? a[k] : sel;
      return __shfl_sync(tl.mask, sel, row & (LANES - 1), LANES);
    };
    // packed index of A[row][q] given the packed starts of rows q (rbq) and row (ib)
#define TREE_AIDX(rbq, q, row, ib) ((q) >= (row) ? (rbq) + (row) : (ib) + (q))
    // row kinds as tile-uniform bit masks (one scan per step instead of three dependent loads per row visit):
    // bit r of `ineq`: row r is clamped at zero (joint limit, frictionless contact); of `head3`: row r opens a condim-3 contact
    unsigned long long ineq = 0ull, head3 = 0ull;
    for (int r = 0; r < nefc; r++) {
      const int ty = s.r_type[r];
      if (ty == kRowLimit) ineq |= 1ull << r;
      else if (ty == kRowContact && s.r_sub[r] == 0) {
        if (s.c_dim[s.r_id[r]] == 1) ineq |= 1ull << r; else head3 |= 1ull << r;
      }
    }
    while (iter < m.iterations) {
      T improvement = 0;
      for (int i = 0, ib = 0; i < nefc;) {            // ib = i (i + 1) / 2: packed start of row i
        const int di = ib + i;
        if (!((head3 >> i) & 1ull)) {
          const T res = bcast(acc, i), old = bcast(fr, i), aii = s.Am[di];
          T fn = old - res * s.r_pos[i];
          if (((ineq >> i) & 1ull) && fn < 0) fn = 0;
          T d0 = fn - old;
          T change = (T)0.5 * d0 * d0 * aii + d0 * res;
          if (change > (T)1e-10) { d0 = 0; change = 0; }
          improvement -= change;
          if (d0 != 0) {
#pragma unroll
            for (int k = 0; k < K; k++) {
              if (k * LANES < nefc) {                       // tile-uniform: slots beyond the row count are skipped whole
                const int q = tl.lane + k * LANES;
                if (q == i) fr[k] = old + d0;
                if (q < nefc) acc[k] += s.Am[TREE_AIDX(rb[k], q, i, ib)] * d0;
              }
            }
          }
          ib += i + 1;
          i += 1;
          continue;
        }
        const int ib1 = ib + i + 1, ib2 = ib1 + i + 2;        // packed starts of rows i + 1, i + 2
        const int d1 = di + i + 1, d2 = d1 + i + 2;
        const T a00 = s.Am[di], a10 = s.Am[d1], a11 = s.Am[d1 + 1], a20 = s.Am[d2], a21 = s.Am[d2 + 1], a22 = s.Am[d2 + 2];
        const T r0 = bcast(acc, i), r1 = bcast(acc, i + 1), r2 = bcast(acc, i + 2);
        const T o0 = bcast(fr, i), o1 = bcast(fr, i + 1), o2 = bcast(fr, i + 2);
        T f0 = o0, f1 = o1, f2 = o2;
        const T* frc = m.pair_friction[s.c_pair[s.r_id[i]]];
        const T mu2[2] = {frc[0], frc[0]};
        if (f0 < (T)kMinVal) {
          f0 -= r0 / a00;
          if (f0 < 0) f0 = 0;
          f1 = f2 = 0;
        } else {
          const T v0 = a00 * f0 + a10 * f1 + a20 * f2, v1 = a10 * f0 + a11 * f1 + a21 * f2, v2 = a20 * f0 + a21 * f1 + a22 * f2;
          const T denom = f0 * v0 + f1 * v1 + f2 * v2;
          if (denom >= (T)kMinVal) {
            T x = -(f0 * r0 + f1 * r1 + f2 * r2) / denom;
            if (f0 + x * f0 < 0) x = -1;
            const T g0 = f0, g1 = f1, g2 = f2;
            f0 += x * g0; f1 += x * g1; f2 += x * g2;
          }
        }
        if (f0 < (T)kMinVal) f1 = f2 = 0;
        else {
          const T Ac[4] = {a11, a21, a21, a22};
          const T bc[2] = {r1 - a11 * o1 - a21 * o2 + a10 * (f0 - o0), r2 - a21 * o1 - a22 * o2 + a20 * (f0 - o0)};
          T v[2];
          const int active = qcqp2(v, Ac, bc, mu2, f0);
          if (active) {
            T sc = v[0] * v[0] / (mu2[0] * mu2[0]) + v[1] * v[1] / (mu2[1] * mu2[1]);
            sc = sqrt(f0 * f0 / fmax((T)kMinVal, sc));
            v[0] *= sc; v[1] *= sc;
          }
          f1 = v[0]; f2 = v[1];
        }
        T e0 = f0 - o0, e1 = f1 - o1, e2 = f2 - o2;
        T change = (T)0.5 * (e0 * (a00 * e0 + a10 * e1 + a20 * e2) + e1 * (a10 * e0 + a11 * e1 + a21 * e2) + e2 * (a20 * e0 + a21 * e1 + a22 * e2)) +
                   e0 * r0 + e1 * r1 + e2 * r2;
        if (change > (T)1e-10) { e0 = e1 = e2 = 0; change = 0; }
        improvement -= change;
        if (e0 != 0 || e1 != 0 || e2 != 0) {
#pragma unroll
          for (int k = 0; k < K; k++) {
            const int q = tl.lane + k * LANES;
            if (q == i) fr[k] = o0 + e0; else if (q == i + 1) fr[k] = o1 + e1; else if (q == i + 2) fr[k] = o2 + e2;
            if (q < nefc)
              acc[k] += s.Am[TREE_AIDX(rb[k], q, i, ib)] * e0 + s.Am[TREE_AIDX(rb[k], q, i + 1, ib1)] * e1 + s.Am[TREE_AIDX(rb[k], q, i + 2, ib2)] * e2;
          }
        }
        ib = ib2 + i + 3;                                   // packed start of row i + 3
        i += 3;
      }
      iter++;
      if (improvement * scale < m.tolerance) break;
    }
#undef TREE_AIDX
#pragma unroll
    for (int k = 0; k < K; k++) {
      const int q = tl.lane + k * LANES;
      if (q < nefc) s.r_f[q] = fr[k];
    }
    tl.sync();
  } else
#endif
  while (iter < m.iterations) {
    T improvement = 0;
    for (int i = 0; i < nefc;) {
      const int type = s.r_type[i];
      const int dim = type == kRowContact ? s.c_dim[s.r_id[i]] : 1;
      const int di = i * (i + 1) / 2 + i;                 // packed index of A[i][i]
      if (dim == 1) {
        // ---- scalar row: connect, joint limit, frictionless contact
        const T res = s.r_acc[i], old = s.r_f[i], aii = s.Am[di];
        T fn = old - res * s.r_pos[i];
        if (type != kRowEq && fn < 0) fn = 0;
        T d0 = fn - old;
        T change = (T)0.5 * d0 * d0 * aii + d0 * res;      // costChange: revert an update that raises the dual cost
        if (change > (T)1e-10) { d0 = 0; change = 0; }
        improvement -= change;
        if (d0 != 0) {                                      // uniform in the tile: every lane holds the same d0
          tl.sync();                                        // every lane has read this row's residual and force
          if (tl.lane == 0) s.r_f[i] = old + d0;
          for (int r = tl.lane; r < nefc; r += LANES) s.r_acc[r] += s.Am[tri(i, r)] * d0;
          tl.sync();
        }
        i += 1;
        continue;
      }
      // ---- condim-3 contact, elliptic cone: rows i (normal), i + 1, i + 2 (tangents); A block symmetric
      const int d1 = di + i + 1, d2 = d1 + i + 2;           // rows i + 1 and i + 2 start i + 1 and 2 i + 3 entries further on
      const T a00 = s.Am[di], a10 = s.Am[d1], a11 = s.Am[d1 + 1], a20 = s.Am[d2], a21 = s.Am[d2 + 1], a22 = s.Am[d2 + 2];
      const T r0 = s.r_acc[i], r1 = s.r_acc[i + 1], r2 = s.r_acc[i + 2];
      const T o0 = s.r_f[i], o1 = s.r_f[i + 1], o2 = s.r_f[i + 2];
      T f0 = o0, f1 = o1, f2 = o2;
      const T* frc = m.pair_friction[s.c_pair[s.r_id[i]]];
      const T mu2[2] = {frc[0], frc[0]};
      if (f0 < (T)kMinVal) {
        f0 -= r0 / a00;
        if (f0 < 0) f0 = 0;
        f1 = f2 = 0;
      } else {
        // ray update: scale the whole force along its own direction
        const T v0 = a00 * f0 + a10 * f1 + a20 * f2, v1 = a10 * f0 + a11 * f1 + a21 * f2, v2 = a20 * f0 + a21 * f1 + a22 * f2;
        const T denom = f0 * v0 + f1 * v1 + f2 * v2;
        if (denom >= (T)kMinVal) {
          T x = -(f0 * r0 + f1 * r1 + f2 * r2) / denom;
          if (f0 + x * f0 < 0) x = -1;
          const T g0 = f0, g1 = f1, g2 = f2;
          f0 += x * g0; f1 += x * g1; f2 += x * g2;
        }
      }
      // tangential update with the normal force fixed
      if (f0 < (T)kMinVal) f1 = f2 = 0;
      else {
        const T Ac[4] = {a11, a21, a21, a22};
        const T bc[2] = {r1 - a11 * o1 - a21 * o2 + a10 * (f0 - o0), r2 - a21 * o1 - a22 * o2 + a20 * (f0 - o0)};
        T v[2];
        const int active = qcqp2(v, Ac, bc, mu2, f0);
        if (active) {
          T sc = v[0] * v[0] / (mu2[0] * mu2[0]) + v[1] * v[1] / (mu2[1] * mu2[1]);
          sc = sqrt(f0 * f0 / fmax((T)kMinVal, sc));
          v[0] *= sc; v[1] *= sc;
        }
        f1 = v[0]; f2 = v[1];
      }
      T e0 = f0 - o0, e1 = f1 - o1, e2 = f2 - o2;
      T change = (T)0.5 * (e0 * (a00 * e0 + a10 * e1 + a20 * e2) + e1 * (a10 * e0 + a11 * e1 + a21 * e2) + e2 * (a20 * e0 + a21 * e1 + a22 * e2)) +
                 e0 * r0 + e1 * r1 + e2 * r2;
      if (change > (T)1e-10) { e0 = e1 = e2 = 0; change = 0; }
      improvement -= change;
      if (e0 != 0 || e1 != 0 || e2 != 0) {
        tl.sync();
        if (tl.lane == 0) { s.r_f[i] = o0 + e0; s.r_f[i + 1] = o1 + e1; s.r_f[i + 2] = o2 + e2; }
        for (int r = tl.lane; r < nefc; r += LANES)
          s.r_acc[r] += s.Am[tri(i, r)] * e0 + s.Am[tri(i + 1, r)] * e1 + s.Am[tri(i + 2, r)] * e2;
        tl.sync();
      }
      i += 3;
    }
    iter++;
    if (improvement * scale < m.tolerance) break;
  }
  if (tl.lane == 0) s.sweeps = iter;
  // z = Y f ; qfrc_constraint = J^T f = L z ; qacc = qacc_smooth + M^-1 J^T f = qacc_smooth + L^-T z
  for (int d = tl.lane; d < nv; d += LANES) {
    T a = 0;
    TREE_UNROLL4
    for (int r = 0; r < nefc; r++) a += s.J[r * kLD + d] * s.r_f[r];
    s.qacc[d] = a;
  }
  tl.sync();
  for (int i = tl.lane; i < nv; i += LANES) {
    T a = 0;
    for (int j = 0; j <= i; j++) a += s.L[i * kLD + j] * s.qacc[j];
    s.qfc[i] = a;
  }
  tl.sync();
  backward_one(tl, nv, s, s.qacc, s.wk);
  for (int d = tl.lane; d < nv; d += LANES) s.qacc[d] = s.qacc_s[d] + s.wk[d];
  tl.sync();
}

// ---------------------------------------------------------------------------------------------- mj_step
struct TreeStats { int nefc, ncon, sweeps, dropped; };

// one simulator step on the state held in the scratch block (s.q, s.qd, s.warm); u = the nu motor controls
// abort_on_overflow: when the step needs more constraint rows / contacts than this instantiation holds, leave the state
// UNTOUCHED and return false (the caller hands the env to the full-capacity instantiation); otherwise the surplus is
// dropped in pair order and counted, like MuJoCo's njmax / nconmax
template <int LANES, typename T, typename SC>
TREE_FN bool tree_step(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* u, TreeStats* st, bool abort_on_overflow = false) {
  const int nv = m.nv;
  dynamics(tl, m, s);                                      // frames, M, bias -> s.tmp
  // smooth force: passive damping - bias + actuation (ctrl clamped to ctrlrange, gear)
  for (int d = tl.lane; d < nv; d += LANES) s.qfrc[d] = -m.damping[d] * s.qd[d] - s.tmp[d];
  tl.sync();
  if (tl.lane == 0)
    for (int a = 0; a < m.nu; a++) {
      T c = u ? u[a] : (T)0;
      if (m.act_limited[a]) c = c < m.act_lo[a] ? m.act_lo[a] : (c > m.act_hi[a] ? m.act_hi[a] : c);
      s.qfrc[m.act_dof[a]] += m.act_gear[a] * c;
    }
  tl.sync();
  cholesky(tl, nv, s, (const T*)nullptr, (T)0);
  for (int d = tl.lane; d < nv; d += LANES) s.qacc_s[d] = s.qfrc[d];
  tl.sync();
  solve_one(tl, nv, s, s.qacc_s);
  collide(tl, m, s);
  make_rows(tl, m, s);
  if (abort_on_overflow && s.overflow) return false;       // tile-uniform (read after make_rows' barrier); q, qd, warm not yet written
  solve_constraints(tl, m, s);
  // mj_Euler: (M + h D) qacc' = qfrc_smooth + qfrc_constraint; qvel += h qacc'; qpos integrated with the NEW velocity
  const T h = m.timestep;
  cholesky(tl, nv, s, m.damping, h);
  for (int d = tl.lane; d < nv; d += LANES) s.tmp[d] = s.qfrc[d] + s.qfc[d];
  tl.sync();
  solve_one(tl, nv, s, s.tmp);
  for (int d = tl.lane; d < nv; d += LANES) {
    s.qd[d] += h * s.tmp[d];
    s.warm[d] = s.qacc[d];
  }
  tl.sync();
  for (int d = tl.lane; d < nv; d += LANES) {
    if (d < 3) s.q[d] += h * s.qd[d];
    else if (d >= 6) s.q[d + 1] += h * s.qd[d];
  }
  if (tl.lane == 0) {
    // mju_quatIntegrate: rotate by h * (body-frame angular velocity), then normalise
    const T w[3] = {s.qd[3], s.qd[4], s.qd[5]};
    const T nw = sqrt(dot3(w, w));
    if (nw > (T)kMinVal) {
      const T ang = (T)0.5 * h * nw, sn = sin(ang) / nw, cs = cos(ang);
      const T r[4] = {cs, sn * w[0], sn * w[1], sn * w[2]};
      const T* q = s.q + 3;
      T o[4] = {q[0] * r[0] - q[1] * r[1] - q[2] * r[2] - q[3] * r[3], q[0] * r[1] + q[1] * r[0] + q[2] * r[3] - q[3] * r[2],
                q[0] * r[2] - q[1] * r[3] + q[2] * r[0] + q[3] * r[1], q[0] * r[3] + q[1] * r[2] - q[2] * r[1] + q[3] * r[0]};
      const T no = (T)1 / sqrt(o[0] * o[0] + o[1] * o[1] + o[2] * o[2] + o[3] * o[3]);
      for (int c = 0; c < 4; c++) s.q[3 + c] = o[c] * no;
    }
  }
  tl.sync();
  if (st) { st->nefc = s.nefc; st->ncon = s.ncon; st->sweeps = s.sweeps; st->dropped += s.n_dropped; }
  return true;
}

}  // namespace tree
}  // namespace cassie
