// Batched ADMM QP core: G adjacent lanes of a warp cooperate on one scenario.
//
// Replaces `problem_full.solve(**kw)` of the reference (tzddpc/tzddpc.py:367), which hands a
// cvxpy-canonicalised cone program to a CPU interior-point solver.  Here the program is the
// parametric QP of tzddpc_b200/program.py in OSQP form, already Ruiz-scaled on the host:
//
//     min 0.5 x'Px + q'x + sum_{kink rows} w_i |(Ax)_i - k_i|    s.t.  l <= Ax <= u
//
// Work split: the rows are sorted by class on the host (two-sided / |.|-cost rows, upper-only
// rows, lower-only rows; each class padded to a multiple of G) and row slot i belongs to lane
// (i mod G) of the scenario's lane group, so every lane owns N2 two-sided, NU upper-only and
// NL lower-only rows -- known at compile time, which removes the dead half of every clip --
// and keeps its rows of (alpha A, bound, z, w, rho) in registers.  The NZ-vector x and the
// NZ x NZ Cholesky factor of the reduced KKT matrix  K = P + sigma I + A' diag(rho) A  are
// replicated in every lane of the group; A'(.) products are group all-reduces with
// xor-shuffles (bitwise identical in every lane, so control flow stays group-uniform).
// ncu evidence for this layout: profiles/r1_v0_* (one thread per scenario: 255 registers,
// spills, 13 % FP64 pipe) and profiles/r1_v1_* (lane groups, un-tuned loop: 20 % of the
// issued instructions were FP64).
//
// Algorithm: OSQP-style ADMM with over-relaxation alpha, plus
//   * the |.| cost rows handled by their prox (soft threshold) inside the z-update, so an
//     LP cost needs no slack variable;
//   * a per-row penalty rho_i switched between rho*rho_active / rho*rho_inactive by the
//     detected activity of the row, on a geometrically growing schedule (updates stop
//     changing once the active set has settled, after which this is plain ADMM);
//   * OSQP's primal-infeasibility certificate on the dual increments;
//   * a masked augmented-Lagrangian polish on the detected active set.
// Inner-loop algebra (per row, 9 FP64 instructions + one 3-instruction clip):
//   the scaled dual w = y / rho is stored instead of y;  Aa = alpha A is stored instead of A
//   and rq = rho / alpha instead of rho, so that  zr = Aa xt + (1-alpha) z  is one chain of
//   FMAs and  A'(rho (z - w)) = Aa'(rq (2 z+ - xi)).
#pragma once
#include "tz_common.cuh"

namespace tz {

#ifndef TZ_SPO_MIN
#define TZ_SPO_MIN 16      // scenarios per output tile (>= 16: full 128-byte lines of every SoA row)
#endif
template <int NZ_, int N2_, int NU_, int NL_, int G_, int NPAR_, int NAG_, int NCHK_, int MINB_>
struct Bucket {
  static constexpr int NZ = NZ_, N2 = N2_, NU = NU_, NL = NL_, G = G_, NPAR = NPAR_, NAG = NAG_, NCHK = NCHK_;
  static constexpr int MINB = MINB_;                  // CTAs per SM the register budget is set for
  static constexpr int NCL = N2 + NU + NL;            // constraint rows per lane
  static constexpr int NC = NCL * G;                  // row slots
  static constexpr int NK = N2 * G;                   // slots that may carry a |.| cost
  static constexpr int NCOL = 1 + 2 * NPAR + NAG;     // [1 | p | |p| | general atoms]
  static constexpr int NCHL = (NCHK + G - 1) / G;
  static constexpr int TPB = 128;
  static constexpr int WPB = TPB / 32;                // warps per CTA
  static constexpr int SPW = 32 / G;                  // scenarios per solve tile of a warp
  static constexpr int TPO = (SPW >= TZ_SPO_MIN) ? 1 : TZ_SPO_MIN / SPW;   // solve tiles per output tile: the output phase always covers
  static constexpr int SPO = SPW * TPO;               //   >= 16 consecutive scenarios = full 128-byte lines of every SoA row
  // layout of the per-scenario vector om = [1 | v (NZ) | xbar0 (HP) | e0 (HP) | centre of Ze[1] (HP) | x+ (HP)], HP = NPAR/2 >= dim_x
  static constexpr int HP = NPAR / 2;
  static constexpr int OM_V = 1, OM_P = 1 + NZ, NW = 1 + NZ + NPAR;
  static constexpr int OM_C = NW, OM_XP = NW + HP, KOM = NW + 2 * HP;
  static constexpr int PRE_ROWS = 4 * HP + G;         // prefetched input rows of an output tile: [xbar0 | e0 | x | noise | hint words]
  static constexpr int NCOL2 = (NCOL + 1) / 2;        // 16-byte pairs of columns per row of R / Rchk
  // row pitch of R / Rchk: even (16-byte aligned rows) and not a multiple of 64 bytes, so that the rows read by the G
  // lanes of a group (16 bytes each, one LDS.128) fall into different banks (a 192-byte pitch gave a 2-way conflict)
  static constexpr int NCOLP = 2 * NCOL2 + ((2 * NCOL2) % 8 == 0 ? 2 : 0);
  static_assert(NCL <= 32 && (G & (G - 1)) == 0 && G <= 32 && N2 >= 1 && NAG >= 1, "bad bucket");
};

// Scaled program, padded to the bucket (padding rows: A = 0, bounds infinite).
template <class BK>
struct QpProg {
  double P[BK::NZ][BK::NZ];
  double A[BK::NC][BK::NZ];            // E A D (NOT multiplied by alpha)
  double l0[BK::NC], u0[BK::NC];
  double kink0[BK::NK], wabs[BK::NK];
  double R[BK::NC][BK::NCOLP];         // UNSCALED shift rows (rows of one tube constraint share them up to a sign, see grp_*)
  double Rs[BK::NC];                   // row scaling E_i:  r_i(p) = Rs_i * (R_i . w)
  double q0[BK::NZ];
  double Qp[BK::NZ][BK::NPAR];
  double Bt[BK::NAG][BK::NPAR];        // general atoms |Bt p + gam| (the unit atoms |p_c| are implicit)
  double gam[BK::NAG];
  double Rchk[BK::NCHK][BK::NCOLP];
  double chk_tol[BK::NCHK];            // 1e-9 max(1, |Rchk[i][0]|)
  double cc[BK::NCOL];
  double CC2[BK::NPAR][BK::NPAR];
  double D[BK::NZ];
  double Einv[BK::NC];
  double sing_inv[BK::NC];              // rows with a single non-zero A[i][j]: 1 / A[i][j] (scaled), else 0
  double cinv;                          // 1 / cost scaling
  int sing_var[BK::NC];                 // ... and j, else -1 (singleton presolve: such rows are bounds on x_j)
  int row_of_slot[BK::NC];              // original row index of a slot, -1 for padding
  // fast_step_kernel's order of the rows: rows that share their shift row R_i up to the sign of its constant / |.| part
  // (the four rows a tube constraint expands into: upper / lower bound x the two signs of its |v| atom) are adjacent, the
  // first of a group computes (L, A) = (linear part, constant + |.| part) of R_i . w and the others reuse it as L +- A
  int grp_order[BK::NC];               // t -> row slot
  int grp_new[BK::NC];                 // t -> 1: first row of a group
  double grp_sgn[BK::NC];              // t -> sign of A relative to the group's first row
  int grp_first[BK::NC + 4];           // group g owns t in [grp_first[g], grp_first[g + 1]); entries beyond ngrp repeat nc
  int ngrp;
  int nz, nc, npar, nag, nchk, has_cc2, has_qp;
};

struct SolverParams {     // TzSolverOpts, device side
  double rho, rho_act, rho_inact, sigma, alpha, eps_abs, eps_rel;
  int max_iter, check_every, polish, warm, cert_first, tube_packed, hot;
};

// compare-select min/max: 3 instructions instead of the ~8 of IEEE fmin/fmax (no NaN quieting needed:
// non-finite inputs are rejected before the solve and NaN iterates are caught by the residual check)
__device__ __forceinline__ double dmin(double a, double b) { return a < b ? a : b; }
__device__ __forceinline__ double dmax(double a, double b) { return a > b ? a : b; }

template <int G>
__device__ __forceinline__ double gsum(double v) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int G>
__device__ __forceinline__ double gmax(double v) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int G>
__device__ __forceinline__ int gor(int v) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) v |= __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int NZ>
__device__ __forceinline__ void chol_factor(double (&K)[NZ][NZ]) {
  // in-place lower Cholesky; the strictly upper part is ignored.  Diagonal stores 1/L_jj.
#pragma unroll
  for (int j = 0; j < NZ; ++j) {
    double d = K[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= K[j][k] * K[j][k];
    d = fmax(d, 1e-300);
    const double inv = rsqrt(d);
    K[j][j] = inv;
#pragma unroll
    for (int i = j + 1; i < NZ; ++i) {
      double s = K[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= K[i][k] * K[j][k];
      K[i][j] = s * inv;
    }
  }
}

template <int NZ>
__device__ __forceinline__ void chol_solve(const double (&L)[NZ][NZ], double (&b)[NZ]) {
#pragma unroll
  for (int i = 0; i < NZ; ++i) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s -= L[i][k] * b[k];
    b[i] = s * L[i][i];
  }
#pragma unroll
  for (int i = NZ - 1; i >= 0; --i) {
    double s = b[i];
#pragma unroll
    for (int k = i + 1; k < NZ; ++k) s -= L[k][i] * b[k];
    b[i] = s * L[i][i];
  }
}

// Per-lane slice of one scenario's QP.  Local row k: k < N2 two-sided / kink, k < N2+NU upper
// only, else lower only.
// This lane's rows of alpha * A, read from shared memory on every use (the matrix is the same for all
// scenarios; keeping the rows in registers cost 2*NCL*NZ registers per thread and a CTA per SM of occupancy).
template <class BK>
struct ARows {
  const double* base;            // &Aa[g][0] of the shared-memory table Aa[NC][NZ]; local row k is slot k*G + g
  __device__ __forceinline__ const double* operator[](int k) const { return base + k * (BK::G * BK::NZ); }
};

template <class BK>
struct LaneQp {
  ARows<BK> Aa;                  // alpha * (this lane's rows of the scaled constraint matrix), in shared memory
  double lo[BK::N2 + BK::NL];    // lower bounds of the two-sided rows, then of the lower-only rows
  double hi[BK::N2 + BK::NU];    // upper bounds of the two-sided rows, then of the upper-only rows
  double kink[BK::N2];
  double q[BK::NZ];
  const double* wk;              // shared memory: |.| weights of this lane's two-sided rows, element k at [k * G]
  const double* sinv;            // shared memory: singleton-row inverse coefficients of this lane's rows, element k at [k * G]
  const int* svar;               // shared memory: singleton-row variable index (-1: not a singleton), element k at [k * G]
  const double (*P)[BK::NZ];     // shared memory: the scaled P (only read at factorisations and residual checks)
  __device__ __forceinline__ double lower(int k) const { return k < BK::N2 ? lo[k] : (k >= BK::N2 + BK::NU ? lo[k - BK::NU] : -INFINITY); }
  __device__ __forceinline__ double upper(int k) const { return k < BK::N2 + BK::NU ? hi[k] : INFINITY; }
  __device__ __forceinline__ double clip(int k, double v) const {
    if (k < BK::N2) return dmin(dmax(v, lo[k]), hi[k]);
    if (k < BK::N2 + BK::NU) return dmin(v, hi[k]);
    return dmax(v, lo[k - BK::NU]);
  }
  __device__ __forceinline__ bool at_bound(int k, double z) const {
    if (k < BK::N2) return (z <= lo[k]) || (z >= hi[k]) || (wk[k * BK::G] > 0.0 && z == kink[k]);
    if (k < BK::N2 + BK::NU) return z >= hi[k];
    return z <= lo[k - BK::NU];
  }
};

template <class BK>
struct LaneState {
  double x[BK::NZ];
  double z[BK::NCL], w[BK::NCL];  // inside admm_solve w = y / rho_row; y on entry (warm) and exit
  uint32_t act;                   // activity bits of the local rows
  bool switched;                  // false: every row still at the base rho
  unsigned long long code;        // active-set code of the returned point (see active_code)
};

// K = P + sigma I + sum_i rho_i a_i a_i'  (group all-reduce of the lower triangle), then factor.
// rq = rho / alpha and Aa = alpha A  =>  rho a a' = (rq / alpha) Aa Aa'.
template <class BK>
__device__ __forceinline__ void build_factor(const LaneQp<BK>& qp, const double (&rq)[BK::NCL], double inv_alpha,
                                             double sigma, double (&L)[BK::NZ][BK::NZ]) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, G = BK::G;
#pragma unroll
  for (int a = 0; a < NZ; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = 0.0;
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
#pragma unroll
    for (int a = 0; a < NZ; ++a) {
      const double ra = rq[k] * qp.Aa[k][a];
#pragma unroll
      for (int b = 0; b <= a; ++b) L[a][b] = fma(ra, qp.Aa[k][b], L[a][b]);
    }
  }
#pragma unroll
  for (int a = 0; a < NZ; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = fma(gsum<G>(L[a][b]), inv_alpha, qp.P[a][b] + (a == b ? sigma : 0.0));
  chol_factor<NZ>(L);
}

// Singleton presolve: a row with one non-zero coefficient is a bound on one variable; if the
// bounds on some x_j collected from all such rows are inconsistent the program is infeasible --
// decided exactly and at once, where ADMM needs ~100 iterations to build its Farkas certificate.
// (All infeasible closed-loop instances of the shipped examples are of this kind: the tightened
// state rows at k = 1 depend on v_0 only.)  Whole warps; returns a group-uniform flag.
template <class BK>
__device__ __forceinline__ bool singleton_infeasible(const LaneQp<BK>& qp) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, G = BK::G;
  double blo[NZ], bhi[NZ];
#pragma unroll
  for (int j = 0; j < NZ; ++j) { blo[j] = -INFINITY; bhi[j] = INFINITY; }
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    const int sv = qp.svar[k * G];
    const double inv = qp.sinv[k * G];
    const double a = qp.lower(k) * inv, b = qp.upper(k) * inv;
    const double lo = inv > 0.0 ? a : b, hi = inv > 0.0 ? b : a;
#pragma unroll
    for (int j = 0; j < NZ; ++j) {
      blo[j] = (sv == j && lo > blo[j]) ? lo : blo[j];
      bhi[j] = (sv == j && hi < bhi[j]) ? hi : bhi[j];
    }
  }
  int bad = 0;
#pragma unroll
  for (int j = 0; j < NZ; ++j) {
    const double lo = gmax<G>(blo[j]), hi = -gmax<G>(-bhi[j]);
    const double sc = fmax(1.0, fmin(fabs(lo), fabs(hi)));
    bad |= (lo - hi > 1e-9 * sc) ? 1 : 0;
  }
  return bad != 0;
}

// ---- active-set codes: 3 bits per local row, packed into one 64-bit word per lane ----------------
//   0 inactive   1 on its lower bound   2 on its upper bound   3 on the kink of its |.| cost
//   4 / 5 |.| row above / below its kink (linear cost)          6 equality row (lower == upper)
// bit 63 marks a valid word when it travels through the hint buffer.
constexpr unsigned long long kCodeValid = 1ull << 63;
// bit 62: the word was copied from the scenario's run-start hint when it restarted (the state is a run's first state)
constexpr unsigned long long kCodeFresh = 1ull << 62;

template <class BK>
__device__ __forceinline__ unsigned long long active_code(const LaneQp<BK>& qp, const double (&z)[BK::NCL]) {
  constexpr int NCL = BK::NCL, N2 = BK::N2, G = BK::G;
  unsigned long long code = 0ull;
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    const double lo = qp.lower(k), hi = qp.upper(k);
    unsigned c = 0u;
    if (z[k] <= lo) c = lo < hi ? 1u : 6u;
    else if (z[k] >= hi) c = 2u;
    else if (k < N2) {
      if (qp.wk[(k < N2 ? k : 0) * G] > 0.0) {
        const double kk = qp.kink[k < N2 ? k : 0];
        c = z[k] == kk ? 3u : (z[k] > kk ? 4u : 5u);
      }
    }
    code |= (unsigned long long)c << (3 * k);
  }
  return code;
}

// Active-set certificate: the polish used as a TERMINATION TEST.
// Given a guess of the active set (the rows ADMM has clipped onto a bound or onto the kink of their |.| cost, or
// the optimal set of the previous closed-loop step), the equality-constrained problem on that set is solved with
// n_iter masked augmented-Lagrangian steps
//   K = P + delta I + mu sum_act b_i b_i',   x <- K^{-1}(delta x - qt + sum_act b_i (mu t_i - lam_i)),   lam_i += mu (b_i x - t_i)
// (b_i = alpha a_i, t_i = alpha * bound: only NZ x NZ systems, no index compaction), and then the KKT conditions
// of the ORIGINAL problem are checked: every row feasible, active rows on their bound, multipliers of the right
// sign (|y| <= w on a kink), |.| rows on the assumed side of their kink.  Stationarity
// P x + qt + B'lam = delta (x_prev - x) holds by construction.  When all hold, (xk, y) is an exact primal-dual
// solution whatever the ADMM residuals are -- after 3 ADMM iterations from a cold start for almost every
// closed-loop instance of the shipped examples, and after none when the previous step's set is still optimal.
// A wrong guess only costs the test.  Must be called by whole warps.  lam: in y / alpha of the current
// iterate (or zeros), out y (when accepted).  Returns a group-uniform flag.
template <class BK>
__device__ __forceinline__ bool admm_certify(const LaneQp<BK>& qp, double inv_alpha, int n_iter, unsigned long long code,
                                             const double (&x0)[BK::NZ], double (&lam)[BK::NCL], double (&xk)[BK::NZ]) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, N2 = BK::N2, G = BK::G;
  const double delta = 1e-9, mu = 1e6, alpha = 1.0 / inv_alpha;
  double L[NZ][NZ], qt[NZ], tgt[NCL];
  double sgs[N2], rlx[N2];               // |.| rows: subgradient of the assumed side; slack of the sign test when bound == kink
  uint32_t am = 0u;                      // active rows (on a bound / on the kink / equality)
  auto cof = [&](int k) { return (unsigned)(code >> (3 * k)) & 7u; };
#pragma unroll
  for (int a = 0; a < NZ; ++a) {
    qt[a] = 0.0;
    xk[a] = x0[a];
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = 0.0;
  }
  // decode the code once: active mask, alpha * (the bound the row sits on), subgradients of the |.| rows off their kink
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    const unsigned c = cof(k);
    const bool ia = (c >= 1u && c <= 3u) || c == 6u;
    double b = (c == 2u) ? qp.upper(k) : qp.lower(k);
    if (k < N2) {
      const double kk = qp.kink[k < N2 ? k : 0];
      const double wgt = qp.wk[(k < N2 ? k : 0) * G];
      if (c == 3u) b = kk;
      // a |.| row off its kink -- free (codes 4 / 5) or resting on a finite bound away from the kink -- contributes the
      // linear cost of its side; when the bound coincides with the kink the whole interval [-w, w] is available
      double sg = 0.0, rl = 0.0;
      if (c == 4u) sg = wgt;
      else if (c == 5u) sg = -wgt;
      else if (wgt > 0.0 && (c == 1u || c == 2u || c == 6u)) {
        if (b > kk) sg = wgt;
        else if (b < kk) sg = -wgt;
        else rl = wgt;
      }
      sgs[k < N2 ? k : 0] = sg;
      rlx[k < N2 ? k : 0] = rl;
      const double sga = sg * inv_alpha;
#pragma unroll
      for (int a = 0; a < NZ; ++a) qt[a] = fma(sga, qp.Aa[k][a], qt[a]);
    }
    tgt[k] = ia ? b * alpha : 0.0;
    am |= ia ? (1u << k) : 0u;
    const double m_ = ia ? mu : 0.0;
    lam[k] = ia ? lam[k] : 0.0;
#pragma unroll
    for (int a = 0; a < NZ; ++a) {
      const double ra = m_ * qp.Aa[k][a];
#pragma unroll
      for (int c2 = 0; c2 <= a; ++c2) L[a][c2] = fma(ra, qp.Aa[k][c2], L[a][c2]);
    }
  }
#pragma unroll
  for (int a = 0; a < NZ; ++a) {
    qt[a] = gsum<G>(qt[a]) + qp.q[a];
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = gsum<G>(L[a][b]) + qp.P[a][b] + (a == b ? delta : 0.0);
  }
  chol_factor<NZ>(L);
  double xprev[NZ];
#pragma unroll
  for (int a = 0; a < NZ; ++a) xprev[a] = xk[a];
#pragma unroll 1
  for (int it = 0; it < n_iter; ++it) {
    double rhs[NZ];
#pragma unroll
    for (int a = 0; a < NZ; ++a) { rhs[a] = 0.0; xprev[a] = xk[a]; }
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      const double t = ((am >> k) & 1u) ? fma(mu, tgt[k], -lam[k]) : 0.0;
#pragma unroll
      for (int a = 0; a < NZ; ++a) rhs[a] = fma(qp.Aa[k][a], t, rhs[a]);
    }
#pragma unroll
    for (int a = 0; a < NZ; ++a) rhs[a] = gsum<G>(rhs[a]) + fma(delta, xk[a], -qt[a]);
    chol_solve<NZ>(L, rhs);
#pragma unroll
    for (int a = 0; a < NZ; ++a) xk[a] = rhs[a];
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      double ax = 0.0;
#pragma unroll
      for (int a = 0; a < NZ; ++a) ax = fma(qp.Aa[k][a], xk[a], ax);
      lam[k] = ((am >> k) & 1u) ? fma(mu, ax - tgt[k], lam[k]) : lam[k];
    }
  }
  // ---- KKT certificate
  double scale = 1.0, lscale = 1.0;
  double axs[NCL];
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    double ax = 0.0;
#pragma unroll
    for (int a = 0; a < NZ; ++a) ax = fma(qp.Aa[k][a], xk[a], ax);
    axs[k] = ax * inv_alpha;
    scale = fmax(scale, fabs(axs[k]));
    lscale = fmax(lscale, fabs(lam[k]));
  }
  scale = gmax<G>(scale);
  lscale = gmax<G>(lscale);
  const double ptol = 1e-9 * scale, ltol = 1e-9 * lscale, etol = 1e-8 * scale;
  int bad = 0;
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    const double ax = axs[k];
    const unsigned c = cof(k);
    bad |= (qp.lower(k) - ax > ptol) || (ax - qp.upper(k) > ptol);                 // primal feasibility
    // the code is caller memory when it comes from a hint: it must mean something for its row -- 6 only where the bounds
    // coincide, 3 only on a row with a |.| cost, 1 / 2 only on a finite bound, and a |.| row is on its kink, on a side of
    // it or on a bound (never 0 / 7, which would drop its cost).  active_code writes nothing else.
    const bool kinked = k < N2 && qp.wk[(k < N2 ? k : 0) * G] > 0.0;
    bad |= (c == 6u && qp.lower(k) < qp.upper(k)) || (c == 3u && !kinked) || (c == 1u && !(qp.lower(k) > -INFINITY)) ||
           (c == 2u && !(qp.upper(k) < INFINITY)) || (kinked && (c == 0u || c == 7u));
    if ((am >> k) & 1u) {
      const double rl = k < N2 ? rlx[k < N2 ? k : 0] * inv_alpha : 0.0;
      bad |= fabs(ax - tgt[k] * inv_alpha) > etol;                                // active rows on their bound
      bad |= (c == 2u) && (lam[k] < -ltol - rl);                                  // multiplier signs
      bad |= (c == 1u) && (lam[k] > ltol + rl);
      if (k < N2) bad |= (c == 3u) && (fabs(lam[k]) * alpha > qp.wk[(k < N2 ? k : 0) * G] * (1.0 + 1e-9));
      lam[k] *= alpha;                                                            // y
      if (k < N2) lam[k] += sgs[k < N2 ? k : 0];                                  // ... of the row: bound multiplier + cost subgradient
    } else if (k < N2 && (c == 4u || c == 5u)) {
      const double kk = qp.kink[k < N2 ? k : 0];
      const double wgt = qp.wk[(k < N2 ? k : 0) * G];
      bad |= (c == 4u) ? !(ax > kk) : !(ax < kk);                                 // side of the kink as assumed
      lam[k] = (c == 4u) ? wgt : -wgt;
    }
  }
  // stationarity: P x + qt + B'lam = delta (x_prev - x) by construction of the sweeps, so the residual is the last
  // proximal step -- small at a KKT point, but NOT when the active set leaves a direction in which the cost is linear
  // and non-zero (an LP with fewer active rows than variables): the iterate then runs away along it
  double qs = lscale;
#pragma unroll
  for (int a = 0; a < NZ; ++a) qs = fmax(qs, fabs(qt[a]));
#pragma unroll
  for (int a = 0; a < NZ; ++a) bad |= !(delta * fabs(xprev[a] - xk[a]) <= 1e-9 * qs);
#pragma unroll
  for (int a = 0; a < NZ; ++a) bad |= !(xk[a] == xk[a]);
  return gor<G>(bad) == 0;
}

// ADMM for the scenario owned by this lane group.  Every lane of the warp must call it
// (shuffles and warp votes inside); `live` is group-uniform.  On a warm start st.x, st.w
// (holding y), st.act, st.switched are inputs.  Returns TZ_STATUS_*; st.w holds y on exit.
template <class BK>
__device__ int admm_solve(const LaneQp<BK>& qp, const SolverParams& sp, bool live, LaneState<BK>& st, bool warm,
                          double* __restrict__ ysave /* lane-private shared scratch, element k at [k * 32] */,
                          int& iters_out, bool& certified, bool presolved_in = false) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, N2 = BK::N2, G = BK::G;
  const double alpha = sp.alpha, sigma = sp.sigma, oma = 1.0 - sp.alpha, inv_alpha = 1.0 / sp.alpha;
  const double rq_base = sp.rho * inv_alpha, rq_act = sp.rho * sp.rho_act * inv_alpha,
               rq_inact = sp.rho * sp.rho_inact * inv_alpha;
  // reciprocals once per solve (a double division costs ~40 instructions): 1 / rho_row and 1 / rq_row
  const double irho_base = 1.0 / sp.rho, irho_act = 1.0 / (sp.rho * sp.rho_act), irho_inact = 1.0 / (sp.rho * sp.rho_inact);
  const double irq_act = irho_act * alpha, irq_inact = irho_inact * alpha;
  auto irho_of = [&](double rqv) { return rqv == rq_act ? irho_act : (rqv == rq_inact ? irho_inact : irho_base); };

  double rq[NCL];                     // rho_row / alpha
  if (!warm) {
#pragma unroll
    for (int k = 0; k < NCL; ++k) rq[k] = rq_base;
    if (live) {             // (a lane that is not solved keeps its state: it may hold a hint-certified solution)
#pragma unroll
      for (int j = 0; j < NZ; ++j) st.x[j] = 0.0;
#pragma unroll
      for (int k = 0; k < NCL; ++k) st.w[k] = 0.0;
      st.act = 0u;
      st.switched = false;
    }
  } else {
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      rq[k] = ((st.act >> k) & 1u) ? rq_act : rq_inact;
      st.w[k] = st.w[k] * irho_of(rq[k]);                  // y -> w
    }
  }
  // initial z = clip(A x)
  if (live) {
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      double ax = 0.0;
#pragma unroll
      for (int j = 0; j < NZ; ++j) ax = fma(qp.Aa[k][j], st.x[j], ax);
      st.z[k] = qp.clip(k, ax * inv_alpha);
    }
  }
  double qn = 0.0;
#pragma unroll
  for (int j = 0; j < NZ; ++j) qn = fmax(qn, fabs(qp.q[j]));

  double L[NZ][NZ];
  build_factor<BK>(qp, rq, inv_alpha, sigma, L);
  double th[N2];                      // soft thresholds wk / rho of the |.| rows
#pragma unroll
  for (int k = 0; k < N2; ++k) th[k] = qp.wk[k * G] * irho_of(rq[k]);

  int status = TZ_STATUS_MAXITER;
  bool done = !live;
  int iters = 0;
  int next_upd = 2, gap = 2;
  int next_cert = sp.cert_first > 0 ? sp.cert_first : sp.max_iter + 1, cert_gap = 2;     // tests at cert_first + {0, 2, 5, 10, 18, ...}
  certified = false;
  bool presolved = presolved_in;
  const int check_every = sp.check_every > 0 ? sp.check_every : 1;
  int until_check = check_every;
  bool have_prev = false;             // ysave holds the duals of the previous check

  for (int it = 1; it <= sp.max_iter; ++it) {
    // ---- x-update: K xt = sigma x - q + A'(rho (z - w))     [shuffles: whole warp]
    double xt[NZ];
#pragma unroll
    for (int j = 0; j < NZ; ++j) xt[j] = 0.0;
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      const double t = rq[k] * (st.z[k] - st.w[k]);
#pragma unroll
      for (int j = 0; j < NZ; ++j) xt[j] = fma(qp.Aa[k][j], t, xt[j]);
    }
#pragma unroll
    for (int j = 0; j < NZ; ++j) xt[j] = gsum<G>(xt[j]) + fma(sigma, st.x[j], -qp.q[j]);
    if (!done) {
      chol_solve<NZ>(L, xt);
      // ---- z / w update (prox of the |.| rows), row by row
#pragma unroll
      for (int k = 0; k < NCL; ++k) {
        double zr = oma * st.z[k];
#pragma unroll
        for (int j = 0; j < NZ; ++j) zr = fma(qp.Aa[k][j], xt[j], zr);        // alpha (A xt) + (1-alpha) z
        const double xi = zr + st.w[k];
        double pr = xi;
        if (k < N2) {                           // prox of wk|z - kink| : soft threshold around the kink
          const double d = xi - qp.kink[k < N2 ? k : 0];
          pr = qp.kink[k < N2 ? k : 0] + copysign(dmax(fabs(d) - th[k < N2 ? k : 0], 0.0), d);
        }
        const double zn = qp.clip(k, pr);
        st.w[k] = xi - zn;
        st.z[k] = zn;
      }
#pragma unroll
      for (int j = 0; j < NZ; ++j) st.x[j] = fma(alpha, xt[j], oma * st.x[j]);
      iters = it;
    }
    bool sync_point = false;
    if (it == next_cert) {
      next_cert += cert_gap;
      cert_gap = (cert_gap * 3 + 1) / 2;
      double lam[NCL], xk[NZ];
#pragma unroll
      for (int k = 0; k < NCL; ++k) lam[k] = rq[k] * st.w[k];
      const unsigned long long code = active_code<BK>(qp, st.z);
      const bool ok = admm_certify<BK>(qp, inv_alpha, sp.polish > 0 ? sp.polish : 3, code, st.x, lam, xk);
      if (ok && !done) {
#pragma unroll
        for (int j = 0; j < NZ; ++j) st.x[j] = xk[j];
#pragma unroll
        for (int k = 0; k < NCL; ++k) st.w[k] = lam[k];         // y itself: the final w -> y conversion is skipped
        st.code = code;
        status = TZ_STATUS_OK;
        done = true;
        certified = true;
      }
      if (!presolved && __any_sync(0xffffffffu, !done)) {      // first failed certificate: is the program infeasible outright?
        presolved = true;
        const bool inf = singleton_infeasible<BK>(qp);
        if (inf && !done) {
          status = TZ_STATUS_INFEASIBLE;
          done = true;
        }
      }
      sync_point = true;
    }
    const bool check = (--until_check == 0) || (it == sp.max_iter);
    if (check) {
      sync_point = true;
      until_check = check_every;
      // ---- residuals (scaled space); dual increment since the previous check for the certificate
      double rp = 0.0, pn = 0.0, dy_norm = 0.0, supp = 0.0, dy_inf = 0.0;
      double aty[NZ], atdy[NZ];
#pragma unroll
      for (int j = 0; j < NZ; ++j) aty[j] = atdy[j] = 0.0;
#pragma unroll
      for (int k = 0; k < NCL; ++k) {
        double ax = 0.0;
#pragma unroll
        for (int j = 0; j < NZ; ++j) ax = fma(qp.Aa[k][j], st.x[j], ax);
        ax *= inv_alpha;
        rp = fmax(rp, fabs(ax - st.z[k]));
        pn = fmax(pn, fmax(fabs(ax), fabs(st.z[k])));
        const double yk = rq[k] * st.w[k];                   // y / alpha (invariant under rho switches)
        const double dy = yk - ysave[k * 32];
        ysave[k * 32] = yk;
        dy_norm = fmax(dy_norm, fabs(dy));
#pragma unroll
        for (int j = 0; j < NZ; ++j) {
          aty[j] = fma(qp.Aa[k][j], yk, aty[j]);
          atdy[j] = fma(qp.Aa[k][j], dy, atdy[j]);
        }
        // support function of [l, u] along dy; a component pushing against an infinite bound
        // must vanish for dy to be a certificate (rounding leaves O(eps) residues there)
        if (k < N2) {
          if (dy > 0.0) { if (qp.upper(k) < 1e300) supp = fma(qp.upper(k), dy, supp); else dy_inf = fmax(dy_inf, dy); }
          if (dy < 0.0) { if (qp.lower(k) > -1e300) supp = fma(qp.lower(k), dy, supp); else dy_inf = fmax(dy_inf, -dy); }
        } else if (k < N2 + BK::NU) {
          if (dy > 0.0) supp = fma(qp.upper(k), dy, supp); else dy_inf = fmax(dy_inf, -dy);
        } else {
          if (dy < 0.0) supp = fma(qp.lower(k), dy, supp); else dy_inf = fmax(dy_inf, dy);
        }
      }
      rp = gmax<G>(rp);
      pn = gmax<G>(pn);
      dy_norm = gmax<G>(dy_norm);
      dy_inf = gmax<G>(dy_inf);
      supp = gsum<G>(supp);
      double rd = 0.0, pxn = 0.0, atyn = 0.0, atdyn = 0.0;
#pragma unroll
      for (int j = 0; j < NZ; ++j) {
        const double atyj = gsum<G>(aty[j]);
        const double atdyj = gsum<G>(atdy[j]);
        double px = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) px = fma(qp.P[j][b], st.x[b], px);
        rd = fmax(rd, fabs(px + qp.q[j] + atyj));
        pxn = fmax(pxn, fabs(px));
        atyn = fmax(atyn, fabs(atyj));
        atdyn = fmax(atdyn, fabs(atdyj));
      }
      const double ep = sp.eps_abs + sp.eps_rel * pn;
      const double ed = sp.eps_abs + sp.eps_rel * fmax(fmax(pxn, atyn), qn);
      if (!done) {
        if (!(rp == rp) || !(rd == rd)) {
          status = TZ_STATUS_NONFINITE;
          done = true;
        } else if (rp <= ep && rd <= ed) {
          status = TZ_STATUS_OK;
          done = true;
        } else if (have_prev && dy_norm > 1e-12 && dy_inf <= 1e-6 * dy_norm && atdyn <= 1e-6 * dy_norm &&
                   supp < -1e-6 * dy_norm) {
          status = TZ_STATUS_INFEASIBLE;     // Farkas certificate (OSQP, Banjac et al. 2019)
          done = true;
        }
      }
      have_prev = true;
    }
    if (sync_point && __all_sync(0xffffffffu, done)) break;
    // ---- activity-driven rho switch on a geometric schedule
    if (it == next_upd) {
      gap = (gap * 3 + 1) / 2;
      next_upd = it + gap;
      uint32_t nm = 0u;
#pragma unroll
      for (int k = 0; k < NCL; ++k) nm |= (qp.at_bound(k, st.z[k]) ? 1u : 0u) << k;
      const int changed = gor<G>((!st.switched || nm != st.act) ? 1 : 0);
      const bool apply = changed && !done;
      if (apply) {
#pragma unroll
        for (int k = 0; k < NCL; ++k) {      // keep y = rho w invariant under the switch
          const bool on = (nm >> k) & 1u;
          st.w[k] *= rq[k] * (on ? irq_act : irq_inact);
          rq[k] = on ? rq_act : rq_inact;
        }
        st.act = nm;
        st.switched = true;
#pragma unroll
        for (int k = 0; k < N2; ++k) th[k] = qp.wk[k * G] * irho_of(rq[k]);
      }
      // the factor is rebuilt with group shuffles, so the whole warp takes the branch together
      if (__any_sync(0xffffffffu, apply)) {
        double Lt[NZ][NZ];
        build_factor<BK>(qp, rq, inv_alpha, sigma, Lt);
        if (apply) {
#pragma unroll
          for (int a = 0; a < NZ; ++a)
#pragma unroll
            for (int c = 0; c <= a; ++c) L[a][c] = Lt[a][c];
        }
      }
    }
  }
  // hand y (not w) back to the caller
  if (!certified && live) {
#pragma unroll
    for (int k = 0; k < NCL; ++k) st.w[k] *= rq[k] * alpha;
    st.code = active_code<BK>(qp, st.z);
  }
  iters_out = iters;
  return live ? status : TZ_STATUS_OK;
}

// Polish: solve the equality-constrained QP on the detected active set with a masked
// augmented-Lagrangian iteration (only NZ x NZ systems, no index compaction):
//   K = P + delta I + mu sum_{i active} a_i a_i',  x <- K^{-1}(delta x - qt + sum_act a_i (mu b_i - lam_i)),
//   lam_i <- lam_i + mu (a_i x - b_i).   Accepted only if the result is feasible.
// st.w holds y on entry and on exit.  Must be called by whole warps (shuffles).
template <class BK>
__device__ bool admm_polish(const LaneQp<BK>& qp, double inv_alpha, LaneState<BK>& st, bool apply, int n_iter) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, N2 = BK::N2, G = BK::G;
  const double delta = 1e-9, mu = 1e6;
  double L[NZ][NZ], qt[NZ], xk[NZ], tgt[NCL];
  double psg[N2];                  // cost subgradient of a |.| row that rests on a bound away from its kink
  uint32_t act = 0u;
#pragma unroll
  for (int a = 0; a < NZ; ++a) {
    qt[a] = 0.0;
    xk[a] = st.x[a];
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    bool ia = false;
    double b = 0.0;
    bool onb = false;
    if (st.z[k] <= qp.lower(k)) { b = qp.lower(k); ia = true; onb = true; }
    else if (st.z[k] >= qp.upper(k)) { b = qp.upper(k); ia = true; onb = true; }
    else if (k < N2) {
      const double kk = qp.kink[k < N2 ? k : 0];
      if (qp.wk[(k < N2 ? k : 0) * G] > 0.0 && st.z[k] == kk) { b = kk; ia = true; }
    }
    tgt[k] = b * (1.0 / inv_alpha);          // compare against Aa x = alpha (A x)
    if (k < N2 && onb) {                     // a |.| row resting on a bound away from its kink: the linear cost of that side
      const double wgt = qp.wk[(k < N2 ? k : 0) * G];
      const double kk = qp.kink[k < N2 ? k : 0];
      const double sg = (wgt > 0.0 && b != kk) ? (b > kk ? wgt : -wgt) : 0.0;
      psg[k < N2 ? k : 0] = sg;
      if (ia) st.w[k] -= sg;                 // the bound's own multiplier
#pragma unroll
      for (int a = 0; a < NZ; ++a) qt[a] = fma(sg * inv_alpha, qp.Aa[k][a], qt[a]);
    } else if (k < N2) psg[k < N2 ? k : 0] = 0.0;
    if (ia) {
      act |= 1u << k;
#pragma unroll
      for (int a = 0; a < NZ; ++a) {
        const double ra = mu * qp.Aa[k][a];
#pragma unroll
        for (int c = 0; c <= a; ++c) L[a][c] = fma(ra, qp.Aa[k][c], L[a][c]);
      }
    } else {
      st.w[k] = 0.0;
      if (k < N2) {              // |.| row away from its kink: a linear cost term
        const double wgt = qp.wk[(k < N2 ? k : 0) * G];
        if (wgt > 0.0) {
          const double sg = st.z[k] > qp.kink[k < N2 ? k : 0] ? wgt : -wgt;
          st.w[k] = sg;          // its multiplier is the subgradient
#pragma unroll
          for (int a = 0; a < NZ; ++a) qt[a] = fma(sg * inv_alpha, qp.Aa[k][a], qt[a]);
        }
      }
    }
  }
  // work with B = Aa (= alpha A): the active equalities B x = alpha b, multipliers lamB = y / alpha
#pragma unroll
  for (int k = 0; k < NCL; ++k)
    if ((act >> k) & 1u) st.w[k] *= inv_alpha;
#pragma unroll
  for (int a = 0; a < NZ; ++a) {
    qt[a] = gsum<G>(qt[a]) + qp.q[a];
#pragma unroll
    for (int b = 0; b <= a; ++b) L[a][b] = gsum<G>(L[a][b]) + qp.P[a][b] + (a == b ? delta : 0.0);
  }
  chol_factor<NZ>(L);
#pragma unroll 1
  for (int it = 0; it < n_iter; ++it) {
    double rhs[NZ];
#pragma unroll
    for (int a = 0; a < NZ; ++a) rhs[a] = 0.0;
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      if ((act >> k) & 1u) {
        const double t = fma(mu, tgt[k], -st.w[k]);
#pragma unroll
        for (int a = 0; a < NZ; ++a) rhs[a] = fma(qp.Aa[k][a], t, rhs[a]);
      }
    }
#pragma unroll
    for (int a = 0; a < NZ; ++a) rhs[a] = gsum<G>(rhs[a]) + fma(delta, xk[a], -qt[a]);
    chol_solve<NZ>(L, rhs);
#pragma unroll
    for (int a = 0; a < NZ; ++a) xk[a] = rhs[a];
#pragma unroll
    for (int k = 0; k < NCL; ++k) {
      if ((act >> k) & 1u) {
        double ax = 0.0;
#pragma unroll
        for (int a = 0; a < NZ; ++a) ax = fma(qp.Aa[k][a], xk[a], ax);
        st.w[k] = fma(mu, ax - tgt[k], st.w[k]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NCL; ++k)
    if ((act >> k) & 1u) st.w[k] = fma(st.w[k], 1.0 / inv_alpha, k < N2 ? psg[k < N2 ? k : 0] : 0.0);      // back to y (+ the cost subgradient)
  // accept only a feasible polished point
  double viol = 0.0, scale = 1.0;
#pragma unroll
  for (int k = 0; k < NCL; ++k) {
    double ax = 0.0;
#pragma unroll
    for (int a = 0; a < NZ; ++a) ax = fma(qp.Aa[k][a], xk[a], ax);
    ax *= inv_alpha;
    viol = fmax(viol, fmax(qp.lower(k) - ax, ax - qp.upper(k)));
    scale = fmax(scale, fabs(ax));
  }
  viol = gmax<G>(viol);
  scale = gmax<G>(scale);
  bool ok = (viol <= 1e-9 * scale);
#pragma unroll
  for (int a = 0; a < NZ; ++a) ok = ok && (xk[a] == xk[a]);
  if (ok && apply) {
#pragma unroll
    for (int a = 0; a < NZ; ++a) st.x[a] = xk[a];
  }
  return ok;
}

}  // namespace tz
