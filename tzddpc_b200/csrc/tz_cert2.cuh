// Closed-form active-set certificate for programs with TWO decision variables (bucket B0: horizon 2, one input --
// every shipped example; tzddpc/tzddpc.py:357-377 solved per closed-loop step).
//
// One THREAD decides one scenario.  Given a guess of the active set (the optimal set of the scenario's previous
// closed-loop step, 3 bits per row as tz_admm.cuh's active_code writes them) the equality-constrained problem on
// that set has at most two active rows in a non-degenerate vertex / edge / interior optimum of a 2-variable program,
// so its KKT system is solved in closed form:
//
//     0 active rows   P x = -qt                         (minimum-norm solution when P is singular)
//     1 active row    x = t a/|a|^2 + s d,  d _|_ a,    s from the reduced curvature d'Pd (s = 0 when it is flat)
//     2 active rows   x = [a; b]^-1 [ta; tb],           multipliers from [a b] lam = -(P x + qt)
//
// with qt = q + sum of the +-w a_i of the |.|-cost rows that sit off their kink.  The KKT conditions of the ORIGINAL
// problem are then checked row by row -- stationarity residual, primal feasibility of every row, multiplier signs
// (|lam| <= w on a kink; a |.| row resting on a finite bound carries the subgradient of its side, and the whole
// interval [-w, w] when the bound coincides with the kink), |.| rows on the assumed side -- so an accepted point is an
// exact primal-dual solution; a wrong or stale guess only costs the test.
//
// The rows are STREAMED: r_i(p) = R_i . w is recomputed from the shared-memory program for every row (all lanes of a
// warp read the same address: one broadcast load serves 32 scenarios) instead of being kept in registers, so a thread
// needs w (24 doubles) and a handful of scalars.  Replaces the three augmented-Lagrangian sweeps of admm_certify on the
// hint path (1,881 straight-line instructions per 8 scenarios, profiles/r1_v12_*).
//
// step_kernel (G lanes per scenario) calls the same function redundantly in the G lanes of a group, so a scenario gets
// bit-identical results whichever kernel decides it.
#pragma once
#include "tz_admm.cuh"

namespace tz {

// (L, A) of row i: L = sum over the parameter columns p, A = constant + |p| + general atoms (columns ascending, one fma
// chain each).  Rows of one tube constraint share L and have A up to a sign (exactly: negation commutes with rounding).
template <class BK>
__device__ __forceinline__ void row_LA(const QpProg<BK>& pg, int i, const double (&w)[2 * BK::NCOL2], double& L, double& A) {
  const double2* Rr = reinterpret_cast<const double2*>(&pg.R[i][0]);
  L = 0.0;
  A = 0.0;
#pragma unroll
  for (int j = 0; j < BK::NCOL2; ++j) {
    const double2 c2 = Rr[j];
    if (2 * j >= 1 && 2 * j <= BK::NPAR) L = fma(c2.x, w[2 * j], L);
    else A = fma(c2.x, w[2 * j], A);
    if (2 * j + 1 >= 1 && 2 * j + 1 <= BK::NPAR) L = fma(c2.y, w[2 * j + 1], L);
    else A = fma(c2.y, w[2 * j + 1], A);
  }
}

// r_i(p) = E_i (R_i . w): the arithmetic every kernel of this library uses for the parametric shift of a row
template <class BK>
__device__ __forceinline__ double row_shift(const QpProg<BK>& pg, int i, const double (&w)[2 * BK::NCOL2]) {
  double L, A;
  row_LA<BK>(pg, i, w, L, A);
  return pg.Rs[i] * (L + A);
}

enum : int { kCertOk = 0, kCertUndecided = 2 };

struct Cert2Result {
  double x[2];      // scaled decision vector
  double obj;       // scaled objective at x: 0.5 x'Px + q'x + sum w_i |a_i x - kink_i|
  int verdict;      // kCertOk / kCertUndecided
  int nact;         // active rows of the guess (diagnostics)
};

struct NoHook {
  __device__ __forceinline__ void operator()() const {}
};

// hw[g] (g < G): the scenario's hint words without the flag bits; word g carries rows k*G + g at bits [3k, 3k+3).
// hook(): called once per row group of the feasibility pass (fast_step_kernel slips a few of its zero stores in there).
template <class BK, class Hook = NoHook>
__device__ __forceinline__ Cert2Result certify2(const QpProg<BK>& pg, const double (&w)[2 * BK::NCOL2], const double (&q)[BK::NZ],
                                                const unsigned long long (&hw)[BK::G], Hook hook = Hook()) {
  static_assert(BK::NZ == 2, "the closed-form certificate is for two decision variables");
  constexpr int G = BK::G, NCL = BK::NCL, NC = BK::NC, NK = BK::NK;
  constexpr unsigned long long M0 = 0x1249249249249249ull & ((NCL >= 21) ? ~0ull : ((1ull << (3 * NCL)) - 1ull));
  Cert2Result out;
  out.x[0] = out.x[1] = 0.0;
  out.obj = 0.0;
  // ---- the (at most two) active rows of the guess: codes 1 lower, 2 upper, 3 kink, 6 equality
  int na = 0, i0 = 0, i1 = 0;
  unsigned c0 = 0u, c1 = 0u;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const unsigned long long h = hw[g];
    const unsigned long long b0 = h & M0, b1 = (h >> 1) & M0, b2 = (h >> 2) & M0;
    unsigned long long act = (~b2 & (b1 | b0)) | (b2 & b1 & ~b0);
#pragma unroll
    for (int rep = 0; rep < 2; ++rep) {
      if (act != 0ull) {
        const int pos = __ffsll((long long)act) - 1;
        const int row = (pos / 3) * G + g;
        const unsigned c = (unsigned)(h >> pos) & 7u;
        if (na == 0) { i0 = row; c0 = c; }
        else if (na == 1) { i1 = row; c1 = c; }
        ++na;
        act &= act - 1ull;
      }
    }
    na += __popcll(act);
  }
  out.nact = na;
  bool bad = na > 2;
  // ---- |.|-cost rows (slots [0, NK)): linear cost terms of the rows off their kink; the subgradient interval of a
  // row whose active bound coincides with its kink relaxes that row's multiplier test by w
  double qt0 = q[0], qt1 = q[1];
  double rl0 = 0.0, rl1 = 0.0;
#pragma unroll
  for (int s = 0; s < NK; ++s) {
    const double wgt = pg.wabs[s];
    if (wgt > 0.0) {                                   // (uniform: the same program for the whole warp)
      const unsigned c = (unsigned)(hw[s % G] >> (3 * (s / G))) & 7u;
      const double r = row_shift<BK>(pg, s, w);
      const double kk = pg.kink0[s] + r;
      double sg = 0.0;
      if (c == 4u) sg = wgt;
      else if (c == 5u) sg = -wgt;
      else if (c == 1u || c == 2u || c == 6u) {
        const double b = (c == 2u ? pg.u0[s] : pg.l0[s]) + r;
        if (b > kk) sg = wgt;
        else if (b < kk) sg = -wgt;
        else { if (na >= 1 && i0 == s) rl0 = wgt; if (na >= 2 && i1 == s) rl1 = wgt; }
      } else if (c != 3u) bad = true;                  // a |.| row is on its kink, on a side of it, or on a bound
      qt0 = fma(sg, pg.A[s][0], qt0);
      qt1 = fma(sg, pg.A[s][1], qt1);
    }
  }
  // ---- closed-form KKT point
  const double P00 = pg.P[0][0], P01 = pg.P[1][0], P11 = pg.P[1][1];
  const double trP = P00 + P11;
  double x0 = 0.0, x1 = 0.0, la = 0.0, lb = 0.0;
  double a0 = 0.0, a1 = 0.0, b0_ = 0.0, b1_ = 0.0;
  // the bound or kink an active row's code pins it to.  The hint is caller memory, so a code that means nothing for its
  // row is rejected: 6 (equality) on a row whose bounds differ, 3 on a slot without a |.| cost, 1 / 2 on a missing bound
  // -- pinned anyway, such a row makes a feasible vertex pass every KKT test that follows (its multiplier sign is never
  // tested).  The predicates are those of active_code, so a hint the solver wrote itself always passes them.
  auto target = [&](int i, unsigned c, double& A0, double& A1) {
    const double r = row_shift<BK>(pg, i, w);
    const double lo = pg.l0[i] + r, hi = pg.u0[i] + r;
    A0 = pg.A[i][0];
    A1 = pg.A[i][1];
    if (c == 6u) bad = bad || (lo < hi);
    else if (c == 3u) bad = bad || !(i < NK && pg.wabs[i < NK ? i : 0] > 0.0);
    else if (c == 1u) bad = bad || !(lo > -INFINITY);
    else bad = bad || !(hi < INFINITY);
    return c == 2u ? hi : (c == 3u ? pg.kink0[i % NK] + r : lo);
  };
  if (na == 0) {
    const double det = P00 * P11 - P01 * P01;
    if (trP > 0.0 && det > 1e-12 * trP * trP) {
      const double id = 1.0 / det;
      x0 = -(P11 * qt0 - P01 * qt1) * id;
      x1 = -(P00 * qt1 - P01 * qt0) * id;
    } else if (trP > 1e-300) {                         // rank one: pseudo-inverse P / tr(P)^2
      const double it = 1.0 / (trP * trP);
      x0 = -(P00 * qt0 + P01 * qt1) * it;
      x1 = -(P01 * qt0 + P11 * qt1) * it;
    }
  } else if (na == 1) {
    const double t = target(i0, c0, a0, a1);
    const double n2 = fma(a0, a0, a1 * a1);
    const double in2 = 1.0 / n2;
    const double xn0 = a0 * (t * in2), xn1 = a1 * (t * in2);
    const double d0 = -a1, d1 = a0;                    // direction along the active row
    const double Pd0 = fma(P00, d0, P01 * d1), Pd1 = fma(P01, d0, P11 * d1);
    const double curv = fma(d0, Pd0, d1 * Pd1);
    const double g0 = fma(P00, xn0, fma(P01, xn1, qt0)), g1 = fma(P01, xn0, fma(P11, xn1, qt1));
    const double gd = fma(d0, g0, d1 * g1);
    const double s = (curv > 1e-12 * fmax(trP, 1e-300) * n2) ? -gd / curv : 0.0;
    x0 = fma(s, d0, xn0);
    x1 = fma(s, d1, xn1);
    const double r0 = fma(P00, x0, fma(P01, x1, qt0)), r1 = fma(P01, x0, fma(P11, x1, qt1));
    la = -fma(a0, r0, a1 * r1) * in2;
    bad = bad || !(n2 > 0.0);
  } else if (na == 2) {
    const double ta = target(i0, c0, a0, a1);
    const double tb = target(i1, c1, b0_, b1_);
    const double det = a0 * b1_ - a1 * b0_;
    const double na2 = fma(a0, a0, a1 * a1), nb2 = fma(b0_, b0_, b1_ * b1_);
    bad = bad || !(det * det > 1e-24 * na2 * nb2);     // (nearly) parallel rows: not a vertex
    const double id = 1.0 / det;
    x0 = (ta * b1_ - tb * a1) * id;
    x1 = (a0 * tb - b0_ * ta) * id;
    const double r0 = -fma(P00, x0, fma(P01, x1, qt0)), r1 = -fma(P01, x0, fma(P11, x1, qt1));
    la = (r0 * b1_ - r1 * b0_) * id;
    lb = (a0 * r1 - a1 * r0) * id;
  }
  // ---- stationarity  P x + qt + lam_a a + lam_b b = 0
  {
    const double s0 = fma(lb, b0_, fma(la, a0, fma(P00, x0, fma(P01, x1, qt0))));
    const double s1 = fma(lb, b1_, fma(la, a1, fma(P01, x0, fma(P11, x1, qt1))));
    const double lscale = fmax(1.0, fmax(fabs(la), fabs(lb)));
    const double qs = fmax(lscale, fmax(fabs(qt0), fabs(qt1)));
    bad = bad || !(fmax(fabs(s0), fabs(s1)) <= 1e-9 * qs);
    // ---- multiplier signs: upper bound lam >= 0, lower bound lam <= 0, kink |lam| <= w
    const double ltol = 1e-9 * lscale;
    if (na >= 1) {
      bad = bad || (c0 == 2u && la < -ltol - rl0) || (c0 == 1u && la > ltol + rl0);
      if (c0 == 3u) bad = bad || (fabs(la) > pg.wabs[i0 % NK] * (1.0 + 1e-9));
    }
    if (na >= 2) {
      bad = bad || (c1 == 2u && lb < -ltol - rl1) || (c1 == 1u && lb > ltol + rl1);
      if (c1 == 3u) bad = bad || (fabs(lb) > pg.wabs[i1 % NK] * (1.0 + 1e-9));
    }
  }
  // ---- every row: primal feasibility (a real loop: the body is 50 instructions, the unrolled form was 1,500 and
  // -- executed once per warp -- missed the instruction cache all the way: profiles/r2_fast_v0_*).  Rows without a lower
  // (upper) bound carry -inf (+inf), so one expression serves the three row classes.
  double viol = -INFINITY, scale = 1.0;
  {
    double L = 0.0, A = 0.0;
#pragma unroll 2
    for (int t = 0; t < pg.nc; ++t) {
      const int i = pg.grp_order[t];
      if (pg.grp_new[t]) {                                          // (uniform branch: the same program for the whole warp)
        row_LA<BK>(pg, i, w, L, A);
        hook();
      }
      const double r = pg.Rs[i] * fma(pg.grp_sgn[t], A, L);          // == row_shift(pg, i, w): sgn = -1 negates A exactly
      const double ax = fma(pg.A[i][1], x1, pg.A[i][0] * x0);
      viol = dmax(viol, dmax((pg.l0[i] + r) - ax, ax - (pg.u0[i] + r)));
      scale = dmax(scale, fabs(ax));
    }
  }
  // ---- |.| rows: cost and the side of the kink the guess assumed
  double kcost = 0.0;
#pragma unroll
  for (int s = 0; s < NK; ++s) {
    const double wgt = pg.wabs[s];
    if (wgt > 0.0) {
      const unsigned c = (unsigned)(hw[s % G] >> (3 * (s / G))) & 7u;
      const double kk = pg.kink0[s] + row_shift<BK>(pg, s, w);
      const double ax = fma(pg.A[s][1], x1, pg.A[s][0] * x0);
      kcost = fma(wgt, fabs(ax - kk), kcost);
      bad = bad || (c == 4u && !(ax > kk)) || (c == 5u && !(ax < kk));
    }
  }
  bad = bad || !(viol <= 1e-9 * scale) || !(x0 == x0) || !(x1 == x1);
  out.x[0] = x0;
  out.x[1] = x1;
  {
    const double px0 = fma(P00, x0, P01 * x1), px1 = fma(P01, x0, P11 * x1);
    double acc = kcost;
    acc = fma(fma(0.5, px0, q[0]), x0, acc);
    acc = fma(fma(0.5, px1, q[1]), x1, acc);
    out.obj = acc;
  }
  out.verdict = !bad ? kCertOk : kCertUndecided;
  return out;
}

// Singleton presolve, one thread per scenario (the lane-group form is tz_admm.cuh's singleton_infeasible): a row with one
// non-zero coefficient is a bound on one variable; inconsistent bounds on a variable decide infeasibility exactly.  Only
// evaluated for the scenarios whose hint did not certify.
template <class BK>
__device__ __forceinline__ bool singleton_infeasible2(const QpProg<BK>& pg, const double (&w)[2 * BK::NCOL2]) {
  static_assert(BK::NZ == 2, "two decision variables");
  double blo0 = -INFINITY, blo1 = -INFINITY, bhi0 = INFINITY, bhi1 = INFINITY;
#pragma unroll 1
  for (int i = 0; i < BK::NC; ++i) {
    const int sv = pg.sing_var[i];                     // (uniform: the same program for the whole warp)
    if (sv < 0) continue;
    const double r = row_shift<BK>(pg, i, w);
    const double inv = pg.sing_inv[i];
    const double ta = (pg.l0[i] + r) * inv, tb = (pg.u0[i] + r) * inv;
    const double l_ = inv > 0.0 ? ta : tb, h_ = inv > 0.0 ? tb : ta;
    if (sv == 0) { blo0 = dmax(blo0, l_); bhi0 = dmin(bhi0, h_); }
    else { blo1 = dmax(blo1, l_); bhi1 = dmin(bhi1, h_); }
  }
  const double sc0 = fmax(1.0, fmin(fabs(blo0), fabs(bhi0))), sc1 = fmax(1.0, fmin(fabs(blo1), fabs(bhi1)));
  return (blo0 - bhi0 > 1e-9 * sc0) || (blo1 - bhi1 > 1e-9 * sc1);
}

}  // namespace tz
