// big_step_kernel: the per-step program for the LARGER programs of the complexity sweep -- build_problem_simplified with
// horizons up to 10 (examples/1.double_integrator_computation_complexity.py:103-122, `-m stzddpc -ho 10 -k0 1`:
// 31 variables, ~120 rows) -- which exceed the register-resident lane-group buckets of step_kernel (NZ <= 12).
//
// Replaces the same reference calls as step_kernel (tzddpc/tzddpc.py:357-377 solve; examples/2.pulley_sim.py:90-96 update).
// One WARP per scenario, everything of the scenario in shared memory, run-time sizes (nz <= 32, nc <= 256):
//   * lane j owns variable j (x, q, the right-hand side of the KKT solve), rows are dealt out i = lane, lane + 32, ...;
//   * K = P + sigma I + A' diag(rho) A is built entry-parallel, factored in shared memory (column Cholesky), and solved with
//     column-oriented substitutions -- one shuffle broadcast per column, no reduction;
//   * the algorithm is tz_admm.cuh's: OSQP-style ADMM with the prox of the |.| cost rows, activity-driven rho switch,
//     the active-set KKT certificate (masked augmented-Lagrangian solve on the guessed active set, exact when it holds),
//     singleton presolve and the Farkas certificate for infeasibility, and the polish for residual exits.
// The program is read from global memory (an unpadded blob; it is shared by all warps and lives in L1 / L2): this path
// serves batch-1 sweeps and small batches, its speed is not the headline.
#include <cmath>
#include <new>
#include <vector>

#include "tz_big.h"

namespace tz {

namespace {

constexpr int kBigWarps = 4;
constexpr int kLP = 33;          // pitch of the factor in shared memory (conflict-free column access)

struct BigArgs {
  BigDev p;
  SolverParams sp;
  StepArgs a;
};

__device__ __forceinline__ double bmax(double a, double b) { return a > b ? a : b; }
__device__ __forceinline__ double wmaxr(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double wsumr(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// K = P + dadd I + sum_i wgt_i a_i a_i'  (lower triangle into L), then in-place column Cholesky; Ld = 1 / diag
__device__ void build_and_factor(const BigDev& B, const double* wgt, double dadd, double* L, double* Ld, int lane) {
  const int nz = B.nz, nc = B.nc;
  const int ntri = nz * (nz + 1) / 2;
  for (int e = lane; e < ntri; e += 32) {
    int a = 0, rem = e;
    while (rem > a) { rem -= a + 1; ++a; }          // e = a (a + 1) / 2 + b, b <= a
    const int b = rem;
    double s = B.P[a * nz + b] + (a == b ? dadd : 0.0);
    for (int i = 0; i < nc; ++i) {
      const double wi = wgt[i];
      if (wi != 0.0) s = fma(wi * B.A[i * nz + a], B.A[i * nz + b], s);
    }
    L[a * kLP + b] = s;
  }
  __syncwarp();
  for (int j = 0; j < nz; ++j) {
    double d = L[j * kLP + j];
    for (int k = 0; k < j; ++k) d -= L[j * kLP + k] * L[j * kLP + k];
    const double inv = rsqrt(fmax(d, 1e-300));
    for (int i = j + 1 + lane; i < nz; i += 32) {
      double s = L[i * kLP + j];
      for (int k = 0; k < j; ++k) s -= L[i * kLP + k] * L[j * kLP + k];
      L[i * kLP + j] = s * inv;
    }
    if (lane == 0) Ld[j] = inv;
    __syncwarp();
  }
}

// solves L L' x = b; lane j holds b_j in, x_j out (nz <= 32)
__device__ __forceinline__ double chol_solve_w(const double* L, const double* Ld, int nz, double b, int lane) {
  for (int j = 0; j < nz; ++j) {
    const double bj = __shfl_sync(0xffffffffu, b, j) * Ld[j];
    if (lane == j) b = bj;
    else if (lane > j && lane < nz) b = fma(-L[lane * kLP + j], bj, b);
  }
  for (int j = nz - 1; j >= 0; --j) {
    const double bj = __shfl_sync(0xffffffffu, b, j) * Ld[j];
    if (lane == j) b = bj;
    else if (lane < j) b = fma(-L[j * kLP + lane], bj, b);
  }
  return b;
}

// per-warp scratch in shared memory
struct Scratch {
  double *L, *Ld, *xs, *z, *y, *lo, *hi, *kk, *rho, *t, *lam, *tgt, *ysave, *axb, *wv, *om;
  int* code;
};

__device__ __forceinline__ int row_code(double z, double lo, double hi, double wabs, double kk) {
  if (z <= lo) return lo < hi ? 1 : 6;
  if (z >= hi) return 2;
  if (wabs > 0.0) return z == kk ? 3 : (z > kk ? 4 : 5);
  return 0;
}

// active-set KKT certificate (tz_admm.cuh admm_certify, warp form).  x_j: the lane's iterate in, the certified point out.
// S.y: duals in (active rows), certified multipliers out.  Returns a warp-uniform flag.
__device__ bool certify_w(const BigDev& B, const Scratch& S, const double* q, int n_iter, double& xj, int lane) {
  const int nz = B.nz, nc = B.nc;
  const double delta = 1e-9, mu = 1e6;
  // decode: weights, targets, subgradients
  double qt = lane < nz ? q[lane] : 0.0;
  for (int i = 0; i < nc; ++i) {                      // (every lane walks all rows: qt_j needs A[i][j] of every |.| row)
    const int c = S.code[i];
    const double wgt = B.wabs[i];
    double sg = 0.0;
    if (wgt > 0.0) {
      if (c == 4) sg = wgt;
      else if (c == 5) sg = -wgt;
      else if (c == 1 || c == 2 || c == 6) {
        const double b = c == 2 ? S.hi[i] : S.lo[i];
        if (b > S.kk[i]) sg = wgt;
        else if (b < S.kk[i]) sg = -wgt;
      }
    }
    if (sg != 0.0 && lane < nz) qt = fma(sg, B.A[i * nz + lane], qt);
  }
  for (int i = lane; i < nc; i += 32) {
    const int c = S.code[i];
    const bool ia = (c >= 1 && c <= 3) || c == 6;
    S.t[i] = ia ? mu : 0.0;
    S.tgt[i] = c == 2 ? S.hi[i] : (c == 3 ? S.kk[i] : S.lo[i]);
    S.lam[i] = ia ? S.y[i] : 0.0;
    if (!ia) S.tgt[i] = 0.0;
  }
  __syncwarp();
  build_and_factor(B, S.t, delta, S.L, S.Ld, lane);
  double xk = xj, xprev = xj;
  for (int it = 0; it < n_iter; ++it) {
    xprev = xk;
    double rhs = lane < nz ? fma(delta, xk, -qt) : 0.0;
    if (lane < nz)
      for (int i = 0; i < nc; ++i)
        if (S.t[i] != 0.0) rhs = fma(B.A[i * nz + lane], fma(mu, S.tgt[i], -S.lam[i]), rhs);
    xk = chol_solve_w(S.L, S.Ld, nz, rhs, lane);
    if (lane < nz) S.xs[lane] = xk;
    __syncwarp();
    for (int i = lane; i < nc; i += 32) {
      if (S.t[i] != 0.0) {
        double ax = 0.0;
        for (int j = 0; j < nz; ++j) ax = fma(B.At[j * nc + i], S.xs[j], ax);
        S.lam[i] = fma(mu, ax - S.tgt[i], S.lam[i]);
      }
    }
    __syncwarp();
  }
  // KKT checks
  double scale = 1.0, lscale = 1.0, qs = lane < nz ? fabs(qt) : 0.0;
  for (int i = lane; i < nc; i += 32) {
    double ax = 0.0;
    for (int j = 0; j < nz; ++j) ax = fma(B.At[j * nc + i], S.xs[j], ax);
    S.axb[i] = ax;
    scale = fmax(scale, fabs(ax));
    lscale = fmax(lscale, fabs(S.lam[i]));
  }
  scale = wmaxr(scale);
  lscale = wmaxr(lscale);
  qs = fmax(wmaxr(qs), lscale);
  const double ptol = 1e-9 * scale, ltol = 1e-9 * lscale, etol = 1e-8 * scale;
  int bad = 0;
  for (int i = lane; i < nc; i += 32) {
    const double ax = S.axb[i];
    const int c = S.code[i];
    const double wgt = B.wabs[i];
    bad |= (S.lo[i] - ax > ptol) || (ax - S.hi[i] > ptol);
    if (S.t[i] != 0.0) {
      double rl = 0.0;
      if (wgt > 0.0 && (c == 1 || c == 2 || c == 6) && (c == 2 ? S.hi[i] : S.lo[i]) == S.kk[i]) rl = wgt;
      bad |= fabs(ax - S.tgt[i]) > etol;
      bad |= (c == 2) && (S.lam[i] < -ltol - rl);
      bad |= (c == 1) && (S.lam[i] > ltol + rl);
      bad |= (c == 3) && (fabs(S.lam[i]) > wgt * (1.0 + 1e-9));
    } else if (wgt > 0.0) {
      bad |= (c == 4) ? !(ax > S.kk[i]) : ((c == 5) ? !(ax < S.kk[i]) : 1);
    }
  }
  if (lane < nz) {
    bad |= !(delta * fabs(xprev - xk) <= 1e-9 * qs);
    bad |= !(xk == xk);
  }
  const bool ok = !__any_sync(0xffffffffu, bad != 0);
  if (ok) {
    xj = xk;
    for (int i = lane; i < nc; i += 32) S.y[i] = S.t[i] != 0.0 ? S.lam[i] : 0.0;
  }
  __syncwarp();
  return ok;
}

// PL: a plant per scenario (StepArgs::AB_true)
template <bool PL = false>
__global__ void __launch_bounds__(kBigWarps * 32) big_step_kernel(const BigArgs g) {
  extern __shared__ __align__(16) double smem_d[];
  const BigDev& B = g.p;
  const SolverParams& sp = g.sp;
  const StepArgs& a = g.a;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t s = (int64_t)blockIdx.x * kBigWarps + wib;
  if (s >= a.S) return;                                  // (whole warps: no CTA barrier below)
  const int nz = B.nz, nc = B.nc, npar = B.npar, ncol = B.ncol, n = B.n, m = B.m, nv = B.nv, nwc = 1 + nv + npar;
  const int64_t LD = a.ld;
  double* base = smem_d + (size_t)wib * B.scratch_doubles;
  Scratch S;
  S.L = base; base += 32 * kLP;
  S.Ld = base; base += 32;
  S.xs = base; base += 32;
  S.wv = base; base += (ncol + 1) & ~1;
  S.om = base; base += (nwc + 1) & ~1;
  S.z = base; base += nc; S.y = base; base += nc; S.lo = base; base += nc; S.hi = base; base += nc; S.kk = base; base += nc;
  S.rho = base; base += nc; S.t = base; base += nc; S.lam = base; base += nc; S.tgt = base; base += nc; S.ysave = base; base += nc;
  S.axb = base; base += nc;
  S.code = reinterpret_cast<int*>(base);

  // ---- parameters and the parametric data: w = [1 | p | |Bt p + gam|], bounds, q, c0, parameter-only rows
  bool finite = true;
  for (int j = lane; j < npar; j += 32) {
    const double v = j < n ? a.xbar0[(int64_t)j * LD + s] : a.e0[(int64_t)(j - n) * LD + s];
    S.wv[1 + j] = v;
    finite = finite && (fabs(v) < 1e300);
  }
  if (lane == 0) S.wv[0] = 1.0;
  finite = !__any_sync(0xffffffffu, !finite);
  __syncwarp();
  for (int i = lane; i < B.na; i += 32) {
    double acc = B.gam[i];
    for (int k = 0; k < npar; ++k) acc = fma(B.Bt[i * npar + k], S.wv[1 + k], acc);
    S.wv[1 + npar + i] = fabs(acc);
  }
  __syncwarp();
  for (int i = lane; i < nc; i += 32) {
    double r = 0.0;
    for (int j = 0; j < ncol; ++j) r = fma(B.R[i * ncol + j], S.wv[j], r);
    S.lo[i] = B.l0[i] + r;
    S.hi[i] = B.u0[i] + r;
    S.kk[i] = B.kink0[i] + r;
  }
  int pbad = 0;
  for (int i = lane; i < B.nchk; i += 32) {
    double r = 0.0;
    for (int j = 0; j < ncol; ++j) r = fma(B.Rchk[i * ncol + j], S.wv[j], r);
    pbad |= r > B.chk_tol[i];
  }
  const bool param_ok = !__any_sync(0xffffffffu, pbad != 0);
  double qj = 0.0;
  if (lane < nz) {
    qj = B.q0[lane];
    for (int k = 0; k < npar; ++k) qj = fma(B.Qp[lane * npar + k], S.wv[1 + k], qj);
  }
  double c0 = 0.0;
  {
    double part = 0.0;
    for (int j = lane; j < ncol; j += 32) part = fma(B.cc[j], S.wv[j], part);
    for (int i = lane; i < npar; i += 32) {
      double acc = 0.0;
      for (int j = 0; j < npar; ++j) acc = fma(B.CC2[i * npar + j], S.wv[1 + j], acc);
      part = fma(acc, S.wv[1 + i], part);
    }
    c0 = wsumr(part);
  }
  __shared__ double qsh[kBigWarps][32];
  qsh[wib][lane] = qj;
  __syncwarp();
  const double* q = qsh[wib];

  int status = TZ_STATUS_MAXITER, iters = 0;
  bool certified = false;
  double xj = 0.0;
  if (!finite) status = TZ_STATUS_NONFINITE;
  else if (!param_ok) status = TZ_STATUS_INFEASIBLE;
  else {
    // ---- singleton presolve: rows with one non-zero coefficient bound one variable
    {
      double blo = -INFINITY, bhi = INFINITY;               // lane j collects the bounds on x_j
      for (int i = 0; i < nc; ++i) {
        const int sv = B.sing_var[i];
        if (sv == lane) {
          const double inv = B.sing_inv[i];
          const double ta = S.lo[i] * inv, tb = S.hi[i] * inv;
          blo = fmax(blo, inv > 0.0 ? ta : tb);
          bhi = fmin(bhi, inv > 0.0 ? tb : ta);
        }
      }
      const double sc = fmax(1.0, fmin(fabs(blo), fabs(bhi)));
      if (__any_sync(0xffffffffu, lane < nz && blo - bhi > 1e-9 * sc)) status = TZ_STATUS_INFEASIBLE;
    }
    if (status != TZ_STATUS_INFEASIBLE) {
      // ---- ADMM
      const double alpha = sp.alpha, sigma = sp.sigma;
      const double rho_act = sp.rho * sp.rho_act, rho_in = sp.rho * sp.rho_inact;
      for (int i = lane; i < nc; i += 32) {
        S.rho[i] = sp.rho;
        S.y[i] = 0.0;
        S.z[i] = fmin(fmax(0.0, S.lo[i]), S.hi[i]);
        S.ysave[i] = 0.0;
        S.code[i] = 0;
      }
      __syncwarp();
      build_and_factor(B, S.rho, sigma, S.L, S.Ld, lane);
      double qn = wmaxr(lane < nz ? fabs(qj) : 0.0);
      int next_upd = 2, gap = 2, next_cert = sp.cert_first > 0 ? sp.cert_first : sp.max_iter + 1, cert_gap = 2;
      const int check_every = sp.check_every > 0 ? sp.check_every : 1;
      int until_check = check_every;
      bool have_prev = false, switched = false, done = false;
      for (int it = 1; it <= sp.max_iter && !done; ++it) {
        for (int i = lane; i < nc; i += 32) S.t[i] = fma(S.rho[i], S.z[i], -S.y[i]);
        __syncwarp();
        double rhs = 0.0;
        if (lane < nz) {
          rhs = fma(sigma, xj, -qj);
          for (int i = 0; i < nc; ++i) rhs = fma(B.A[i * nz + lane], S.t[i], rhs);
        }
        const double xt = chol_solve_w(S.L, S.Ld, nz, rhs, lane);
        if (lane < nz) S.xs[lane] = xt;
        __syncwarp();
        for (int i = lane; i < nc; i += 32) {
          double ax = 0.0;
          for (int j = 0; j < nz; ++j) ax = fma(B.At[j * nc + i], S.xs[j], ax);
          const double zr = fma(alpha, ax, (1.0 - alpha) * S.z[i]);
          const double irho = 1.0 / S.rho[i];
          const double u = fma(S.y[i], irho, zr);
          double pr = u;
          const double wgt = B.wabs[i];
          if (wgt > 0.0) {
            const double d = u - S.kk[i];
            pr = S.kk[i] + copysign(bmax(fabs(d) - wgt * irho, 0.0), d);
          }
          const double zn = fmin(fmax(pr, S.lo[i]), S.hi[i]);
          S.y[i] = S.rho[i] * (u - zn);
          S.z[i] = zn;
        }
        xj = fma(alpha, xt, (1.0 - alpha) * xj);
        iters = it;
        __syncwarp();
        // ---- active-set certificate
        if (it == next_cert) {
          next_cert += cert_gap;
          cert_gap = (cert_gap * 3 + 1) / 2;
          for (int i = lane; i < nc; i += 32) S.code[i] = row_code(S.z[i], S.lo[i], S.hi[i], B.wabs[i], S.kk[i]);
          __syncwarp();
          double xc = xj;
          if (certify_w(B, S, q, sp.polish > 0 ? sp.polish : 3, xc, lane)) {
            xj = xc;
            status = TZ_STATUS_OK;
            certified = true;
            done = true;
          } else {
            build_and_factor(B, S.rho, sigma, S.L, S.Ld, lane);      // (the certificate factored its own K into S.L)
          }
        }
        // ---- residuals, infeasibility certificate
        if (!done && ((--until_check == 0) || it == sp.max_iter)) {
          until_check = check_every;
          if (lane < nz) S.xs[lane] = xj;
          __syncwarp();
          double rp = 0.0, pn = 0.0, dyn = 0.0, supp = 0.0, dyinf = 0.0;
          for (int i = lane; i < nc; i += 32) {
            double ax = 0.0;
            for (int j = 0; j < nz; ++j) ax = fma(B.At[j * nc + i], S.xs[j], ax);
            rp = fmax(rp, fabs(ax - S.z[i]));
            pn = fmax(pn, fmax(fabs(ax), fabs(S.z[i])));
            const double dy = S.y[i] - S.ysave[i];
            S.ysave[i] = S.y[i];
            S.t[i] = dy;
            dyn = fmax(dyn, fabs(dy));
            if (dy > 0.0) { if (S.hi[i] < 1e300) supp = fma(S.hi[i], dy, supp); else dyinf = fmax(dyinf, dy); }
            if (dy < 0.0) { if (S.lo[i] > -1e300) supp = fma(S.lo[i], dy, supp); else dyinf = fmax(dyinf, -dy); }
          }
          rp = wmaxr(rp); pn = wmaxr(pn); dyn = wmaxr(dyn); dyinf = wmaxr(dyinf); supp = wsumr(supp);
          __syncwarp();
          double aty = 0.0, atdy = 0.0, px = 0.0;
          if (lane < nz) {
            for (int i = 0; i < nc; ++i) {
              aty = fma(B.A[i * nz + lane], S.y[i], aty);
              atdy = fma(B.A[i * nz + lane], S.t[i], atdy);
            }
            for (int b = 0; b < nz; ++b) px = fma(B.P[lane * nz + b], S.xs[b], px);
          }
          const double rd = wmaxr(lane < nz ? fabs(px + qj + aty) : 0.0);
          const double pxn = wmaxr(fabs(px)), atyn = wmaxr(fabs(aty)), atdyn = wmaxr(fabs(atdy));
          const double ep = sp.eps_abs + sp.eps_rel * pn, ed = sp.eps_abs + sp.eps_rel * fmax(fmax(pxn, atyn), qn);
          if (!(rp == rp) || !(rd == rd)) { status = TZ_STATUS_NONFINITE; done = true; }
          else if (rp <= ep && rd <= ed) { status = TZ_STATUS_OK; done = true; }
          else if (have_prev && dyn > 1e-12 && dyinf <= 1e-6 * dyn && atdyn <= 1e-6 * dyn && supp < -1e-6 * dyn) {
            status = TZ_STATUS_INFEASIBLE;          // Farkas certificate (OSQP, Banjac et al. 2019)
            done = true;
          }
          have_prev = true;
        }
        // ---- activity-driven rho switch on a geometric schedule
        if (!done && it == next_upd) {
          gap = (gap * 3 + 1) / 2;
          next_upd = it + gap;
          int changed = switched ? 0 : 1;
          for (int i = lane; i < nc; i += 32) {
            const int c = row_code(S.z[i], S.lo[i], S.hi[i], B.wabs[i], S.kk[i]);
            const bool on = c == 1 || c == 2 || c == 3 || c == 6;        // on a bound / on the kink
            const double rn = on ? rho_act : rho_in;
            changed |= rn != S.rho[i];
            S.t[i] = rn;
          }
          if (__any_sync(0xffffffffu, changed != 0)) {
            for (int i = lane; i < nc; i += 32) S.rho[i] = S.t[i];
            switched = true;
            __syncwarp();
            build_and_factor(B, S.rho, sigma, S.L, S.Ld, lane);
          }
        }
      }
      // ---- polish of a residual exit: certificate on the final active set (accepted only if it holds)
      if (!certified && (status == TZ_STATUS_OK || status == TZ_STATUS_MAXITER) && sp.polish) {
        for (int i = lane; i < nc; i += 32) S.code[i] = row_code(S.z[i], S.lo[i], S.hi[i], B.wabs[i], S.kk[i]);
        __syncwarp();
        double xc = xj;
        if (certify_w(B, S, q, sp.polish, xc, lane)) { xj = xc; status = TZ_STATUS_OK; certified = true; }
      }
    }
  }
  const bool good = status == TZ_STATUS_OK || status == TZ_STATUS_MAXITER;
  // ---- objective value, outputs
  if (lane < nz) S.xs[lane] = xj;
  __syncwarp();
  double cost = NAN;
  if (good) {
    double part = 0.0;
    for (int i = lane; i < nc; i += 32) {
      const double wgt = B.wabs[i];
      if (wgt > 0.0) {
        double ax = 0.0;
        for (int j = 0; j < nz; ++j) ax = fma(B.At[j * nc + i], S.xs[j], ax);
        part = fma(wgt, fabs(ax - S.kk[i]), part);
      }
    }
    if (lane < nz) {
      double px = 0.0;
      for (int b = 0; b < nz; ++b) px = fma(B.P[lane * nz + b], S.xs[b], px);
      part = fma(fma(0.5, px, qj), xj, part);
    }
    cost = fma(wsumr(part), B.cinv, c0);
  } else if (status == TZ_STATUS_INFEASIBLE) {
    cost = INFINITY;
  }
  // om = [1 | v | p]
  if (lane == 0) S.om[0] = 1.0;
  for (int j = lane; j < nv; j += 32) S.om[1 + j] = good ? B.D[j] * S.xs[j] : NAN;
  for (int j = lane; j < npar; j += 32) S.om[1 + nv + j] = S.wv[1 + j];
  __syncwarp();
  if (lane == 0) {
    a.status[s] = status;
    if (a.iters) a.iters[s] = iters;
    if (a.cost) a.cost[s] = cost;
  }
  if (a.v)
    for (int j = lane; j < nv; j += 32) a.v[(int64_t)j * LD + s] = S.om[1 + j];
  const int nrows = (B.N + 1) * n;
  if (a.xbar_traj)
    for (int i = lane; i < nrows; i += 32) {
      double acc = 0.0;
      for (int j = 0; j < nwc; ++j) acc = fma(B.XB[i * nwc + j], S.om[j], acc);
      a.xbar_traj[(int64_t)i * LD + s] = acc;
    }
  if (a.ze1) {
    const int nent = n * (1 + B.g1);
    if (sp.tube_packed) {
      for (int k = lane; k < B.n_nz; k += 32) {
        const int e = B.tube_ent[k];
        double acc = 0.0;
        for (int t = B.ze1_ptr[e]; t < B.ze1_ptr[e + 1]; ++t) acc = fma(B.ze1_val[t], S.om[B.ze1_idx[t]], acc);
        a.ze1[(int64_t)k * LD + s] = acc;
      }
    } else {
      for (int e = lane; e < nent; e += 32) {
        double acc = 0.0;
        for (int t = B.ze1_ptr[e]; t < B.ze1_ptr[e + 1]; ++t) acc = fma(B.ze1_val[t], S.om[B.ze1_idx[t]], acc);
        a.ze1[(int64_t)e * LD + s] = acc;
      }
    }
  }
  // ---- closed-loop update (examples/2.pulley_sim.py:90-94): lane i owns state i
  if (a.x != nullptr) {
    double u[kMaxM];
    for (int j = 0; j < m; ++j) {
      double acc = S.om[1 + j];
      for (int i = 0; i < n; ++i) acc = fma(B.K[j * n + i], S.wv[1 + n + i], acc);
      u[j] = acc;
      if (a.u_out && lane == 0) a.u_out[(int64_t)j * LD + s] = good ? acc : NAN;
    }
    if (lane < n) {
      const int i = lane;
      double xn = a.noise ? a.noise[(int64_t)i * LD + s] : 0.0;
      if constexpr (PL) {
        const double* ab = a.AB_true + (int64_t)i * (n + m) * LD + s;
        for (int k = 0; k < n; ++k) xn = fma(ab[(int64_t)k * LD], a.x[(int64_t)k * LD + s], xn);
        for (int k = 0; k < m; ++k) xn = fma(ab[(int64_t)(n + k) * LD], u[k], xn);
      } else {
        for (int k = 0; k < n; ++k) xn = fma(a.A_true[i * n + k], a.x[(int64_t)k * LD + s], xn);
        for (int k = 0; k < m; ++k) xn = fma(a.B_true[i * m + k], u[k], xn);
      }
      double xb1 = 0.0;
      for (int j = 0; j < nwc; ++j) xb1 = fma(B.XB[(n + i) * nwc + j], S.om[j], xb1);
      double en = xn - xb1;
      if (!good) {
        const double xo = a.x[(int64_t)i * LD + s];
        const double xr = a.x_restart ? a.x_restart[(int64_t)i * LD + s] : xo;
        xn = xr;
        xb1 = a.x_restart ? xr : S.wv[1 + i];
        en = a.x_restart ? 0.0 : S.wv[1 + n + i];
      }
      S.t[i] = xn;                                  // (all lanes have read the old x through the barrier below)
      S.lam[i] = xb1;
      S.tgt[i] = en;
    }
    __syncwarp();
    if (lane < n) {
      a.x[(int64_t)lane * LD + s] = S.t[lane];
      a.xbar[(int64_t)lane * LD + s] = S.lam[lane];
      a.e[(int64_t)lane * LD + s] = S.tgt[lane];
    }
    if (a.stats != nullptr) {
      double nrm2 = 0.0;
      for (int i = 0; i < n; ++i) nrm2 = fma(S.t[i], S.t[i], nrm2);
      if (lane == 0) {
        if (good) { atomicAdd(a.stats + 0, sqrt(nrm2)); atomicAdd(a.stats + 1, nrm2); atomicAdd(a.stats + 2, cost); }
        if (status == TZ_STATUS_INFEASIBLE) atomicAdd(a.stats + 3, 1.0);
        if (status == TZ_STATUS_MAXITER) atomicAdd(a.stats + 4, 1.0);
        atomicAdd(a.stats + 5, (double)iters);
        if (status == TZ_STATUS_NONFINITE) atomicAdd(a.stats + 6, 1.0);
        atomicAdd(a.stats + 7, 1.0);
      }
    }
  }
}

}  // namespace

// ---- host side: the blob ---------------------------------------------------------------------------------------------
bool big_fits(const TzProgramDesc& d) {
  return d.nz <= 32 && d.nc <= 256 && d.npar <= 16 && d.na <= 64 && d.n <= kMaxN && d.m <= kMaxM;
}

int big_create(const TzProgramDesc& d, BigProgram** out) {
  BigProgram* bp = new (std::nothrow) BigProgram();
  if (!bp) return fail(TZ_ENOMEM, "out of host memory");
  const int nz = d.nz, nc = d.nc, npar = d.npar, na = d.na, ncol = 1 + npar + na, n = d.n, m = d.m, nv = d.nv, nwc = 1 + nv + npar;
  const int nent = n * (1 + d.g1), nrows = (d.horizon + 1) * n;
  std::vector<double> hd;
  std::vector<int32_t> hi;
  auto pushd = [&](size_t cnt) { const size_t o = hd.size(); hd.resize(o + cnt, 0.0); return o; };
  auto pushi = [&](size_t cnt) { const size_t o = hi.size(); hi.resize(o + cnt, 0); return o; };
  const size_t oP = pushd((size_t)nz * nz), oA = pushd((size_t)nc * nz), oAt = pushd((size_t)nz * nc), ol0 = pushd(nc), ou0 = pushd(nc),
               okink = pushd(nc), owabs = pushd(nc), oR = pushd((size_t)nc * ncol), oq0 = pushd(nz), oQp = pushd((size_t)nz * npar),
               oBt = pushd((size_t)na * npar), ogam = pushd(na), oRchk = pushd((size_t)d.nchk * ncol), otol = pushd(d.nchk), occ = pushd(ncol),
               oCC2 = pushd((size_t)npar * npar), oD = pushd(nz), osinv = pushd(nc), oXB = pushd((size_t)nrows * nwc), oK = pushd((size_t)m * n),
               oval = pushd(d.nterms);
  const size_t osv = pushi(nc), optr = pushi(nent + 1), oidx = pushi(d.nterms);
  for (int a = 0; a < nz; ++a) {
    hd[oD + a] = d.D[a];
    hd[oq0 + a] = d.c * d.D[a] * d.q0[a];
    for (int b = 0; b < nz; ++b) hd[oP + (size_t)a * nz + b] = d.c * d.D[a] * d.P[a * nz + b] * d.D[b];
    for (int k = 0; k < npar; ++k) hd[oQp + (size_t)a * npar + k] = d.c * d.D[a] * d.Qp[a * npar + k];
  }
  for (int i = 0; i < nc; ++i) {
    const double E = d.E[i];
    int nnz = 0, where = -1;
    for (int a = 0; a < nz; ++a) {
      const double v = E * d.A[i * nz + a] * d.D[a];
      hd[oA + (size_t)i * nz + a] = v;
      hd[oAt + (size_t)a * nc + i] = v;
      if (v != 0.0) { ++nnz; where = a; }
    }
    hi[osv + i] = nnz == 1 ? where : -1;
    hd[osinv + i] = nnz == 1 ? 1.0 / hd[oA + (size_t)i * nz + where] : 0.0;
    hd[ol0 + i] = E * d.l0[i];
    hd[ou0 + i] = E * d.u0[i];
    hd[okink + i] = E * d.kink0[i];
    hd[owabs + i] = d.wabs[i] > 0.0 ? d.c * d.wabs[i] / E : 0.0;
    for (int j = 0; j < ncol; ++j) hd[oR + (size_t)i * ncol + j] = E * d.R[i * ncol + j];
  }
  for (int i = 0; i < na; ++i) {
    hd[ogam + i] = d.gam[i];
    for (int k = 0; k < npar; ++k) hd[oBt + (size_t)i * npar + k] = d.Bt[i * npar + k];
  }
  for (int i = 0; i < d.nchk; ++i) {
    for (int j = 0; j < ncol; ++j) hd[oRchk + (size_t)i * ncol + j] = d.Rchk[i * ncol + j];
    hd[otol + i] = 1e-9 * std::fmax(1.0, std::fabs(d.Rchk[i * ncol]));
  }
  for (int j = 0; j < ncol; ++j) hd[occ + j] = d.cc[j];
  for (int i = 0; i < npar * npar; ++i) hd[oCC2 + i] = d.CC2[i];
  for (int i = 0; i < nrows * nwc; ++i) hd[oXB + i] = d.XB[i];
  for (int i = 0; i < m * n; ++i) hd[oK + i] = d.K[i];
  for (int t = 0; t < d.nterms; ++t) {
    if (d.ze1_idx[t] < 0 || d.ze1_idx[t] >= nwc) { delete bp; return fail(TZ_EINVAL, "ze1_idx[%d] out of range", t); }
    hd[oval + t] = d.ze1_val[t];
    hi[oidx + t] = d.ze1_idx[t];
  }
  for (int e = 0; e <= nent; ++e) hi[optr + e] = d.ze1_ptr[e];
  for (int e = 0; e < nent; ++e)
    if (d.ze1_ptr[e + 1] > d.ze1_ptr[e]) bp->tube_ent.push_back(e);
  const size_t oent = pushi(bp->tube_ent.size());
  for (size_t k = 0; k < bp->tube_ent.size(); ++k) hi[oent + k] = bp->tube_ent[k];
  cudaError_t err = cudaMalloc(&bp->dbl_dev, hd.size() * sizeof(double));
  if (err == cudaSuccess) err = cudaMemcpy(bp->dbl_dev, hd.data(), hd.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMalloc(&bp->int_dev, hi.size() * sizeof(int32_t));
  if (err == cudaSuccess) err = cudaMemcpy(bp->int_dev, hi.data(), hi.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    big_destroy(bp);
    return fail(TZ_ECUDA, "big program upload: %s", cudaGetErrorString(err));
  }
  const double* D0 = bp->dbl_dev;
  const int32_t* I0 = bp->int_dev;
  BigDev& B = bp->dev;
  B.nz = nz; B.nc = nc; B.npar = npar; B.na = na; B.ncol = ncol; B.nchk = d.nchk; B.n = n; B.m = m; B.N = d.horizon; B.nv = nv; B.g1 = d.g1;
  B.n_nz = (int)bp->tube_ent.size();
  B.cinv = 1.0 / d.c;
  B.P = D0 + oP; B.A = D0 + oA; B.At = D0 + oAt; B.l0 = D0 + ol0; B.u0 = D0 + ou0; B.kink0 = D0 + okink; B.wabs = D0 + owabs; B.R = D0 + oR;
  B.q0 = D0 + oq0; B.Qp = D0 + oQp; B.Bt = D0 + oBt; B.gam = D0 + ogam; B.Rchk = D0 + oRchk; B.chk_tol = D0 + otol; B.cc = D0 + occ;
  B.CC2 = D0 + oCC2; B.D = D0 + oD; B.sing_inv = D0 + osinv; B.XB = D0 + oXB; B.K = D0 + oK; B.ze1_val = D0 + oval;
  B.sing_var = I0 + osv; B.ze1_ptr = I0 + optr; B.ze1_idx = I0 + oidx; B.tube_ent = I0 + oent;
  const size_t sd = (size_t)32 * kLP + 32 + 32 + ((ncol + 1) & ~1) + ((nwc + 1) & ~1) + (size_t)11 * nc + (size_t)(nc + 1) / 2 + 2;
  B.scratch_doubles = (int)((sd + 1) & ~(size_t)1);
  *out = bp;
  return TZ_OK;
}

void big_destroy(BigProgram* bp) {
  if (!bp) return;
  if (bp->dbl_dev) cudaFree(bp->dbl_dev);
  if (bp->int_dev) cudaFree(bp->int_dev);
  delete bp;
}

int big_launch(const BigProgram* bp, const SolverParams& sp, const StepArgs& a, cudaStream_t st) {
  BigArgs g;
  g.p = bp->dev;
  g.sp = sp;
  g.a = a;
  const size_t smem = (size_t)kBigWarps * bp->dev.scratch_doubles * sizeof(double);
  if (smem > 200 * 1024) return fail(TZ_ERANGE, "program needs %zu bytes of shared memory per CTA", smem);
  const unsigned grid = (unsigned)((a.S + kBigWarps - 1) / kBigWarps);
  return with_plant(a, [&](auto pl) {
    constexpr auto kernel = big_step_kernel<decltype(pl)::value>;
    TZ_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, kBigWarps * 32, smem, st>>>(g);
    TZ_CUDA(cudaGetLastError());
    return TZ_OK;
  });
}

}  // namespace tz
