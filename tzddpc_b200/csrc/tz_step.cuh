// The fused per-step kernel of the TZDDPC hot path and its launcher, as templates over the kernel bucket.  Every
// bucket is instantiated in its own translation unit (tz_fused.cu: B0, tz_bucket*.cu: the larger ones) so that they
// compile in parallel.  See tz_fused.cu for the description of the kernel.
#pragma once
#include <atomic>
#include <cmath>
#include <new>
#include <type_traits>
#include <vector>

#include "tz_admm.cuh"
#include "tz_cert2.cuh"
#include "tz_param.cuh"

#define TZ_LIKELY(x) __builtin_expect(!!(x), 1)
#define TZ_UNLIKELY(x) __builtin_expect(!!(x), 0)

namespace tz {

// Run-time sized tables of a program, one device blob staged into shared memory by every CTA:
//   doubles: XB ((N+1)n x NW) | CZ (n x NW) | K (m x n) | nz_coef (n_nz)      [+ A_true, B_true appended in smem]
//   int32  : nz_ent (n_nz) | nz_idx (n_nz)
// XB / CZ columns and nz_idx address the per-scenario vector om (layout in Bucket: OM_*).
struct Aux {
  const double* tab;
  int n_dbl, n_int;                // sizes of the two parts
  int o_XB, o_CZ, o_K, o_coef;     // offsets (doubles)
  int o_ent, o_idx;                // offsets (int32, from the start of the int part)
  int o_tt;                        // (doubles, even) term table of fast_step_kernel: n_nz pairs (coef, bits of idx | ent << 32)
  int o_zrun, n_zrun;              // (doubles) zero runs of the dense Ze[1].Z between its non-zero entries: int32 pairs (first row, length)
  int zrun_split;                  // runs [0, zrun_split) hold about half of the zero entries (the two halves of a CTA share the zero-fill)
  int o_zrow, n_zrow_half;         // (doubles, even) the zero rows as a flat int32 list in two halves of n_zrow_half entries (a
                                   // multiple of 4: each half padded by repeating its last row), for 16-byte index loads
  int n_nz;                        // entries of Ze[1].Z that are not structurally zero (centre column included)
  int n, m, N, nv, g1;
};

struct StepArgs {
  int64_t S;                       // scenarios in this launch
  int64_t ld;                      // leading dimension of every SoA array (>= S)
  int vec2;                        // 1: S, ld even and every array 16-byte aligned -> two scenarios per lane in the output phase
  const double* xbar0;             // parameters (n x S); aliases xbar/e in closed loop
  const double* e0;
  double* x;                       // closed loop only (NULL = solve only)
  double* xbar;
  double* e;
  const double* noise;
  const double* x_restart;         // closed loop only: state an infeasible scenario restarts from (NULL: it keeps its state)
  const double* A_true;
  const double* B_true;
  double* cost;
  double* v;
  double* xbar_traj;
  double* ze1;
  double* u_out;
  int32_t* status;
  int32_t* iters;
  double* warm;
  double* stats;
  // explicit-instance mode (tz_qp_solve): q, l, u given, z / y returned
  const double* q_in;
  const double* l_in;
  const double* u_in;
  double* z_out;
  double* y_out;
  // deferred tiles (fast_step_kernel -> step_kernel): defer[0] = number of listed tiles, defer[1] = exit ticket of step_kernel's
  // CTAs (the last one zeroes both); defer_list[i] = index of a 16-scenario output tile.  list_mode: step_kernel walks the list
  int32_t* defer;
  int32_t* defer_list;
  int list_mode;
  // fused run (tz_closed_loop_run): nsteps > 1 closed-loop steps in one launch; noise and every per-step output then hold
  // nsteps consecutive blocks (step-major), x_hist (nsteps x n x ld, or NULL) receives the state after every step
  int nsteps;
  double* x_hist;
  double* xbar_hist;
  double* e_hist;
  // plant per scenario (tz_closed_loop_*_plants): [A_true B_true] of scenario s, entry (i, k), at AB_true[(i (n+m) + k) ld + s];
  // NULL: A_true / B_true, shared by the whole batch.  Selects the kernel instantiation (template parameter PL) on the host.
  const double* AB_true;
};

// Calls f(std::true_type) for a plant per scenario (a.AB_true != NULL), f(std::false_type) for a plant shared by the batch:
// the launchers pick the kernel instantiation of template parameter PL = decltype(arg)::value.
template <class F>
int with_plant(const StepArgs& a, F&& f) {
  return a.AB_true != nullptr ? f(std::true_type{}) : f(std::false_type{});
}

// Shared-memory image of one CTA: the program (read-only after staging) and, per warp, the
// exchange buffers between the solve phase and the output phase of a tile.
template <class BK>
struct alignas(16) WarpBuf {
  double pre[2][BK::PRE_ROWS][BK::SPO];  // cp.async double buffer: rows [xbar0 | e0 | x | noise] (n each) of this / the next output tile
  double om[BK::KOM][BK::SPO];     // [1 | v | xbar0 | e0 | centre of Ze[1] | x+] per scenario of the warp's output tile
  double ysave[BK::NCL][32];       // duals at the previous residual check (certificate of infeasibility)
  double cost[BK::SPO];
  double stacc[TZ_NSTATS][BK::SPO];   // closed-loop statistics of this warp's tiles, reduced once at the end of the kernel
  int status[BK::SPO];
  int iters[BK::SPO];
};
template <class BK>
struct alignas(16) Smem {
  double Aa[BK::NC][BK::NZ];       // alpha * A (alpha is a solver option, so this is built when the program is staged)
  QpProg<BK> pg;
  WarpBuf<BK> wb[BK::WPB];
};

// ---- W scenarios per lane (1: scalar accesses, 2: 16-byte accesses) ----------------------------
template <int W> struct Vec;
template <> struct Vec<1> { double a; };
template <> struct Vec<2> { double a, b; };
__device__ __forceinline__ Vec<1> vld(const double* p, Vec<1>*) { return Vec<1>{*p}; }
__device__ __forceinline__ Vec<2> vld(const double* p, Vec<2>*) { const double2 t = *reinterpret_cast<const double2*>(p); return Vec<2>{t.x, t.y}; }
__device__ __forceinline__ void vst(double* p, Vec<1> v) { *p = v.a; }
__device__ __forceinline__ void vst(double* p, Vec<2> v) { *reinterpret_cast<double2*>(p) = make_double2(v.a, v.b); }
__device__ __forceinline__ void vstcs(double* p, Vec<1> v) { __stcs(p, v.a); }
__device__ __forceinline__ void vstcs(double* p, Vec<2> v) { __stcs(reinterpret_cast<double2*>(p), make_double2(v.a, v.b)); }
__device__ __forceinline__ Vec<1> vfma(double c, Vec<1> x, Vec<1> acc) { return Vec<1>{fma(c, x.a, acc.a)}; }
__device__ __forceinline__ Vec<2> vfma(double c, Vec<2> x, Vec<2> acc) { return Vec<2>{fma(c, x.a, acc.a), fma(c, x.b, acc.b)}; }
__device__ __forceinline__ Vec<1> vfma2(Vec<1> c, Vec<1> x, Vec<1> acc) { return Vec<1>{fma(c.a, x.a, acc.a)}; }
__device__ __forceinline__ Vec<2> vfma2(Vec<2> c, Vec<2> x, Vec<2> acc) { return Vec<2>{fma(c.a, x.a, acc.a), fma(c.b, x.b, acc.b)}; }
__device__ __forceinline__ Vec<1> vmul(double c, Vec<1> x) { return Vec<1>{c * x.a}; }
__device__ __forceinline__ Vec<2> vmul(double c, Vec<2> x) { return Vec<2>{c * x.a, c * x.b}; }
__device__ __forceinline__ Vec<1> vsub(Vec<1> x, Vec<1> y) { return Vec<1>{x.a - y.a}; }
__device__ __forceinline__ Vec<2> vsub(Vec<2> x, Vec<2> y) { return Vec<2>{x.a - y.a, x.b - y.b}; }
__device__ __forceinline__ Vec<1> vzero(Vec<1>*) { return Vec<1>{0.0}; }
__device__ __forceinline__ Vec<2> vzero(Vec<2>*) { return Vec<2>{0.0, 0.0}; }
__device__ __forceinline__ Vec<1> vsel(const bool* g, Vec<1> x, double other) { return Vec<1>{g[0] ? x.a : other}; }
__device__ __forceinline__ Vec<2> vsel(const bool* g, Vec<2> x, double other) { return Vec<2>{g[0] ? x.a : other, g[1] ? x.b : other}; }
__device__ __forceinline__ double vget(Vec<1> x, int) { return x.a; }
__device__ __forceinline__ double vget(Vec<2> x, int i) { return i == 0 ? x.a : x.b; }

// ---- cp.async prefetch of the per-scenario inputs of an output tile (hides the DRAM latency of the only loads of the step)
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

template <class BK>
__device__ __forceinline__ void prefetch_inputs(double (*dst)[BK::SPO], const StepArgs& a, const double* hint, int n,
                                                int64_t otile, int lane) {
  constexpr int SPO = BK::SPO;
  const double* src[4] = {a.xbar0, a.e0, a.x, a.noise};
  const int64_t s0 = otile * SPO;
  const int narr = a.x != nullptr ? 4 : 2;
  if (hint != nullptr) {                                 // active-set hint words: G rows behind the 4n input rows
    if (a.vec2) {
      for (int c = lane; c < BK::G * (SPO / 2); c += 32) {
        const int row = c / (SPO / 2), ch = c - row * (SPO / 2);
        const int64_t s = s0 + 2 * ch;
        if (s < a.S) cp_async16(&dst[4 * n + row][2 * ch], hint + (int64_t)row * a.ld + s);
      }
    } else {
      for (int c = lane; c < BK::G * SPO; c += 32) {
        const int row = c / SPO, ch = c - row * SPO;
        const int64_t s = s0 + ch;
        if (s < a.S) cp_async8(&dst[4 * n + row][ch], hint + (int64_t)row * a.ld + s);
      }
    }
  }
  if (a.vec2) {
    constexpr int CPR = SPO / 2;                        // 16-byte chunks per row
    const int total = narr * n * CPR;
    for (int c = lane; c < total; c += 32) {
      const int row = c / CPR, ch = c - row * CPR, arr = row / n, r = row - arr * n;
      const int64_t s = s0 + 2 * ch;
      if (src[arr] != nullptr && s < a.S) cp_async16(&dst[row][2 * ch], src[arr] + (int64_t)r * a.ld + s);
    }
  } else {
    const int total = narr * n * SPO;
    for (int c = lane; c < total; c += 32) {
      const int row = c / SPO, ch = c - row * SPO, arr = row / n, r = row - arr * n;
      const int64_t s = s0 + ch;
      if (src[arr] != nullptr && s < a.S) cp_async8(&dst[row][ch], src[arr] + (int64_t)r * a.ld + s);
    }
  }
  cp_async_commit();
}

// Zero-fill of the dense Ze[1].Z block of one output tile (88 % of its entries are structural zeros, but the reference
// returns the matrix dense, examples/2.pulley_sim.py:96).  It depends on nothing the solve computes, so half of the
// warps issue it BEFORE solving their tile and the other half after: the stores of one half drain while the other half
// computes (all warps in lock step would alternate between an idle DRAM and a saturated one: profiles/r1_v8).
template <class BK, int W>
__device__ __forceinline__ void zero_fill(const Aux& ax, const StepArgs& a, int64_t tile, int lane) {
  constexpr int SPW = BK::SPO, NGRP = SPW / W, NSL = 32 / NGRP;
  using V = Vec<W>;
  V* const vt = nullptr;
  const int pc = lane % NGRP, slice = lane / NGRP;
  const int64_t so = tile * SPW + pc * W;
  if (so >= a.S) return;
  const int64_t LD = a.ld;
  const int nent = ax.n * (1 + ax.g1);
  const int64_t stepb = (int64_t)NSL * LD;
  double* ptr = a.ze1 + so + (int64_t)slice * LD;
  const V z0 = vzero(vt);
  // (a down-counter: with the trip count as loop bound the compiler spilled it and re-loaded it from local memory in
  // every iteration, behind the stores in the same LSU queue -- 20 % of all stall samples in profiles/r1_v6)
#pragma unroll 4
  for (int cnt = (nent - slice + NSL - 1) / NSL; cnt > 0; --cnt, ptr += stepb) vstcs(ptr, z0);
}

// Output phase of one output tile (SPO >= 16 consecutive scenarios = TPO solve tiles): lane -> (W consecutive
// scenarios, slice); one store instruction of the warp covers NSL entries x SPO scenarios = NSL runs of SPO*8 >= 128
// contiguous bytes (full lines) of the scenario-fastest arrays.
template <class BK, int W, bool PL>
__device__ __forceinline__ void output_phase(WarpBuf<BK>& wb, const double (*pre)[BK::SPO], const Aux& ax, const StepArgs& a,
                                             const double* __restrict__ tabd, const int* __restrict__ tabi, int64_t tile, int lane,
                                             bool zero_done, bool packed) {
  constexpr int SPW = BK::SPO, NW = BK::NW, NGRP = SPW / W, NSL = 32 / NGRP;
  using V = Vec<W>;
  V* const vt = nullptr;
  const int pc = lane % NGRP, slice = lane / NGRP, sc0 = pc * W;
  const int64_t so = tile * SPW + sc0;
  const int64_t LD = a.ld;
  const int n = ax.n, m = ax.m, nv = ax.nv;
  const double* sXB = tabd + ax.o_XB;
  int stt[W];
  bool olive[W], ogood[W];
  bool any_live = false, all_good = true;
#pragma unroll
  for (int t = 0; t < W; ++t) {
    stt[t] = wb.status[sc0 + t];
    olive[t] = stt[t] >= 0;
    ogood[t] = stt[t] == TZ_STATUS_OK || stt[t] == TZ_STATUS_MAXITER;
    any_live = any_live || olive[t];
    all_good = all_good && ogood[t];
  }
  // (vector path: S is even, so the scenarios of a pair are live together)
  auto om = [&](int j) { return vld(&wb.om[j][sc0], vt); };
  // ---- Ze[1].Z at the optimum (examples/2.pulley_sim.py:96: Zek.Z.value), dense n x (1+g1): zero-fill, then overwrite
  // the ~12 % entries that are not structurally zero (both writes merge in L2 before reaching HBM).  The warp barrier
  // between the two sits outside every lane-dependent branch (tiles at the end of a batch have dead lanes).
  if (a.ze1 && packed) {
    // packed tube: row i of the output is entry ent[i] of Ze[1].Z (tz_program_tube_pattern); structural zeros are not stored
    if (any_live) {
      double* base = a.ze1 + so;
      const double* coef = tabd + ax.o_coef;
      const int* idx = tabi + ax.o_idx;
#pragma unroll 4
      for (int i = slice; i < ax.n_nz; i += NSL) vstcs(base + (int64_t)i * LD, vmul(coef[i], om(idx[i])));
    }
  } else if (a.ze1) {
    if (any_live && !zero_done) zero_fill<BK, W>(ax, a, tile, lane);
    __syncwarp();
    if (any_live) {
      double* base = a.ze1 + so;
      const double* coef = tabd + ax.o_coef;
      const int* ent = tabi + ax.o_ent;
      const int* idx = tabi + ax.o_idx;
#pragma unroll 4
      for (int i = slice; i < ax.n_nz; i += NSL) vstcs(base + (int64_t)ent[i] * LD, vmul(coef[i], om(idx[i])));
    }
  }
  if (any_live) {
    // ---- nominal trajectory xbar_0..xbar_N = XB om  (tzddpc/tzddpc.py:166-170)
    if (a.xbar_traj) {
      const int nrows = (ax.N + 1) * n;
      for (int i = slice; i < nrows; i += NSL) {
        const double* row = sXB + i * NW;
        V acc = vzero(vt);
#pragma unroll
        for (int j = 0; j < NW; ++j) acc = vfma(row[j], om(j), acc);
        vst(a.xbar_traj + (int64_t)i * LD + so, acc);
      }
    }
    if (a.v)
      for (int j = slice; j < nv; j += NSL) vst(a.v + (int64_t)j * LD + so, om(BK::OM_V + j));
    if (slice == 0) {
#pragma unroll
      for (int t = 0; t < W; ++t) {
        if (olive[t]) {
          if (a.status) a.status[so + t] = stt[t];
          if (a.iters) a.iters[so + t] = wb.iters[sc0 + t];
          if (a.cost) a.cost[so + t] = wb.cost[sc0 + t];
        }
      }
    }
  }
  // ---- closed-loop update (examples/2.pulley_sim.py:90-94): row i of the update by slice i
  if (a.x != nullptr) {
    const double* sK = tabd + ax.o_K;
    const double* sA = tabd + ax.n_dbl;
    const double* sB = sA + n * n;
    if (any_live) {
      V us[kMaxM];
#pragma unroll
      for (int j = 0; j < kMaxM; ++j) {
        V acc = vzero(vt);
        if (j < m) {
          acc = om(BK::OM_V + j);                                              // v[0]
          for (int i = 0; i < n; ++i) acc = vfma(sK[j * n + i], om(BK::OM_P + BK::NPAR / 2 + i), acc);
          if (a.u_out && slice == 0) vst(a.u_out + (int64_t)j * LD + so, vsel(ogood, acc, NAN));
        }
        us[j] = acc;                                                           // u = K e + v[0]
      }
      for (int i = slice; i < n; i += NSL) {
        V acc = a.noise ? vld(&pre[3 * n + i][sc0], vt) : vzero(vt);
        if constexpr (PL) {
          // this scenario's plant, row i of [A_true B_true]: the same W-scenario vector loads as x (vec2_ok checks AB_true)
          const double* ab = a.AB_true + (int64_t)i * (n + m) * LD + so;
          for (int k = 0; k < n; ++k) acc = vfma2(vld(ab + (int64_t)k * LD, vt), vld(&pre[2 * n + k][sc0], vt), acc);
#pragma unroll
          for (int k = 0; k < kMaxM; ++k)
            if (k < m) acc = vfma2(vld(ab + (int64_t)(n + k) * LD, vt), us[k], acc);
        } else {
          for (int k = 0; k < n; ++k) acc = vfma(sA[i * n + k], vld(&pre[2 * n + k][sc0], vt), acc);
#pragma unroll
          for (int k = 0; k < kMaxM; ++k)
            if (k < m) acc = vfma(sB[i * m + k], us[k], acc);
        }
        const double* row = sXB + (n + i) * NW;                                // xbar+ = xbar_traj[1]
        V xb1 = vzero(vt);
#pragma unroll
        for (int j = 0; j < NW; ++j) xb1 = vfma(row[j], om(j), xb1);
        V en = vsub(acc, xb1);                                                 // e+ = x+ - xbar+
        if (TZ_UNLIKELY(!all_good)) {
          // a scenario whose step failed keeps its state, or -- the reference raises and the run ends
          // (tzddpc/tzddpc.py:374-375) -- starts a new run from x_restart: x = xbar = x_restart, e = 0
          const V xo = vld(&pre[2 * n + i][sc0], vt);
          const V xbo = om(BK::OM_P + i), eo = om(BK::OM_P + BK::NPAR / 2 + i);
          const V xr = a.x_restart ? vld(a.x_restart + (int64_t)i * LD + so, vt) : xo;
          double xa[W], ba[W], ea[W];
#pragma unroll
          for (int t = 0; t < W; ++t) {
            xa[t] = ogood[t] ? vget(acc, t) : vget(xr, t);
            ba[t] = ogood[t] ? vget(xb1, t) : (a.x_restart ? vget(xr, t) : vget(xbo, t));
            ea[t] = ogood[t] ? vget(en, t) : (a.x_restart ? 0.0 : vget(eo, t));
          }
          if constexpr (W == 1) { acc = V{xa[0]}; xb1 = V{ba[0]}; en = V{ea[0]}; }
          else { acc = V{xa[0], xa[1]}; xb1 = V{ba[0], ba[1]}; en = V{ea[0], ea[1]}; }
        }
        vst(&wb.om[BK::OM_XP + i][sc0], acc);
        vst(a.x + (int64_t)i * LD + so, acc);                                  // x+ = A x + B u + w
        if (a.x_hist != nullptr) vst(a.x_hist + (int64_t)i * LD + so, acc);
        if (a.xbar_hist != nullptr) vst(a.xbar_hist + (int64_t)i * LD + so, xb1);
        if (a.e_hist != nullptr) vst(a.e_hist + (int64_t)i * LD + so, en);
        vst(a.xbar + (int64_t)i * LD + so, xb1);
        vst(a.e + (int64_t)i * LD + so, en);
      }
    }
    if (a.stats != nullptr) {       // per-scenario-slot partial sums in shared memory, reduced once at the end of the kernel
      __syncwarp();
      if (slice == 0) {
#pragma unroll
        for (int t = 0; t < W; ++t) {
          if (olive[t]) {
            const int c = sc0 + t;
            double nrm2 = 0.0;
            for (int i = 0; i < n; ++i) { const double xv = wb.om[BK::OM_XP + i][c]; nrm2 = fma(xv, xv, nrm2); }
            if (ogood[t]) { wb.stacc[0][c] += sqrt(nrm2); wb.stacc[1][c] += nrm2; wb.stacc[2][c] += wb.cost[c]; }
            if (stt[t] == TZ_STATUS_INFEASIBLE) wb.stacc[3][c] += 1.0;
            if (stt[t] == TZ_STATUS_MAXITER) wb.stacc[4][c] += 1.0;
            wb.stacc[5][c] += (double)wb.iters[c];
            if (stt[t] == TZ_STATUS_NONFINITE) wb.stacc[6][c] += 1.0;
            wb.stacc[7][c] += 1.0;
          }
        }
      }
    }
  }
}

// Persistent kernel; every WARP loops on its own over tiles of SPW = 32/G scenarios, so there is
// no CTA barrier after the program has been staged (a CTA barrier made fast warps wait for the
// slowest ADMM solve of the CTA: 8 % of the samples in profiles/r1_v2_*).
//
// run_program: the work of one CTA on one program.  Warp w of the CTA takes the output tiles tile_first + w,
// tile_first + w + tile_stride, ... below tile_limit of that program's scenarios [0, a.S).
// step_kernel calls it once (tiles strided over the whole grid); step_kernel_set (data-set axis: many programs in one
// launch) calls it once per program that intersects the CTA's contiguous range of tiles.
template <class BK, bool PL>
__device__ __forceinline__ void run_program(unsigned char* smem_raw, const QpProg<BK>* __restrict__ gpg, const Aux& ax,
                                            const SolverParams& sp, const StepArgs& a, const int64_t tile_first,
                                            const int64_t tile_stride, const int64_t tile_limit, const unsigned zseed,
                                            const bool stage = true) {
  constexpr int NZ = BK::NZ, NCL = BK::NCL, N2 = BK::N2, NU = BK::NU, NPAR = BK::NPAR, NAG = BK::NAG, NCHL = BK::NCHL,
                NCOL = BK::NCOL, TPB = BK::TPB, G = BK::G, SPW = BK::SPW, NW = BK::NW, HP = BK::NPAR / 2;
  Smem<BK>& sm = *reinterpret_cast<Smem<BK>*>(smem_raw);
  double* tabd = reinterpret_cast<double*>(smem_raw + sizeof(Smem<BK>));
  const int tid = threadIdx.x;
  const int n = ax.n, m = ax.m, nv = ax.nv;
  int* tabi = reinterpret_cast<int*>(tabd + ax.n_dbl + n * n + n * m);
  const int lane = tid & 31, wib = tid >> 5;
  WarpBuf<BK>& wb = sm.wb[wib];
  const bool explicit_qp = a.q_in != nullptr;
  const int64_t ntiles = tile_limit;
  const int64_t nwarps = tile_stride;
  const int64_t otile0 = tile_first + wib;
  // list mode (the tiles fast_step_kernel deferred): iteration i works on output tile defer_list[i]
  const int64_t tile_max = (a.S + BK::SPO - 1) / BK::SPO - 1;
  auto tile_at = [&](int64_t i) {
    if (!a.list_mode) return i;
    const int64_t t = a.defer_list[i];
    return t < 0 ? (int64_t)0 : (t > tile_max ? tile_max : t);
  };
  const double* hintp = (sp.warm == 2 && !explicit_qp) ? a.warm : nullptr;
  // inputs of this warp's first output tile: in flight while the program is staged (cp.async group 0)
  if (!explicit_qp && otile0 < ntiles) prefetch_inputs<BK>(wb.pre[0], a, hintp, n, tile_at(otile0), lane);
  if (stage) {  // stage the program and its tables once per CTA (persistent kernel: amortised over all tiles of this CTA): 16-byte
     // cp.async copies, all in flight at once (a load/store loop serialised ~10 dependent round trips to L2 per thread)
    const char* src = reinterpret_cast<const char*>(gpg);
    char* dst = reinterpret_cast<char*>(&sm.pg);
    static_assert(sizeof(QpProg<BK>) % 8 == 0, "QpProg must be a whole number of doubles");
    constexpr int NCH = (int)(sizeof(QpProg<BK>) / 16);
    for (int i = tid; i < NCH; i += TPB) cp_async16(dst + 16 * i, src + 16 * i);
    if (tid == 0 && (sizeof(QpProg<BK>) % 16) != 0) cp_async8(dst + 16 * NCH, src + 16 * NCH);
    for (int i = tid; i < ax.n_dbl; i += TPB) cp_async8(tabd + i, ax.tab + i);
    if (a.x != nullptr && !PL) {
      for (int i = tid; i < n * n; i += TPB) cp_async8(tabd + ax.n_dbl + i, a.A_true + i);
      for (int i = tid; i < n * m; i += TPB) cp_async8(tabd + ax.n_dbl + n * n + i, a.B_true + i);
    }
    const int* gi = reinterpret_cast<const int*>(ax.tab + ax.n_dbl);
    for (int i = tid; i < ax.n_int; i += TPB) tabi[i] = gi[i];
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    for (int i = tid; i < BK::NC * NZ; i += TPB) (&sm.Aa[0][0])[i] = sp.alpha * (&sm.pg.A[0][0])[i];
    __syncthreads();
  }
  const QpProg<BK>& pg = sm.pg;
  const int g = lane % G;                 // lane within the scenario's group
  const int sl = lane / G;                // scenario within the warp's tile (solve-phase mapping)
  const int64_t LD = a.ld;
  const double inv_alpha = 1.0 / sp.alpha;
  const double* sCZ = tabd + ax.o_CZ;
  for (int i = lane; i < TZ_NSTATS * BK::SPO; i += 32) (&wb.stacc[0][0])[i] = 0.0;
  __syncwarp();

  int buf = 0;
  for (int64_t it = otile0; it < ntiles; it += nwarps, buf ^= 1) {
    const int64_t otile = tile_at(it);
    if (!explicit_qp) {        // inputs of the NEXT output tile stream in while this one is solved
      if (it + nwarps < ntiles) {
        prefetch_inputs<BK>(wb.pre[buf ^ 1], a, hintp, n, tile_at(it + nwarps), lane);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncwarp();
    }
    const double (*pre)[BK::SPO] = wb.pre[buf];
    // zero-fill slot of this warp: before solve tile 0, .., before solve tile TPO-1, or (== TPO) in the output phase
    const int zslot = (!explicit_qp && a.ze1 != nullptr && !sp.tube_packed) ? (int)((zseed + wib) % (BK::TPO + 1)) : BK::TPO;
   #pragma unroll 1
   for (int half = 0; half < BK::TPO; ++half) {
    if (half == zslot) {
      if (a.vec2) zero_fill<BK, 2>(ax, a, otile, lane);
      else zero_fill<BK, 1>(ax, a, otile, lane);
    }
    const int col = half * SPW + sl;        // column of this scenario in the warp's exchange buffers
    const int64_t s = otile * BK::SPO + col;
    const bool live = s < a.S;
    double c0 = 0.0;
    bool param_ok = true, finite = true;
    LaneQp<BK> qp;
    double w[2 * BK::NCOL2];                 // w = [1 | p | |p| | general atoms |Bt p + gam|] (+ a zero pad)

    if (!explicit_qp) {
      // ---- parameters p = [xbar0 | e0] (every lane of the group loads them: same sectors)
      w[0] = 1.0;
      if constexpr (2 * BK::NCOL2 > NCOL) w[2 * BK::NCOL2 - 1] = 0.0;
#pragma unroll
      for (int j = 0; j < HP; ++j) {
        double xv = 0.0, ev = 0.0;
        if (live && j < n) { xv = pre[j][col]; ev = pre[n + j][col]; }
        w[1 + j] = xv;
        w[1 + HP + j] = ev;
        w[1 + NPAR + j] = fabs(xv);
        w[1 + NPAR + HP + j] = fabs(ev);
        finite = finite && (fabs(xv) < 1e300) && (fabs(ev) < 1e300);
        if (g == 0) { wb.om[BK::OM_P + j][col] = xv; wb.om[BK::OM_P + HP + j][col] = ev; }   // kept for the output phase
      }
      eval_atoms<BK>(pg, w);
      // ---- this lane's rows of the bounds: l = l0 + R w, u = u0 + R w (scaled), kinks
#pragma unroll
      for (int k = 0; k < NCL; ++k) {
        const int i = k * G + g;
        const double r = row_shift<BK>(pg, i, w);     // (16-byte shared loads, two accumulation chains per row)
        if (k < N2) {
          qp.lo[k < N2 ? k : 0] = pg.l0[i] + r;
          qp.hi[k < N2 ? k : 0] = pg.u0[i] + r;
          qp.kink[k < N2 ? k : 0] = pg.kink0[i % BK::NK] + r;
        } else if (k < N2 + NU) {
          qp.hi[k < N2 + NU ? k : 0] = pg.u0[i] + r;
        } else {
          qp.lo[k - NU] = pg.l0[i] + r;
        }
      }
      eval_q<BK>(pg, w, qp.q);
      // ---- parameter-only feasibility rows, split over the group:  sum_j R_j w_j <= 1e-9 max(1, sum_j |R_j| |w_j|)
      int bad = 0;
#pragma unroll
      for (int k = 0; k < NCHL; ++k) {
        const int i = k * G + g;
        if (i < pg.nchk) bad |= param_row_violated<BK>(pg, i % BK::NCHK, w) ? 1 : 0;
      }
      param_ok = gor<G>(bad) == 0;
      // ---- cost constant c0(p)
      c0 = cost_const<BK>(pg, w);
    } else {
      // explicit instance: scale the caller's q, l, u  (qbar = c D q, lbar = E l)
#pragma unroll
      for (int j = 0; j < NZ; ++j)
        qp.q[j] = (live && j < pg.nz) ? a.q_in[(int64_t)j * LD + s] * pg.D[j] / pg.cinv : 0.0;
#pragma unroll
      for (int k = 0; k < NCL; ++k) {
        const int i = k * G + g;
        const int row = pg.row_of_slot[i];
        const bool rr = live && row >= 0;
        const double lv = rr ? a.l_in[(int64_t)row * LD + s] / pg.Einv[i] : -INFINITY;
        const double uv = rr ? a.u_in[(int64_t)row * LD + s] / pg.Einv[i] : INFINITY;
        if (k < N2) {
          qp.lo[k < N2 ? k : 0] = lv;
          qp.hi[k < N2 ? k : 0] = uv;
          qp.kink[k < N2 ? k : 0] = 0.0;
        } else if (k < N2 + NU) {
          qp.hi[k < N2 + NU ? k : 0] = uv;
        } else {
          qp.lo[k - NU] = lv;
        }
      }
    }
    qp.Aa.base = &sm.Aa[g][0];
    qp.P = pg.P;
    qp.wk = &pg.wabs[g];
    qp.sinv = &pg.sing_inv[g];
    qp.svar = &pg.sing_var[g];

    // ---- ADMM (+ certificate / polish)
    LaneState<BK> st;
    bool warm = false;
    if (TZ_UNLIKELY(sp.warm == 1 && a.warm != nullptr && live)) {
      // layout: [x (NZ) | y (NC, slot-indexed) | activity words (G) | valid flag] x LD
      warm = (a.warm[(int64_t)(NZ + BK::NC + G) * LD + s] == 1.0);
      if (warm) {
#pragma unroll
        for (int j = 0; j < NZ; ++j) st.x[j] = a.warm[(int64_t)j * LD + s];
#pragma unroll
        for (int k = 0; k < NCL; ++k) st.w[k] = a.warm[(int64_t)(NZ + k * G + g) * LD + s];
        st.act = (uint32_t)__double_as_longlong(a.warm[(int64_t)(NZ + BK::NC + g) * LD + s]);
        st.switched = true;
      }
    }
    const bool solve_it = live && param_ok && finite;
    int iters = 0;
    bool certified = false;
    int status = TZ_STATUS_OK;
    // ---- active-set hint (warm_start == 2): the optimal active set of the scenario's previous closed-loop step is
    // tried first; when its KKT certificate holds the step is solved exactly without a single ADMM iteration
    const bool use_hint = sp.warm == 2 && a.warm != nullptr;
    bool hint_ok = false;
    double hint_obj = 0.0;          // NZ == 2: scaled objective of the hint-certified point (tz_cert2.cuh)
    bool fresh = false;             // first step of a run (or no usable hint): its active set becomes the run-start hint
    if (use_hint) {
      unsigned long long hint = 0ull;
      if (live) hint = (unsigned long long)__double_as_longlong(pre[4 * n + g][col]);
      fresh = !(hint & kCodeValid) || (hint & kCodeFresh);
      // (the group reduction is a warp-wide shuffle: every lane must execute it, so no short-circuit on solve_it)
      const int invalid = gor<G>((hint & kCodeValid) ? 0 : 1);
      const bool valid = solve_it && invalid == 0;
      if (__any_sync(0xffffffffu, valid)) {
        const unsigned long long code = hint & ~(kCodeValid | kCodeFresh);
        if constexpr (NZ == 2) {
          // two-variable programs: the closed-form certificate of tz_cert2.cuh, evaluated redundantly by the G lanes of
          // the group -- the function fast_step_kernel runs with one thread per scenario, hence bit-identical results
          unsigned long long hwv[G];
#pragma unroll
          for (int j = 0; j < G; ++j) hwv[j] = __shfl_sync(0xffffffffu, code, (lane & ~(G - 1)) + j);
          const Cert2Result cr = certify2<BK>(pg, w, qp.q, hwv);
          if (cr.verdict == kCertOk && valid) {
            st.x[0] = cr.x[0];
            st.x[NZ - 1] = cr.x[1];
            st.code = code;
            hint_obj = cr.obj;
            hint_ok = true;
          }
        } else {
          double lam[NCL], xk[NZ], x0[NZ];
#pragma unroll
          for (int k = 0; k < NCL; ++k) lam[k] = 0.0;
#pragma unroll
          for (int j = 0; j < NZ; ++j) x0[j] = 0.0;
          const bool ok = admm_certify<BK>(qp, inv_alpha, sp.polish > 0 ? sp.polish : 3, code, x0, lam, xk);
          if (ok && valid) {
#pragma unroll
            for (int j = 0; j < NZ; ++j) st.x[j] = xk[j];
#pragma unroll
            for (int k = 0; k < NCL; ++k) st.w[k] = lam[k];
            st.code = code;
            hint_ok = true;
          }
        }
      }
    }
    if (TZ_UNLIKELY(!__all_sync(0xffffffffu, hint_ok || !solve_it))) {
      // no (valid) hint: is the program infeasible outright?  (singleton presolve, exact; saves the ADMM iterations and
      // the failed certificate an infeasible scenario would otherwise need before the same test inside admm_solve)
      const bool inf = singleton_infeasible<BK>(qp);
      const bool run = solve_it && !hint_ok && !inf;
      bool cert2 = false;
      int st2 = TZ_STATUS_INFEASIBLE;
      if (__any_sync(0xffffffffu, run)) {
        const int st3 = admm_solve<BK>(qp, sp, run, st, warm, &wb.ysave[0][lane], iters, cert2, true);
        if (run) st2 = st3;
      }
      if (!hint_ok) { status = st2; certified = cert2; }
    }
    if (hint_ok) { certified = true; iters = 0; }
    if (live && !finite) status = TZ_STATUS_NONFINITE;
    else if (live && !param_ok) status = TZ_STATUS_INFEASIBLE;
    const bool good = live && (status == TZ_STATUS_OK || status == TZ_STATUS_MAXITER);
    if (use_hint) {
      // hint rows [0, G): the active set for the next step; rows [G, 2G): the active set of the run's first step, which
      // becomes the hint again when the scenario restarts from x_restart (same state, same program, same active set)
      if (live) {
        unsigned long long wnext = 0ull;
        if (good) {
          if (status == TZ_STATUS_OK) {        // (a MAXITER iterate is applied but its active set is not trusted as a hint)
            wnext = st.code | kCodeValid;
            if (fresh) a.warm[(int64_t)(G + g) * LD + s] = __longlong_as_double((long long)wnext);
          }
        } else if (a.x_restart != nullptr) {
          const unsigned long long h0 = (unsigned long long)__double_as_longlong(a.warm[(int64_t)(G + g) * LD + s]);
          wnext = (h0 & kCodeValid) ? (h0 | kCodeFresh) : 0ull;
        }
        a.warm[(int64_t)g * LD + s] = __longlong_as_double((long long)wnext);
      }
    } else if (good && a.warm != nullptr) {
      if (g == 0) {
#pragma unroll
        for (int j = 0; j < NZ; ++j) a.warm[(int64_t)j * LD + s] = st.x[j];
        a.warm[(int64_t)(NZ + BK::NC + G) * LD + s] = 1.0;
      }
#pragma unroll
      for (int k = 0; k < NCL; ++k) a.warm[(int64_t)(NZ + k * G + g) * LD + s] = st.w[k];
      a.warm[(int64_t)(NZ + BK::NC + g) * LD + s] = __longlong_as_double((long long)st.act);
    }
    // residual exits are polished; certified exits already are an exact KKT point
    if (TZ_UNLIKELY(sp.polish && __any_sync(0xffffffffu, good && !certified))) (void)admm_polish<BK>(qp, inv_alpha, st, good && !certified, sp.polish);

    if (TZ_UNLIKELY(explicit_qp)) {
      if (live) {
        if (g == 0) {
          a.status[s] = status;
          if (a.iters) a.iters[s] = iters;
          if (a.z_out) {
#pragma unroll
            for (int j = 0; j < NZ; ++j)
              if (j < pg.nz) a.z_out[(int64_t)j * LD + s] = good ? pg.D[j] * st.x[j] : NAN;
          }
        }
        if (a.y_out) {
#pragma unroll
          for (int k = 0; k < NCL; ++k) {
            const int i = k * G + g;
            const int row = pg.row_of_slot[i];
            if (row >= 0) a.y_out[(int64_t)row * LD + s] = good ? st.w[k] * pg.cinv / pg.Einv[i] : NAN;
          }
        }
      }
      continue;
    }

    // ---- objective value (reference `result`, tzddpc/tzddpc.py:367,377; constant terms included, quirk Q7)
    double kcost = 0.0;
#pragma unroll
    for (int k = 0; k < N2; ++k) {
      double axv = 0.0;
#pragma unroll
      for (int j = 0; j < NZ; ++j) axv = fma(qp.Aa[k][j], st.x[j], axv);
      kcost = fma(qp.wk[k * G], fabs(axv * inv_alpha - qp.kink[k]), kcost);
    }
    kcost = gsum<G>(kcost);
    double cost = NAN;
    if (good) {
      double acc = kcost;
#pragma unroll
      for (int j = 0; j < NZ; ++j) {
        double px = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) px = fma(qp.P[j][b], st.x[b], px);
        acc = fma(0.5 * px + qp.q[j], st.x[j], acc);
      }
      cost = fma(acc, pg.cinv, c0);
      if (NZ == 2 && hint_ok) cost = fma(hint_obj, pg.cinv, c0);      // the arithmetic of fast_step_kernel
    } else if (live && status == TZ_STATUS_INFEASIBLE) {
      cost = INFINITY;                      // cvxpy returns +inf for an infeasible Minimize (:374)
    }
    // ---- hand om = [1 | v | p | centre of Ze[1]], cost, status to the output phase (warp-private buffer)
    if (g == 0) {
      wb.om[0][col] = 1.0;
#pragma unroll
      for (int j = 0; j < NZ; ++j) wb.om[BK::OM_V + j][col] = (j < nv) ? (good ? pg.D[j] * st.x[j] : NAN) : 0.0;
      wb.cost[col] = cost;
      wb.status[col] = live ? status : -1;
      wb.iters[col] = iters;
    }
    __syncwarp();
    for (int r = g; r < n; r += G) {        // centre of Ze[1]: rows split over the group
      const double* row = sCZ + r * NW;
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < NW; ++j) acc = fma(row[j], wb.om[j][col], acc);
      wb.om[BK::OM_C + r][col] = acc;
    }
   }     // solve tiles of this output tile
    if (explicit_qp) continue;
    __syncwarp();
    if (TZ_LIKELY(a.vec2)) output_phase<BK, 2, PL>(wb, pre, ax, a, tabd, tabi, otile, lane, zslot < BK::TPO, sp.tube_packed != 0);
    else output_phase<BK, 1, PL>(wb, pre, ax, a, tabd, tabi, otile, lane, zslot < BK::TPO, sp.tube_packed != 0);
    __syncwarp();     // wb is rewritten by the next tile
  }
  if (a.stats != nullptr && a.x != nullptr) {
    __syncwarp();
    if (lane < TZ_NSTATS) {
      double v_ = 0.0;
#pragma unroll
      for (int c = 0; c < BK::SPO; ++c) v_ += wb.stacc[lane][c];
      if (v_ != 0.0) atomicAdd(a.stats + lane, v_);
    }
  }
}

// Step k of a fused run: noise and every per-step output advanced to their k-th block (blocks of leading dimension a.ld).
// tube_rows: the rows of one Ze[1].Z block (0 without a tube).  step_kernel's fused run below spells the same offsets out:
// written as a call to this function they change its register allocation (more spills).
__device__ __forceinline__ StepArgs step_block(const StepArgs& a, const Aux& ax, const int64_t tube_rows, const int k) {
  const int64_t LD = a.ld;
  StepArgs ak = a;
  if (ak.noise) ak.noise += (int64_t)k * ax.n * LD;
  if (ak.cost) ak.cost += (int64_t)k * LD;
  if (ak.v) ak.v += (int64_t)k * ax.nv * LD;
  if (ak.xbar_traj) ak.xbar_traj += (int64_t)k * (ax.N + 1) * ax.n * LD;
  if (ak.ze1) ak.ze1 += (int64_t)k * tube_rows * LD;
  if (ak.u_out) ak.u_out += (int64_t)k * ax.m * LD;
  ak.status += (int64_t)k * LD;
  if (ak.iters) ak.iters += (int64_t)k * LD;
  if (ak.stats) ak.stats += (int64_t)k * TZ_NSTATS;
  if (ak.x_hist) ak.x_hist += (int64_t)k * ax.n * LD;
  if (ak.xbar_hist) ak.xbar_hist += (int64_t)k * ax.n * LD;
  if (ak.e_hist) ak.e_hist += (int64_t)k * ax.n * LD;
  return ak;
}

// Persistent kernel of one program: one wave of CTAs.  PL: a plant per scenario (StepArgs::AB_true).
template <class BK, bool PL = false>
__global__ void __launch_bounds__(BK::TPB, BK::MINB) step_kernel(const QpProg<BK>* __restrict__ gpg, const Aux ax,
                                                                const SolverParams sp, const StepArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  pdl_wait();
  int64_t ntiles = (a.S + BK::SPO - 1) / BK::SPO;
  if (a.list_mode) {
    // the tiles fast_step_kernel could not decide; every CTA takes an exit ticket and the last one clears the list
    const int64_t cnt = *reinterpret_cast<volatile const int32_t*>(a.defer);
    ntiles = cnt < 0 ? 0 : (cnt < ntiles ? cnt : ntiles);          // (a foreign scratch buffer cannot send the kernel out of bounds)
    if ((int64_t)blockIdx.x * BK::WPB < ntiles)
      run_program<BK, PL>(smem_raw, gpg, ax, sp, a, (int64_t)blockIdx.x * BK::WPB, (int64_t)gridDim.x * BK::WPB, ntiles,
                          blockIdx.x * BK::WPB);
    __syncthreads();
    if (threadIdx.x == 0) {
      const int t = atomicAdd(a.defer + 1, 1);
      if (t == (int)gridDim.x - 1) { a.defer[0] = 0; a.defer[1] = 0; }
    }
    return;
  }
  if (a.nsteps <= 1) {
    run_program<BK, PL>(smem_raw, gpg, ax, sp, a, (int64_t)blockIdx.x * BK::WPB, (int64_t)gridDim.x * BK::WPB, ntiles,
                    blockIdx.x * BK::WPB);
    return;
  }
  // fused run: a warp keeps its tiles for all steps (scenarios are independent, so nothing has to cross warps); the
  // state, the hints and the outputs of step k are ordinary global stores of this warp, read back by the same warp in
  // step k + 1 behind a warp barrier.  The program is staged once.
  const int64_t LD = a.ld;
  const int64_t tube_rows = a.ze1 ? (sp.tube_packed ? ax.n_nz : ax.n * (1 + ax.g1)) : 0;
#pragma unroll 1
  for (int k = 0; k < a.nsteps; ++k) {
    StepArgs ak = a;
    if (ak.noise) ak.noise += (int64_t)k * ax.n * LD;
    if (ak.cost) ak.cost += (int64_t)k * LD;
    if (ak.v) ak.v += (int64_t)k * ax.nv * LD;
    if (ak.xbar_traj) ak.xbar_traj += (int64_t)k * (ax.N + 1) * ax.n * LD;
    if (ak.ze1) ak.ze1 += (int64_t)k * tube_rows * LD;
    if (ak.u_out) ak.u_out += (int64_t)k * ax.m * LD;
    ak.status += (int64_t)k * LD;
    if (ak.iters) ak.iters += (int64_t)k * LD;
    if (ak.stats) ak.stats += (int64_t)k * TZ_NSTATS;
    if (ak.x_hist) ak.x_hist += (int64_t)k * ax.n * LD;
    if (ak.xbar_hist) ak.xbar_hist += (int64_t)k * ax.n * LD;
    if (ak.e_hist) ak.e_hist += (int64_t)k * ax.n * LD;
    run_program<BK, PL>(smem_raw, gpg, ax, sp, ak, (int64_t)blockIdx.x * BK::WPB, (int64_t)gridDim.x * BK::WPB, ntiles,
                        blockIdx.x * BK::WPB + k, k == 0);
    __threadfence_block();
    __syncwarp();
  }
}

// Data-set axis (BASELINE.json north_star: scenarios = noise realisations x initial states x DATA SETS): `nprog` programs
// of identical structure -- the same problem built from different data sets, hence different (P, A, R, ...) -- in ONE
// launch.  Scenarios [e.begin, e.end) of the batch belong to program e.  The output tiles of all programs are numbered
// consecutively (e.tile_begin) and dealt out exactly as step_kernel deals out the tiles of one program: in round k the
// WPB warps of CTA b take the tiles (b + k * gridDim.x) * WPB + w.  At any moment the grid therefore writes one contiguous
// window of scenarios (DRAM page locality: giving every CTA its own contiguous range of tiles cost 12 %), the load is
// balanced whatever the number and the sizes of the programs, and a CTA re-stages the program image in shared memory
// only when its next tiles belong to another program (every round once the programs are smaller than a wave).
struct SetEntry {
  const void* pg;         // QpProg<bucket> image on the device
  const double* tab;      // run-time tables (Aux::tab) of this program
  int64_t begin, end;     // its scenarios
  int64_t tile_begin;     // number of output tiles of the programs before it
};

template <bool PL>
__device__ __forceinline__ StepArgs shift_args(const StepArgs& a, int64_t b, int64_t cnt) {
  StepArgs r = a;
  r.S = cnt;
#define TZ_SH(f) if (r.f) r.f += b;
  TZ_SH(xbar0) TZ_SH(e0) TZ_SH(x) TZ_SH(xbar) TZ_SH(e) TZ_SH(noise) TZ_SH(x_restart) TZ_SH(cost) TZ_SH(v) TZ_SH(xbar_traj)
  TZ_SH(ze1) TZ_SH(u_out) TZ_SH(status) TZ_SH(iters) TZ_SH(warm)
  if constexpr (PL) r.AB_true += b;
#undef TZ_SH
  return r;
}

template <class BK, bool PL = false>
__global__ void __launch_bounds__(BK::TPB, BK::MINB) step_kernel_set(const SetEntry* __restrict__ entries, const int nprog,
                                                                    const int64_t total_tiles, const Aux ax0,
                                                                    const SolverParams sp, const StepArgs a0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  pdl_wait();
  int staged = -1;                                 // program whose image is in shared memory
  int lo = 0;
  // round k: the CTA's WPB warps take the consecutive tiles [base, base + WPB) of the global numbering
  for (int64_t base = (int64_t)blockIdx.x * BK::WPB; base < total_tiles; base += (int64_t)gridDim.x * BK::WPB) {
    const int64_t t1 = base + BK::WPB < total_tiles ? base + BK::WPB : total_tiles;
    int hi = nprog - 1;                            // last program with tile_begin <= base (programs are visited in order)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (entries[mid].tile_begin <= base) lo = mid;
      else hi = mid - 1;
    }
    int j = lo;
    for (int64_t t = base; t < t1 && j < nprog; ++j) {
      const SetEntry en = entries[j];
      const int64_t ntl = (en.end - en.begin + BK::SPO - 1) / BK::SPO;
      const int64_t tend = en.tile_begin + ntl < t1 ? en.tile_begin + ntl : t1;
      if (tend <= t) continue;                     // (an empty program)
      Aux ax = ax0;
      ax.tab = en.tab;
      const StepArgs a = shift_args<PL>(a0, en.begin, en.end - en.begin);
      const bool stage = staged != j;
      if (stage && staged >= 0) __syncthreads();   // every warp is done with the previous program's image
      staged = j;
      // warp w takes tile (t + w) of the round when it belongs to this program (tile_stride: beyond the limit)
      run_program<BK, PL>(smem_raw, reinterpret_cast<const QpProg<BK>*>(en.pg), ax, sp, a, t - en.tile_begin, BK::WPB,
                          tend - en.tile_begin, (unsigned)(base % 1024), stage);
      t = tend;
    }
  }
}

// Fused run over a program set (tz_closed_loop_run_set): nsteps > 0 closed-loop steps in one launch.  The tiles are dealt
// out as step_kernel_set deals them; scenarios are independent, so a warp keeps its tile of a (round, program) segment for
// all steps, and the segment's steps run back to back behind one staging of the program image (as step_kernel's fused run
// does for one program).  The per-step blocks are laid out with the batch's leading dimension (step_block on a0, before
// shift_args narrows S to the program's scenarios); the histories, which shift_args leaves alone, start at the program's
// first scenario.
template <class BK, bool PL = false>
__global__ void __launch_bounds__(BK::TPB, BK::MINB) step_kernel_set_run(const SetEntry* __restrict__ entries, const int nprog,
                                                                        const int64_t total_tiles, const Aux ax0,
                                                                        const SolverParams sp, const StepArgs a0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  pdl_wait();
  const int64_t tube_rows = a0.ze1 ? (sp.tube_packed ? ax0.n_nz : ax0.n * (1 + ax0.g1)) : 0;
  int staged = -1;                                 // program whose image is in shared memory
  int lo = 0;
  for (int64_t base = (int64_t)blockIdx.x * BK::WPB; base < total_tiles; base += (int64_t)gridDim.x * BK::WPB) {
    const int64_t t1 = base + BK::WPB < total_tiles ? base + BK::WPB : total_tiles;
    int hi = nprog - 1;                            // last program with tile_begin <= base (programs are visited in order)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (entries[mid].tile_begin <= base) lo = mid;
      else hi = mid - 1;
    }
    int j = lo;
    for (int64_t t = base; t < t1 && j < nprog; ++j) {
      const SetEntry en = entries[j];
      const int64_t ntl = (en.end - en.begin + BK::SPO - 1) / BK::SPO;
      const int64_t tend = en.tile_begin + ntl < t1 ? en.tile_begin + ntl : t1;
      if (tend <= t) continue;                     // (an empty program)
      Aux ax = ax0;
      ax.tab = en.tab;
      const bool stage = staged != j;
      if (stage && staged >= 0) __syncthreads();   // every warp is done with the previous program's image
      staged = j;
#pragma unroll 1
      for (int k = 0; k < a0.nsteps; ++k) {
        StepArgs a = shift_args<PL>(step_block(a0, ax0, tube_rows, k), en.begin, en.end - en.begin);
        if (a.x_hist) a.x_hist += en.begin;
        if (a.xbar_hist) a.xbar_hist += en.begin;
        if (a.e_hist) a.e_hist += en.begin;
        run_program<BK, PL>(smem_raw, reinterpret_cast<const QpProg<BK>*>(en.pg), ax, sp, a, t - en.tile_begin, BK::WPB,
                            tend - en.tile_begin, (unsigned)((base + k) % 1024), stage && k == 0);
        __threadfence_block();                     // step k + 1 of this warp's tile reads what step k stored
        __syncwarp();
      }
      t = tend;
    }
  }
}

// The tiles fast_step_kernel deferred, for a program set: listed tile t (a global 16-scenario tile) belongs to program
// tile_prog[t]; a CTA takes one listed tile at a time (its first warp solves it), re-staging the program image when the
// program changes.  Every CTA takes an exit ticket and the last one clears the list, as step_kernel does.
template <class BK, bool PL = false>
__global__ void __launch_bounds__(BK::TPB, BK::MINB) step_kernel_set_list(const SetEntry* __restrict__ entries,
                                                                         const int32_t* __restrict__ tile_prog, const Aux ax0,
                                                                         const SolverParams sp, const StepArgs a0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  pdl_trigger();
  pdl_wait();
  const int64_t max_tiles = (a0.S + BK::SPO - 1) / BK::SPO;
  const int64_t cnt = *reinterpret_cast<volatile const int32_t*>(a0.defer);
  const int64_t ntl = cnt < 0 ? 0 : (cnt < max_tiles ? cnt : max_tiles);
  int staged = -1;
  for (int64_t i = blockIdx.x; i < ntl; i += gridDim.x) {
    int64_t t = a0.defer_list[i];
    t = t < 0 ? 0 : (t >= max_tiles ? max_tiles - 1 : t);
    const int j = tile_prog[t];
    const SetEntry en = entries[j];
    Aux ax = ax0;
    ax.tab = en.tab;
    StepArgs a = shift_args<PL>(a0, en.begin, en.end - en.begin);
    a.list_mode = 0;
    const bool stage = staged != j;
    if (stage && staged >= 0) __syncthreads();     // every warp is done with the previous program's image
    staged = j;
    const int64_t tl = t - en.begin / BK::SPO;     // the tile within its program (programs start on whole tiles)
    run_program<BK, PL>(smem_raw, reinterpret_cast<const QpProg<BK>*>(en.pg), ax, sp, a, tl, BK::WPB, tl + 1, (unsigned)(t % 1024), stage);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int tk = atomicAdd(a0.defer + 1, 1);
    if (tk == (int)gridDim.x - 1) { a0.defer[0] = 0; a0.defer[1] = 0; }
  }
}

// ---- compiled buckets: <NZ, N2, NU, NL, G, NPAR, NAG, NCHK, MINB> -------------------------------
using B0 = Bucket<2, 1, 3, 3, 4, 10, 2, 12, 3>;      // N = 2, m = 1, n <= 5: the three shipped examples (28 row slots)
using B1 = Bucket<4, 2, 4, 4, 8, 16, 8, 32, 3>;      // generic small   (80 row slots)
using B2 = Bucket<8, 3, 5, 5, 8, 16, 24, 32, 2>;     // generic medium  (104 row slots, N = 3..4)
using B3 = Bucket<12, 1, 4, 4, 8, 16, 24, 32, 1>;    // large           (72 row slots, nz <= 12: N = 5 of the complexity sweep)

}  // namespace tz

namespace tz { struct BigProgram; }

struct TzProgram {
  int bucket = -1;
  void* packed_dev = nullptr;            // device image of QpProg<bucket>, staged into shared memory by every CTA
  void* aux_dev = nullptr;               // one allocation holding the run-time sized tables
  tz::Aux aux{};
  int nz = 0, nc = 0, n = 0, m = 0, N = 0, nv = 0, g1 = 0, npar = 0;
  int NZ = 0, NC = 0, G = 0;
  int NW = 0, OM_V = 0, OM_P = 0, OM_C = 0, HP = 0;     // om layout of the bucket (Bucket::OM_*)
  std::vector<int32_t> tube_ent;         // entries of Ze[1].Z (row-major index) that are not structurally zero, in table order
  size_t smem_tab = 0;                   // bytes of the run-time tables staged behind Smem<bucket>
  int num_sms = 148;
  int device = -1;                       // the CUDA device the program image lives on: launches on another device are refused
  bool owns_device = true;               // false: packed_dev / aux_dev are slices of a TzProgramBatch's allocations
  tz::BigProgram* big = nullptr;         // bucket 4: the generic large-program path (tz_big.cu) instead of a packed image
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute of a kernel.  The only process-wide state of the
// library is this cache of "already set on device d" bits, one word per kernel; setting the attribute is idempotent, so a
// race between two threads only repeats the call.
template <class K>
int ensure_dynamic_smem(K kernel, int bytes, int device, std::atomic<unsigned long long>& done) {
  const unsigned long long bit = 1ull << (device & 63);
  if (device >= 0 && device < 64 && (done.load(std::memory_order_relaxed) & bit)) return TZ_OK;
  TZ_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  if (device >= 0 && device < 64) done.fetch_or(bit, std::memory_order_relaxed);
  return TZ_OK;
}

constexpr int kMaxTabBytes = 24 * 1024;


namespace tz {

// Launches `kernel`, a step kernel of bucket BK, on `grid` CTAs with the shared memory of the bucket and program p's tables.
// The kernel is a template argument so that every kernel keeps its own cache of the devices its attribute is set on.
template <class BK, auto kernel, class... Args>
int launch_step(const TzProgram* p, unsigned grid, cudaStream_t st, int64_t S, Args... args) {
  static std::atomic<unsigned long long> configured{0ull};
  if (const int rc = ensure_dynamic_smem(kernel, (int)(sizeof(Smem<BK>) + kMaxTabBytes), p->device, configured)) return rc;
  TZ_CUDA(launch_kernel(kernel, grid, BK::TPB, sizeof(Smem<BK>) + p->smem_tab, st, pdl_enabled(S), args...));
  return TZ_OK;
}

template <class BK>
int launch_bucket(const TzProgram* p, const SolverParams& sp, const StepArgs& a, cudaStream_t st) {
  // persistent grid: one wave of CTAs (MINB per SM); every warp loops over tiles of SPW scenarios
  const int64_t ntiles = (a.S + BK::SPO - 1) / BK::SPO;
  const int64_t need = (ntiles + BK::WPB - 1) / BK::WPB;
  // (list mode -- the tiles fast_step_kernel deferred, normally none or a handful: one CTA per SM keeps the empty pass short)
  const int64_t wave = (int64_t)p->num_sms * (a.list_mode ? 1 : BK::MINB);
  const unsigned grid = (unsigned)(need < wave ? need : wave);
  return with_plant(a, [&](auto pl) {
    return launch_step<BK, step_kernel<BK, decltype(pl)::value>>(p, grid, st, a.S, reinterpret_cast<const QpProg<BK>*>(p->packed_dev),
                                                                 p->aux, sp, a);
  });
}

// data-set axis: one launch over `nprog` programs (entries on the device); see step_kernel_set
template <class BK>
int launch_bucket_set(const TzProgram* p0, const SetEntry* entries_dev, int nprog, int64_t total_tiles, const SolverParams& sp,
                      const StepArgs& a, cudaStream_t st) {
  static_assert(BK::SPO == TZ_SPO_MIN, "tz_program_set_create counts output tiles of TZ_SPO_MIN scenarios");
  // one wave of CTAs, each with an equal contiguous share of the tiles of all programs (at least one tile per warp)
  const int64_t wave = (int64_t)p0->num_sms * BK::MINB;
  const int64_t need = (total_tiles + BK::WPB - 1) / BK::WPB;
  const unsigned grid = (unsigned)(need < wave ? need : wave);
  return with_plant(a, [&](auto pl) {
    return launch_step<BK, step_kernel_set<BK, decltype(pl)::value>>(p0, grid, st, a.S, entries_dev, nprog, total_tiles, p0->aux, sp, a);
  });
}

// fused run over a program set (a.nsteps steps); see step_kernel_set_run.  The grid of launch_bucket_set.
template <class BK>
int launch_bucket_set_run(const TzProgram* p0, const SetEntry* entries_dev, int nprog, int64_t total_tiles, const SolverParams& sp,
                          const StepArgs& a, cudaStream_t st) {
  static_assert(BK::SPO == TZ_SPO_MIN, "tz_program_set_create counts output tiles of TZ_SPO_MIN scenarios");
  const int64_t wave = (int64_t)p0->num_sms * BK::MINB;
  const int64_t need = (total_tiles + BK::WPB - 1) / BK::WPB;
  const unsigned grid = (unsigned)(need < wave ? need : wave);
  return with_plant(a, [&](auto pl) {
    return launch_step<BK, step_kernel_set_run<BK, decltype(pl)::value>>(p0, grid, st, a.S, entries_dev, nprog, total_tiles, p0->aux, sp,
                                                                         a);
  });
}

template <class BK>
int launch_bucket_set_list(const TzProgram* p0, const SetEntry* entries_dev, const int32_t* tile_prog, const SolverParams& sp,
                           const StepArgs& a, cudaStream_t st) {
  const int64_t ntiles = (a.S + BK::SPO - 1) / BK::SPO;
  const unsigned grid = (unsigned)(ntiles < p0->num_sms ? ntiles : p0->num_sms);
  return with_plant(a, [&](auto pl) {
    return launch_step<BK, step_kernel_set_list<BK, decltype(pl)::value>>(p0, grid, st, a.S, entries_dev, tile_prog, p0->aux, sp, a);
  });
}

}  // namespace tz
