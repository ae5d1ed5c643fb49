// fast_step_kernel: the closed-loop step of the two-variable programs (bucket B0) with ONE THREAD PER SCENARIO.
//
// Replaces, per closed-loop step, tzddpc/tzddpc.py:357-377 (solve) and examples/2.pulley_sim.py:90-96 (update), as
// step_kernel does -- for the scenarios whose active-set hint (the optimal active set of their previous step) still
// certifies.  In a running closed loop that is all but a fraction of a percent of the scenario-steps, and for them
// the solve is the closed-form KKT test of tz_cert2.cuh: no ADMM iteration, no lane group, no shuffle.
//
// Why a second kernel (profiles/r1_v12_*): step_kernel needs 168 registers (3 CTAs = 12 warps per SM) because it
// carries the whole ADMM machinery, issues 29.5 M warp instructions per 65,536 scenarios (replicated x / factor /
// certificate in the 4 lanes of a group, 12 % of them shuffles) and sits on dependent-issue latency at IPC 1.
// Here a warp owns 32 consecutive scenarios, lane = scenario:
//   * every load / store of the scenario-fastest arrays is one fully coalesced 256-byte access per row, straight from /
//     to registers (no exchange buffer, no re-mapping between solve and output phase);
//   * program coefficients (R, A, XB, ...) are read from shared memory at warp-uniform addresses: one broadcast load
//     serves 32 scenarios;
//   * the code is kept COMPACT (row loops are real loops): a warp runs through the kernel once, so straight-line code is
//     fetched from L2 by every warp -- the first, fully unrolled version spent 3-4 stall cycles per issued instruction
//     waiting for instructions (profiles/r2_fast_v0_*: no_instruction);
//   * the dense Ze[1].Z (88 % structural zeros, but dense by the reference's contract) is written once: the zero rows as
//     16-byte streaming stores DRIPPED between the stages of the solve (a flat row list in the program tables: one
//     16-byte index load and one IMAD.WIDE + STG.128 per row), the other entries from the term table.
//     (Measured and dropped: zero-filling the CTA's [entries x scenarios] block with cp.async.bulk.tensor stores of a
//     shared-memory tile of zeros, UTMASTG.2D through a tensor map over the caller's array: the entries that are not
//     structurally zero can only be stored once the bulk group has completed -- 0.0784 ms per step against 0.0705,
//     profiles/r2_fast_v1_tma_*.  Odd warps storing the zeros before they solve and even warps behind: 0.0711 ms against
//     0.0646 dripped.  A dedicated zero warp per CTA, 1D bulk copies per zero row: DESIGN.md section 5.1.)
//   * all loads of the step (parameters, hints, and by cp.async the state x and the noise of the closed-loop update) are
//     in flight before the first store is issued.
// Scenarios the hint cannot decide (no hint yet, active set changed) are DEFERRED in units of 16-scenario output
// tiles: the tile index goes to a list in the caller's warm-start scratch and step_kernel, launched right behind on
// the same stream, solves exactly those tiles (ADMM + certificate).  Both kernels use the same closed-form function
// for hint-certified scenarios, so a scenario's result does not depend on which kernel handled its tile.
#pragma once
#include <cstdlib>

#include "tz_step.cuh"

namespace tz {

constexpr int kDeferTile = TZ_SPO_MIN;     // scenarios per deferred tile = output tile of step_kernel

// NSLOT = 0: one program for the whole batch, staged once per CTA of a persistent grid.
// NSLOT = 1 / 2: a program SET (the data-set axis, tz_closed_loop_step_set): one block of TPB scenarios per CTA; its
// 16-scenario tiles look their program up in tile_prog.  NSLOT = 1: the set guarantees that a block lies within one
// program; NSLOT = 2 (TPB = 32): the two half-warps of the warp may belong to two programs, each staged in its own slot --
// a coefficient load then has two distinct addresses per warp instead of one.
// resident CTAs per SM the register budget is set for (128 registers per thread)
constexpr int fast_ctas_per_sm(int tpb) { return tpb >= 512 ? 1 : 512 / tpb; }

// (Output stores are st.cs: default-policy and write-through stores measured 0.0689 / 0.0674 ms against 0.0598.)
// H > 1 (small batches, where SMs would otherwise host one or two warps): the CTA carries H threads per scenario,
// threads [hq * TPB, (hq + 1) * TPB) being helper group hq.  Group 0 loads, solves and updates exactly as for H = 1; the
// helper groups store the structural zeros of the block's dense tube meanwhile (they do not depend on the solve), and
// behind a CTA barrier all H groups share the tube entries and trajectory rows of the block's scenarios, read from om.
// Per-scenario arithmetic is the same expressions on the same operands: results do not depend on H.
// (First version: zeros split row-wise within every run, behind the barrier: 17 instructions per store, no gain.)
// (Measured and dropped, round 2 again: the zeros as bulk copies -- cp.async.bulk shared -> global of a TPB * 8-byte block
// of zeros, one 2 KB copy per zero row and CTA block, issued by the block's threads a row each, either all behind the
// staging barrier or spread over the drip sites: 0.072-0.073 ms against 0.060-0.061 with the dripped 16-byte stores.)
// PL: a plant per scenario (StepArgs::AB_true), read at the update.  Loads there come after the step's first stores, so every
// thread prefetches its scenario's n(n+m) plant entries into L2 together with the step's other loads; holding them in registers
// instead would need 2 n(n+m) = 60 of them for the 5-dim system on top of a budget of 128, and staging them in shared memory
// next to x and the noise 30 rows of om, 60 KB per 256-thread CTA (one resident CTA per SM instead of two).
template <class BK, int TPB, int NSLOT, int H = 1, bool PL = false>
__global__ void __launch_bounds__(TPB * H, fast_ctas_per_sm(TPB * H))
    fast_step_kernel(const QpProg<BK>* __restrict__ gpg, const Aux ax, const SolverParams sp, const StepArgs a,
                     const SetEntry* __restrict__ entries, const int32_t* __restrict__ tile_prog, const int slot_bytes) {
  constexpr int NZ = BK::NZ, NPAR = BK::NPAR, HP = BK::NPAR / 2, NCOL = BK::NCOL, NW = BK::NW, G = BK::G;
  static_assert(kDeferTile == 16 && BK::SPO == 16, "deferred tiles are the 16-scenario output tiles of step_kernel");
  static_assert(NSLOT <= 1 || TPB == 32, "two program slots: one warp per CTA");
  constexpr int OM_X = NW + HP, OM_NS = NW + 2 * HP;        // om rows of this kernel: [1 | v | p | centre | x | noise]
  constexpr int QPB = (int)((sizeof(QpProg<BK>) + 15) & ~(size_t)15);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tix = threadIdx.x, tid = tix % TPB, hq = tix / TPB, lane = tix & 31;      // (hq is warp-uniform: TPB % 32 == 0)
  constexpr int NT = TPB * H;
  const int n = ax.n, m = ax.m, nv = ax.nv;
  const bool closed = a.x != nullptr;
  const int64_t LD = a.ld;
  const bool dense = a.ze1 != nullptr && !sp.tube_packed;
  // shared memory: NSLOT (or one) x [QpProg | tables | A_true | B_true], then om[KOM][TPB]
  double (*om)[TPB] = reinterpret_cast<double (*)[TPB]>(smem_raw + (NSLOT > 1 ? NSLOT : 1) * (size_t)slot_bytes);
  int* sflag = reinterpret_cast<int*>(&om[NW + 3 * HP][0]);                 // H > 1: (emit | good << 1) per scenario of the block
  // tables staged per slot: with helper groups the flat zero-row list (the tail of the tables, 2 KB) is not used -- the
  // helpers walk the runs -- and stays in global memory: the two-slot set kernel then fits 5 CTAs on an SM instead of 4
  const int n_tab = H > 1 ? ax.o_zrow : ax.n_dbl;
  // ---- stage a program and its tables into a slot (cp.async, all in flight at once)
  auto stage = [&](unsigned char* slot, const void* pg_src, const double* tab_src) {
    const char* src = reinterpret_cast<const char*>(pg_src);
    char* dst = reinterpret_cast<char*>(slot);
    double* td = reinterpret_cast<double*>(slot + QPB);
    constexpr int NCH = (int)(sizeof(QpProg<BK>) / 16);
    for (int i = tix; i < NCH; i += NT) cp_async16(dst + 16 * i, src + 16 * i);
    if (tix == 0 && (sizeof(QpProg<BK>) % 16) != 0) cp_async8(dst + 16 * NCH, src + 16 * NCH);
    for (int i = tix; i < n_tab; i += NT) cp_async8(td + i, tab_src + i);
  };
  auto stage_plant = [&](unsigned char* slot) {              // (caller-owned arrays: behind pdl_wait)
    double* td = reinterpret_cast<double*>(slot + QPB);
    if (closed && !PL) {
      for (int i = tix; i < n * n; i += NT) cp_async8(td + n_tab + i, a.A_true + i);
      for (int i = tix; i < n * m; i += NT) cp_async8(td + n_tab + n * n + i, a.B_true + i);
    }
  };
  pdl_trigger();
  unsigned char* my_slot = smem_raw;
  if constexpr (NSLOT == 0) {
    stage(smem_raw, gpg, ax.tab);
  } else {
    constexpr int TILES = TPB / kDeferTile;
    const int64_t last_tile = (a.S + kDeferTile - 1) / kDeferTile - 1;
    const int64_t t0 = (int64_t)blockIdx.x * TILES;
    const int j0 = tile_prog[t0 < last_tile ? t0 : last_tile];
    stage(smem_raw, entries[j0].pg, entries[j0].tab);
    if constexpr (NSLOT == 2) {
      const int j1 = tile_prog[t0 + 1 < last_tile ? t0 + 1 : last_tile];
      if (j1 != j0) {                      // (uniform: one warp)
        stage(smem_raw + slot_bytes, entries[j1].pg, entries[j1].tab);
        if (lane >= 16) my_slot = smem_raw + slot_bytes;
      }
    }
  }
  cp_async_commit();
  pdl_wait();                                    // from here on: data earlier kernels of the stream may have written
  stage_plant(smem_raw);
  if constexpr (NSLOT == 2) stage_plant(smem_raw + slot_bytes);
  cp_async_commit();
  double* tabd = reinterpret_cast<double*>(my_slot + QPB);
  bool staged = false;
  const QpProg<BK>& pg = *reinterpret_cast<const QpProg<BK>*>(my_slot);
  const double* sXB = tabd + ax.o_XB;
  const double* sCZ = tabd + ax.o_CZ;
  const double* sK = tabd + ax.o_K;
  const double* sA = tabd + n_tab;
  const double* sB = sA + n * n;
  const double2* tt = reinterpret_cast<const double2*>(tabd + ax.o_tt);      // term table: (coef, idx | ent << 32)
  const int* zs = reinterpret_cast<const int*>(tabd + ax.o_zrun);           // zero runs: (first row, length) pairs
  // 16-byte zero stores need 16-byte aligned rows and an even batch (a pair of scenarios is in or out together)
  // (... and a row offset in bytes that fits 32 bits, for the one-instruction address)
  const bool zvec = dense && (reinterpret_cast<uintptr_t>(a.ze1) & 15u) == 0 && (a.ld & 1) == 0 && (a.S & 1) == 0 &&
                    (int64_t)(ax.n * (1 + ax.g1)) * a.ld * 8 < (int64_t)0x7fffffff;
  const int* zrow = reinterpret_cast<const int*>(tabd + ax.o_zrow);         // the zero rows as a flat list, two padded halves
  const int64_t nblk = (a.S + TPB - 1) / TPB;
  const unsigned long long* hint = reinterpret_cast<const unsigned long long*>(a.warm);
  unsigned long long* hint_w = reinterpret_cast<unsigned long long*>(a.warm);
  const unsigned half_mask = lane < 16 ? 0x0000ffffu : 0xffff0000u;
  const double* omc = &om[0][tid];                                          // this thread's column of om

  for (int64_t blk = blockIdx.x; blk < nblk; blk += (NSLOT == 0 ? (int64_t)gridDim.x : nblk)) {
    const int64_t s = blk * TPB + tid;
    const bool live = s < a.S;
    const int64_t sc = live ? s : a.S - 1;                 // dead lanes shadow the last scenario and write nothing
    bool emit = false, good = false;
    enum { kDefer = -2 };
    int status = kDefer;
    double omr[NW];
    double nrm2 = 0.0, cost = NAN;
    // ---- zero runs of the dense tube: odd warps before the solve, even warps behind it
    auto zero_runs = [&]() {
      double* base = a.ze1 + s;
#pragma unroll 1
      for (int r = 0; r < ax.n_zrun; ++r) {
        double* ptr = base + (int64_t)zs[2 * r] * LD;
#pragma unroll 4
        for (int c = zs[2 * r + 1]; c > 0; --c, ptr += LD) __stcs(ptr, 0.0);
      }
    };
    // Vector form (16-byte aligned rows): a thread keeps a 16-byte chunk (two scenarios) of the block's [entries x TPB
    // scenarios] slab and walks down the flat list of zero rows -- the first half of the CTA the first half of the list, the
    // second half the rest -- so a warp instruction stores 512 contiguous bytes.  The zero entries are disjoint from the
    // table's entries, so no ordering is needed, and the stores are DRIPPED: a few at a time between the stages of the solve
    // (`drip(k)`, k a multiple of 4, resumes where the previous call stopped).  Issued in one burst -- before or behind the
    // solve -- the step took solve + stores, 0.071 ms (profiles/r2_fast_v3_*); spread over the solve the stores ride along.
    // Four rows per trip: one 16-byte load of four row indices, one IMAD.WIDE per address (row * 8 ld fits 32 bits: zvec),
    // no remainder code (the list is padded to a multiple of 4) -- ~3 instructions per store where walking the (first row,
    // length) runs, 8 rows long on average, took 11 and made the dense step 74 % longer in instructions than the packed one.
    constexpr int CPR = TPB / 2;                                     // 16-byte chunks per entry row of the slab
    const int z_half = tid / CPR;
    const int64_t z_sv = blk * TPB + 2 * (tid % CPR);
    int z_pos = z_half * ax.n_zrow_half;                             // next entry of the zero-row list
    const int z_stop = z_pos + ax.n_zrow_half;
    if (!(zvec && z_sv < a.S) || H > 1) z_pos = z_stop;              // (H > 1: the helper groups store the zero rows)
    char* const z_base = reinterpret_cast<char*>(a.ze1 + z_sv);
    const int ld8 = (int)(LD * 8);
    auto drip = [&](int budget) {
      int k = z_stop - z_pos;
      k = k < budget ? k : budget;
#pragma unroll 2
      for (; k > 0; k -= 4, z_pos += 4) {
        const int4 r = *reinterpret_cast<const int4*>(zrow + z_pos);
        const double2 z2 = make_double2(0.0, 0.0);
        __stcs(reinterpret_cast<double2*>(z_base + (int64_t)r.x * ld8), z2);
        __stcs(reinterpret_cast<double2*>(z_base + (int64_t)r.y * ld8), z2);
        __stcs(reinterpret_cast<double2*>(z_base + (int64_t)r.z * ld8), z2);
        __stcs(reinterpret_cast<double2*>(z_base + (int64_t)r.w * ld8), z2);
      }
    };
    const bool zero_first = H == 1 && dense && !zvec && (((tid >> 5) + (int)blk) & 1);
    if (hq == 0) {
    // ---- inputs: parameters p = [xbar0 | e0] and the hint words (coalesced: lane = scenario)
    double w[2 * BK::NCOL2];                               // w = [1 | p | |p| | general atoms] (+ a zero pad)
    w[0] = 1.0;
    if constexpr (2 * BK::NCOL2 > NCOL) w[2 * BK::NCOL2 - 1] = 0.0;
    unsigned long long hw[G];
#pragma unroll
    for (int g = 0; g < G; ++g) hw[g] = hint[(int64_t)g * LD + sc];
    bool finite = true;
#pragma unroll
    for (int j = 0; j < HP; ++j) {
      double xv = 0.0, ev = 0.0;
      if (j < n) { xv = a.xbar0[(int64_t)j * LD + sc]; ev = a.e0[(int64_t)j * LD + sc]; }
      w[1 + j] = xv;
      w[1 + HP + j] = ev;
      w[1 + NPAR + j] = fabs(xv);
      w[1 + NPAR + HP + j] = fabs(ev);
      finite = finite && (fabs(xv) < 1e300) && (fabs(ev) < 1e300);
    }
    // the closed-loop update's inputs (x, noise) are fetched now, into this thread's column of om: every load of the step is
    // in flight before the first store is issued (a load queued behind the step's ~300 MB of stores waits microseconds)
    if (closed) {
#pragma unroll
      for (int i = 0; i < HP; ++i)
        if (i < n) {
          cp_async8(&om[OM_X + i][tid], a.x + (int64_t)i * LD + sc);
          if (a.noise) cp_async8(&om[OM_NS + i][tid], a.noise + (int64_t)i * LD + sc);
        }
      cp_async_commit();
      if constexpr (PL) {
        const int nm = n + m;
        for (int r = 0; r < n * nm; ++r) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.AB_true + (int64_t)r * LD + sc));
      }
    }
    if (!staged) {
      cp_async_wait<0>();
      __syncthreads();
      staged = true;
    }
    if (zero_first && live) zero_runs();
    drip(24);

    eval_atoms<BK>(pg, w);
    double q[NZ];
    eval_q<BK>(pg, w, q);
    drip(8);
    bool param_ok = true;
    {
      int bad_rows = 0;                                     // (two rows per trip: four independent fma chains)
#pragma unroll 1
      for (int i = 0; i < pg.nchk; i += 2) {
        bad_rows |= param_rows_violated<BK, 2>(pg, i, w) ? 1 : 0;
        drip(4);
      }
      param_ok = bad_rows == 0;
    }
    const double c0 = cost_const<BK>(pg, w);

    bool valid = true;
#pragma unroll
    for (int g = 0; g < G; ++g) valid = valid && (hw[g] & kCodeValid);
    const bool fresh = !(hw[0] & kCodeValid) || (hw[0] & kCodeFresh);
    unsigned long long code[G];
#pragma unroll
    for (int g = 0; g < G; ++g) code[g] = hw[g] & ~(kCodeValid | kCodeFresh);
    if (!finite) status = TZ_STATUS_NONFINITE;
    else if (!param_ok) status = TZ_STATUS_INFEASIBLE;
    Cert2Result res;
    res.x[0] = res.x[1] = 0.0;
    res.obj = 0.0;
    res.verdict = kCertUndecided;
    if (__any_sync(0xffffffffu, status == kDefer && valid)) {
      res = certify2<BK>(pg, w, q, code, [&]() { drip(12); });
      if (status == kDefer && valid && res.verdict == kCertOk) status = TZ_STATUS_OK;
    }
    // a hint that does not certify: is the program infeasible outright (singleton presolve, exact)?  Otherwise defer.
    if (__any_sync(0xffffffffu, status == kDefer && valid)) {
      const bool inf = singleton_infeasible2<BK>(pg, w);
      if (status == kDefer && valid && inf) status = TZ_STATUS_INFEASIBLE;
    }
    // ---- deferral, per 16-scenario tile
    const unsigned dmask = __ballot_sync(0xffffffffu, live && status == kDefer);
    const bool deferred = (dmask & half_mask) != 0u;
    if (deferred && (lane & 15) == 0 && live) {
      const int slot = atomicAdd(a.defer, 1);
      if (slot >= 0 && slot < (a.S + kDeferTile - 1) / kDeferTile) a.defer_list[slot] = (int32_t)(s / kDeferTile);
    }
    emit = live && !deferred;
    good = status == TZ_STATUS_OK;
    drip(16);
    if (emit) {
      // ---- hints: rows [0, G) the active set for the next step, rows [G, 2G) the active set of the run's first step
#pragma unroll
      for (int g = 0; g < G; ++g) {
        unsigned long long wnext = 0ull;
        if (good) {
          wnext = code[g] | kCodeValid;
          if (fresh) hint_w[(int64_t)(G + g) * LD + s] = wnext;
        } else if (a.x_restart != nullptr) {
          const unsigned long long h0 = hint[(int64_t)(G + g) * LD + s];
          wnext = (h0 & kCodeValid) ? (h0 | kCodeFresh) : 0ull;
        }
        hint_w[(int64_t)g * LD + s] = wnext;
      }
      // ---- om = [1 | v | p | centre of Ze[1]]
      omr[0] = 1.0;
#pragma unroll
      for (int j = 0; j < NZ; ++j) omr[BK::OM_V + j] = (j < nv) ? (good ? pg.D[j] * res.x[j] : NAN) : 0.0;
#pragma unroll
      for (int j = 0; j < NPAR; ++j) omr[BK::OM_P + j] = w[1 + j];
      if (good) cost = fma(res.obj, pg.cinv, c0);
      else if (status == TZ_STATUS_INFEASIBLE) cost = INFINITY;      // cvxpy returns +inf for an infeasible Minimize (:374)
#pragma unroll
      for (int j = 0; j < NW; ++j) om[j][tid] = omr[j];
#pragma unroll 2
      for (int r = 0; r < n; ++r) {
        const double* row = sCZ + r * NW;
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < NW; ++j) acc = fma(row[j], omr[j], acc);
        om[BK::OM_C + r][tid] = acc;
      }
      drip(16);
    }
    if constexpr (H > 1) sflag[tid] = (emit ? 1 : 0) | (good ? 2 : 0);
    } else {
      if (!staged) {                                       // helper groups: the staging barrier of the CTA
        cp_async_wait<0>();
        __syncthreads();
        staged = true;
      }
      // while group 0 solves, the helper groups store the structural zeros of the block (whole runs each; the zeros do not
      // depend on the solve, and a deferred tile is rewritten by step_kernel anyway)
      if (dense && live) {
        double* base = a.ze1 + s;
#pragma unroll 1
        for (int r = hq - 1; r < ax.n_zrun; r += H - 1) {
          double* ptr = base + (int64_t)zs[2 * r] * LD;
#pragma unroll 4
          for (int c = zs[2 * r + 1]; c > 0; --c, ptr += LD) __stcs(ptr, 0.0);
        }
      }
    }
    if constexpr (H > 1) {
      __syncthreads();                                     // om and the flags of the block are complete
      if (hq > 0) {
        const int f = sflag[tid];
        emit = (f & 1) != 0;
        good = (f & 2) != 0;
        if (emit) {
#pragma unroll
          for (int j = 0; j < NW; ++j) omr[j] = omc[j * TPB];
        }
      }
    }
    if (emit) {
      // (H == 1: om columns are thread-private, no barrier)
      // ---- Ze[1].Z at the optimum (examples/2.pulley_sim.py:96): the entries of the term table
      if (a.ze1 != nullptr) {
        double* base = a.ze1 + s;
        if (sp.tube_packed) {
          double* ptr = base + (int64_t)hq * LD;
#pragma unroll 4
          for (int i = hq; i < ax.n_nz; i += H, ptr += H * LD) {
            const double2 e = tt[i];
            __stcs(ptr, e.x * omc[(int)(__double_as_longlong(e.y) & 0xffffffffll) * TPB]);
          }
        } else {
          if constexpr (H == 1) {
            if (!zero_first && !zvec) zero_runs();
          }
#pragma unroll 4
          for (int i = hq; i < ax.n_nz; i += H) {
            const double2 e = tt[i];
            const long long ie = __double_as_longlong(e.y);
            __stcs(base + (ie >> 32) * LD, e.x * omc[(int)(ie & 0xffffffffll) * TPB]);
          }
        }
      }
      // ---- nominal trajectory xbar_0..xbar_N = XB om  (tzddpc/tzddpc.py:166-170); xbar_1 is kept for the update
      double xb1[HP];
#pragma unroll
      for (int i = 0; i < HP; ++i) xb1[i] = 0.0;
      auto xb_row = [&](int i) {
        const double* row = sXB + i * NW;
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < NW; ++j) acc = fma(row[j], omr[j], acc);
        if (a.xbar_traj != nullptr) a.xbar_traj[(int64_t)i * LD + s] = acc;
        return acc;
      };
      if constexpr (H == 1) {
        if (a.xbar_traj != nullptr) {
#pragma unroll 2
          for (int i = 0; i < n; ++i) (void)xb_row(i);
        }
        drip(16);
        if (a.xbar_traj != nullptr || closed) {
#pragma unroll
          for (int k = 0; k < HP; ++k)
            if (k < n) xb1[k] = xb_row(n + k);
        }
        drip(16);
        if (a.xbar_traj != nullptr) {
#pragma unroll 2
          for (int i = 2 * n; i < (ax.N + 1) * n; ++i) (void)xb_row(i);
        }
      } else {
        // rows [n, 2n) (xbar_1: needed by the update) stay with group 0, the others are shared by the helper groups
        if (hq == 0 && (a.xbar_traj != nullptr || closed)) {
#pragma unroll
          for (int k = 0; k < HP; ++k)
            if (k < n) xb1[k] = xb_row(n + k);
        }
        if (a.xbar_traj != nullptr && hq > 0) {
#pragma unroll 1
          for (int i = hq - 1; i < (ax.N + 1) * n; i += H - 1)
            if (i < n || i >= 2 * n) (void)xb_row(i);
        }
      }
      if (hq == 0) {
      if (a.v != nullptr)
        for (int j = 0; j < nv; ++j) a.v[(int64_t)j * LD + s] = omc[(BK::OM_V + j) * TPB];
      if (a.status) a.status[s] = status;
      if (a.iters) a.iters[s] = 0;
      if (a.cost) a.cost[s] = cost;
      // ---- closed-loop update (examples/2.pulley_sim.py:90-94)
      if (closed) {
        double us[kMaxM];
#pragma unroll
        for (int j = 0; j < kMaxM; ++j) {
          double acc = 0.0;
          if (j < m) {
            acc = omr[BK::OM_V + (j < NZ ? j : 0)];                                  // v[0]
#pragma unroll
            for (int i = 0; i < HP; ++i)
              if (i < n) acc = fma(sK[j * n + i], omr[BK::OM_P + HP + i], acc);
            if (a.u_out) a.u_out[(int64_t)j * LD + s] = good ? acc : NAN;
          }
          us[j] = acc;                                                              // u = K e + v[0]
        }
        double xo[HP];
        cp_async_wait<0>();
#pragma unroll
        for (int i = 0; i < HP; ++i) xo[i] = (i < n) ? omc[(OM_X + i) * TPB] : 0.0;
#pragma unroll
        for (int i = 0; i < HP; ++i) {
          if (i < n) {
            double acc = a.noise ? omc[(OM_NS + i) * TPB] : 0.0;
            if constexpr (PL) {
              const double* ab = a.AB_true + (int64_t)i * (n + m) * LD + s;        // row i of this scenario's [A_true B_true]
#pragma unroll
              for (int k = 0; k < HP; ++k)
                if (k < n) acc = fma(ab[(int64_t)k * LD], xo[k], acc);
#pragma unroll
              for (int k = 0; k < kMaxM; ++k)
                if (k < m) acc = fma(ab[(int64_t)(n + k) * LD], us[k], acc);
            } else {
#pragma unroll
              for (int k = 0; k < HP; ++k)
                if (k < n) acc = fma(sA[i * n + k], xo[k], acc);
#pragma unroll
              for (int k = 0; k < kMaxM; ++k)
                if (k < m) acc = fma(sB[i * m + k], us[k], acc);
            }
            double xb = xb1[i];                                                      // xbar+ = xbar_traj[1]
            double en = acc - xb;                                                    // e+ = x+ - xbar+
            if (!good) {
              // a scenario whose step failed keeps its state, or -- the reference raises and the run ends
              // (tzddpc/tzddpc.py:374-375) -- starts a new run from x_restart: x = xbar = x_restart, e = 0
              const double xr = a.x_restart ? a.x_restart[(int64_t)i * LD + s] : xo[i];
              acc = xr;
              xb = a.x_restart ? xr : omr[BK::OM_P + i];
              en = a.x_restart ? 0.0 : omr[BK::OM_P + HP + i];
            }
            nrm2 = fma(acc, acc, nrm2);
            a.x[(int64_t)i * LD + s] = acc;                                          // x+ = A x + B u + w
            a.xbar[(int64_t)i * LD + s] = xb;
            a.e[(int64_t)i * LD + s] = en;
          }
        }
      }
      }      // hq == 0
    }
    drip(1 << 20);      // whatever is left of this thread's share of the zero entries (every thread: the shares cover other lanes' scenarios)
    // ---- closed-loop statistics: warp reduction, one atomic per statistic and warp
    if (a.stats != nullptr && closed && hq == 0) {
      const bool eg = emit && good;
      double s0 = eg ? sqrt(nrm2) : 0.0, s1 = eg ? nrm2 : 0.0, s2 = eg ? cost : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      }
      const unsigned binf = __ballot_sync(0xffffffffu, emit && status == TZ_STATUS_INFEASIBLE);
      const unsigned bnf = __ballot_sync(0xffffffffu, emit && status == TZ_STATUS_NONFINITE);
      const unsigned bem = __ballot_sync(0xffffffffu, emit);
      if (lane == 0 && bem) {
        if (s0 != 0.0) atomicAdd(a.stats + 0, s0);
        if (s1 != 0.0) atomicAdd(a.stats + 1, s1);
        if (s2 != 0.0) atomicAdd(a.stats + 2, s2);
        if (binf) atomicAdd(a.stats + 3, (double)__popc(binf));
        if (bnf) atomicAdd(a.stats + 6, (double)__popc(bnf));
        atomicAdd(a.stats + 7, (double)__popc(bem));
      }
    }
    if constexpr (H > 1) __syncthreads();                  // the helper groups are done with om before the next block overwrites it
  }
  if (!staged) cp_async_wait<0>();
}

template <class BK>
size_t fast_slot_bytes(const TzProgram* p, int h = 1) {
  const size_t qpb = (sizeof(QpProg<BK>) + 15) & ~(size_t)15;
  if (h <= 1) return qpb + p->smem_tab;
  // helper-group kernels: [tables up to the flat zero-row list | A_true | B_true]
  const size_t tab = ((size_t)p->aux.o_zrow + (size_t)p->aux.n * p->aux.n + (size_t)p->aux.n * p->aux.m) * sizeof(double);
  return qpb + ((tab + 15) & ~(size_t)15);
}

// CTAs of `tpb` threads that are resident on one SM: registers (launch bounds) and shared memory (227 KB, 1 KB per CTA reserved)
template <class BK>
int fast_resident(const TzProgram* p, int tpb, int nslot, int h = 1) {
  const size_t per_cta = (nslot > 1 ? nslot : 1) * fast_slot_bytes<BK>(p, h) + sizeof(double) * (BK::NW + 3 * (BK::NPAR / 2)) * tpb + 4 * tpb + 1024;
  const int by_smem = (int)((size_t)227 * 1024 / per_cta);
  const int by_regs = fast_ctas_per_sm(tpb * h);
  return by_smem < by_regs ? (by_smem > 0 ? by_smem : 1) : by_regs;
}

template <class BK, int TPB, int NSLOT, int H = 1>
int launch_fast_tpb(const TzProgram* p, const SolverParams& sp, const StepArgs& a, const SetEntry* entries, const int32_t* tile_prog,
                    cudaStream_t st) {
  const size_t slot = fast_slot_bytes<BK>(p, H);
  constexpr size_t om_bytes = sizeof(double) * (BK::NW + 3 * (BK::NPAR / 2)) * TPB + sizeof(int) * TPB;      // om + the H > 1 flags
  const size_t smem = (NSLOT > 1 ? NSLOT : 1) * slot + om_bytes;
  const size_t smem_max = (NSLOT > 1 ? NSLOT : 1) * (((sizeof(QpProg<BK>) + 15) & ~(size_t)15) + kMaxTabBytes) + om_bytes;
  const int64_t nblk = (a.S + TPB - 1) / TPB;
  const int64_t wave = (int64_t)p->num_sms * fast_resident<BK>(p, TPB, NSLOT, H);
  const unsigned grid = (unsigned)(NSLOT == 0 ? (nblk < wave ? nblk : wave) : nblk);
  return with_plant(a, [&](auto pl) {
    constexpr auto kernel = fast_step_kernel<BK, TPB, NSLOT, H, decltype(pl)::value>;
    static std::atomic<unsigned long long> configured{0ull};
    if (const int rc = ensure_dynamic_smem(kernel, (int)smem_max, p->device, configured)) return rc;
    TZ_CUDA(launch_kernel(kernel, grid, TPB * H, smem, st, pdl_enabled(a.S),
                          reinterpret_cast<const QpProg<BK>*>(p->packed_dev), p->aux, sp, a, entries, tile_prog, (int)slot));
    return TZ_OK;
  });
}

// CTA size by batch size, measured on 148 SMs (profiles/r2_fast_cta_size_sweep.txt; ms per dense 5-dim step):
//   65,536 scenarios:  32: 0.077   64: 0.0626   96: 0.0645   128: 0.0649   160: 0.0632   224: 0.0621   256: 0.0598   512: 0.0644
//   32,768:  64: 0.0377  128: 0.0390  256: 0.0412        16,384:  64: 0.0319  128: 0.0318  256: 0.0380        8,192:  64: 0.0293  128: 0.0307
// Two effects: a CTA's stores of one output row are TPB * 8 contiguous bytes (256 threads: 2 KB runs, kinder to DRAM than the
// 1 KB of 128), and a batch below ~1.5 scenarios per thread slot of the wave wants many small CTAs so that every SM has work.
// Beyond one wave of 256-thread CTAs the persistent loop takes over; the size that leaves the fullest SM least full is used.
template <class BK>
int launch_fast(const TzProgram* p, const SolverParams& sp, const StepArgs& a, cudaStream_t st) {
  int tpb = 0;
  if (const char* e = getenv("TZDDPC_FAST_TPB")) tpb = atoi(e);      // tuning knob (read per launch, no state): force the CTA size
  if (tpb == 0) {
    const int64_t sms = p->num_sms;
    if (a.S <= sms * 512) tpb = a.S >= sms * 384 ? 256 : 64;
    else {
      int64_t best = INT64_MAX;
      for (int t = 256; t >= 64; t >>= 1) {
        const int64_t ctas = (a.S + t - 1) / t, per_sm = (ctas + sms - 1) / sms, cap = fast_resident<BK>(p, t, 0);
        const int64_t rounds = (per_sm + cap - 1) / cap;
        const int64_t load = (int64_t)t * ((per_sm + rounds - 1) / rounds) * rounds;
        if (load < best) { best = load; tpb = t; }
      }
    }
  }
  // helper groups (H = 2: a second thread per scenario stores the zeros while the first one solves, then both share the tube
  // and trajectory rows): 8,192 scenarios 0.0298 -> 0.0232 ms per step, 16,384: 0.0322 -> 0.0272, 32,768: no gain (0.0394
  // against 0.0383) -- below one scenario per two thread slots of the chip the step is one warp's latency, above it the
  // helpers take issue slots from other scenarios' solves
  int h = (tpb == 64 && a.S <= (int64_t)p->num_sms * 128) ? 2 : 1;
  if (const char* e = getenv("TZDDPC_FAST_H")) h = atoi(e);        // tuning knob: helper groups per scenario
  if (h > 1) {
    if (tpb == 64 && h == 2) return launch_fast_tpb<BK, 64, 0, 2>(p, sp, a, nullptr, nullptr, st);
    if (tpb == 64 && h == 4) return launch_fast_tpb<BK, 64, 0, 4>(p, sp, a, nullptr, nullptr, st);
  }
  switch (tpb) {
    case 256: return launch_fast_tpb<BK, 256, 0>(p, sp, a, nullptr, nullptr, st);
    case 128: return launch_fast_tpb<BK, 128, 0>(p, sp, a, nullptr, nullptr, st);
    case 32: return launch_fast_tpb<BK, 32, 0>(p, sp, a, nullptr, nullptr, st);
    default: return launch_fast_tpb<BK, 64, 0>(p, sp, a, nullptr, nullptr, st);
  }
}

// Program set: `block` = the largest of 128 / 64 / 32 that divides every program's first scenario (so that a CTA's block of
// scenarios lies within one program), or 16: two program slots per one-warp CTA.
template <class BK>
int launch_fast_set(const TzProgram* p0, const SolverParams& sp, const StepArgs& a, const SetEntry* entries, const int32_t* tile_prog,
                    int block, cudaStream_t st) {
  // small blocks keep few warps on an SM (two 16.5 KB program slots per one-warp CTA: 5 CTAs): a helper group per CTA
  // (zeros during the solve, half of the output rows) -- 4,096 data sets x 16 scenarios 0.109 -> 0.100 ms per step,
  // 1,024 x 64: 0.093 -> 0.075
  int h = 2;
  if (const char* e = getenv("TZDDPC_FAST_SET_H")) h = atoi(e);      // tuning knob: helper groups in the small-block set kernels
  if (block >= 128) return launch_fast_tpb<BK, 128, 1>(p0, sp, a, entries, tile_prog, st);
  if (block >= 64) return h == 2 ? launch_fast_tpb<BK, 64, 1, 2>(p0, sp, a, entries, tile_prog, st)
                                 : launch_fast_tpb<BK, 64, 1>(p0, sp, a, entries, tile_prog, st);
  if (block >= 32) return h == 2 ? launch_fast_tpb<BK, 32, 1, 2>(p0, sp, a, entries, tile_prog, st)
                                 : launch_fast_tpb<BK, 32, 1>(p0, sp, a, entries, tile_prog, st);
  return h == 2 ? launch_fast_tpb<BK, 32, 2, 2>(p0, sp, a, entries, tile_prog, st)
                : launch_fast_tpb<BK, 32, 2>(p0, sp, a, entries, tile_prog, st);
}

}  // namespace tz
