// Stand-alone batched zonotope kernels (AoS: one zonotope = one contiguous n x (1+g) block).
//   tz_interval_hull   Zonotope.interval                      tzddpc/tzddpc.py:191-197
//   tz_reach_step      MatrixZonotope * Zonotope (+ Zonotope)  tzddpc/tzddpc.py:175-176,181,185,205
//   tz_girard_reduce   Zonotope.reduce / MatrixZonotope.reduce tzddpc/tzddpc.py:126-128,
//                                                              examples/1.double_integrator_sim.py:170
// All three are HBM-bound (1-2 flop per byte): a warp / CTA owns one zonotope, rows are
// contiguous so every global access is a full-line coalesced access, the generator block is
// staged once in shared memory and never re-read from HBM.
#include <cstdlib>
#include <cstring>

#include "tz_common.cuh"

namespace tz {

// ---------------------------------------------------------------------------------------
// interval hull: one warp per zonotope; lanes stride the columns of a row, shuffle-reduce.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) hull_kernel(int64_t S, int n, int g, const double* __restrict__ Z,
                                                   double* __restrict__ lo, double* __restrict__ hi) {
  const int lane = threadIdx.x & 31;
  const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= S) return;
  const int ld = 1 + g;
  const double* Zs = Z + s * (int64_t)n * ld;
  for (int r = 0; r < n; ++r) {
    const double* row = Zs + (int64_t)r * ld;
    double acc = 0.0;
    for (int j = 1 + lane; j < ld; j += 32) acc += fabs(__ldcs(row + j));
    acc = warp_sum(acc);
    if (lane == 0) {
      const double c = row[0];
      lo[s * n + r] = c - acc;
      hi[s * n + r] = c + acc;
    }
  }
}

// ---------------------------------------------------------------------------------------
// MatrixZonotope x Zonotope (+ W): one CTA per scenario.
//   out[r][b*(1+g) + j] = sum_k M_b[r][k] Z[k][j],  M_0 = C, M_b = G_b     (b = 0..N)
//   out[:,0] += W[:,0];  out[:, (N+1)(1+g) + t] = W[:, 1+t]
// The (N+1) small matrices are staged in shared memory; Z columns are read coalesced and
// each thread produces the n rows of one output column (n independent FMA chains).
// ---------------------------------------------------------------------------------------
template <int NMAX>
__global__ void __launch_bounds__(256) reach_kernel(int n, int p, int N, int g, int gW, const double* __restrict__ C,
                                                    const double* __restrict__ Gm, int per_scenario,
                                                    const double* __restrict__ Z, const double* __restrict__ W,
                                                    double* __restrict__ Zout) {
  extern __shared__ double sm[];                  // (N+1) * n * p
  const int64_t s = blockIdx.x;
  const int np_ = n * p;
  const double* Cs = C + (per_scenario ? s * (int64_t)np_ : 0);
  const double* Gs = Gm + (per_scenario ? s * (int64_t)N * np_ : 0);
  for (int i = threadIdx.x; i < np_; i += blockDim.x) sm[i] = Cs[i];
  for (int i = threadIdx.x; i < N * np_; i += blockDim.x) sm[np_ + i] = Gs[i];
  __syncthreads();
  const int ldz = 1 + g;
  const int ldo = (N + 1) * ldz + gW;
  const double* Zs = Z + s * (int64_t)p * ldz;
  double* Os = Zout + s * (int64_t)n * ldo;
  const int total = (N + 1) * ldz;
  for (int col = threadIdx.x; col < total; col += blockDim.x) {
    const int b = col / ldz, j = col - b * ldz;
    const double* M = sm + (size_t)b * np_;
    double acc[NMAX];
#pragma unroll
    for (int r = 0; r < NMAX; ++r) acc[r] = 0.0;
    for (int k = 0; k < p; ++k) {
      const double zk = Zs[(int64_t)k * ldz + j];
#pragma unroll
      for (int r = 0; r < NMAX; ++r)
        if (r < n) acc[r] = fma(M[r * p + k], zk, acc[r]);
    }
    if (col == 0 && W != nullptr) {
#pragma unroll
      for (int r = 0; r < NMAX; ++r)
        if (r < n) acc[r] += W[(int64_t)r * (1 + gW)];
    }
#pragma unroll
    for (int r = 0; r < NMAX; ++r)
      if (r < n) __stcs(Os + (int64_t)r * ldo + col, acc[r]);
  }
  for (int t = threadIdx.x; t < gW * n; t += blockDim.x) {
    const int r = t / gW, c = t - r * gW;
    Os[(int64_t)r * ldo + total + c] = W[(int64_t)r * (1 + gW) + 1 + c];
  }
}

// Fast path for the dimensions of the shipped systems (NN = n, PP = p exactly): the generic kernel above spends ~370 warp
// instructions per output column (predicated NMAX-wide loops, one scalar shared load per FMA, an integer division per
// column) and is ISSUE-bound at 64 % (profiles/r2_reach_girard_ncu.txt).  Here a thread owns column j of Z, keeps its PP
// entries in registers and walks over the blocks b = 0..N: per output column NN*PP FMAs, NN*PP/2 16-byte broadcast loads
// of the transposed, padded matrices and NN streaming stores -- the kernel becomes what it should be, a stream of writes.
// Threads are arranged (column, block group) so that short zonotopes (1+g < 256) still fill the CTA.
template <int NN, int PP>
__global__ void __launch_bounds__(256) reach_kernel_fast(int N, int g, int gW, const double* __restrict__ C,
                                                         const double* __restrict__ Gm, int per_scenario,
                                                         const double* __restrict__ Z, const double* __restrict__ W,
                                                         double* __restrict__ Zout, int jthreads) {
  constexpr int NNP = NN + (NN & 1);               // padded row count: 16-byte aligned pairs
  constexpr int MS = PP * NNP;                     // doubles per staged matrix, layout [k][r]
  extern __shared__ __align__(16) double smf[];    // (N+1) * MS
  const int64_t s = blockIdx.x;
  const double* Cs = C + (per_scenario ? s * (int64_t)(NN * PP) : 0);
  const double* Gs = Gm + (per_scenario ? s * (int64_t)N * (NN * PP) : 0);
  for (int i = threadIdx.x; i < (N + 1) * MS; i += blockDim.x) {
    const int b = i / MS, e = i - b * MS, k = e / NNP, r = e - k * NNP;
    double v = 0.0;
    if (r < NN) v = b == 0 ? Cs[r * PP + k] : Gs[(int64_t)(b - 1) * (NN * PP) + r * PP + k];
    smf[i] = v;
  }
  __syncthreads();
  const int ldz = 1 + g;
  const int64_t ldo = (int64_t)(N + 1) * ldz + gW;
  const double* Zs = Z + s * (int64_t)PP * ldz;
  double* Os = Zout + s * (int64_t)NN * ldo;
  const int tj = threadIdx.x % jthreads, tb = threadIdx.x / jthreads, bgroups = blockDim.x / jthreads;
  for (int j = tj; j < ldz; j += jthreads) {
    double z[PP];
#pragma unroll
    for (int k = 0; k < PP; ++k) z[k] = __ldg(Zs + (int64_t)k * ldz + j);
    for (int b = tb; b <= N; b += bgroups) {
      const double2* M2 = reinterpret_cast<const double2*>(smf + (size_t)b * MS);
      double acc[NNP];
#pragma unroll
      for (int r = 0; r < NNP; ++r) acc[r] = 0.0;
#pragma unroll
      for (int k = 0; k < PP; ++k) {
#pragma unroll
        for (int r2 = 0; r2 < NNP / 2; ++r2) {
          const double2 mv = M2[k * (NNP / 2) + r2];
          acc[2 * r2] = fma(mv.x, z[k], acc[2 * r2]);
          acc[2 * r2 + 1] = fma(mv.y, z[k], acc[2 * r2 + 1]);
        }
      }
      if (b == 0 && j == 0 && W != nullptr) {
#pragma unroll
        for (int r = 0; r < NN; ++r) acc[r] += W[(int64_t)r * (1 + gW)];
      }
      double* o = Os + (int64_t)b * ldz + j;
#pragma unroll
      for (int r = 0; r < NN; ++r) __stcs(o + (int64_t)r * ldo, acc[r]);
    }
  }
  for (int t = threadIdx.x; t < gW * NN; t += blockDim.x) {
    const int r = t / gW, c = t - r * gW;
    Os[(int64_t)r * ldo + (int64_t)(N + 1) * ldz + c] = W[(int64_t)r * (1 + gW) + 1 + c];
  }
}

template <int NN, int PP>
static int launch_reach_fast(int64_t S, int N, int g, int gW, const double* C, const double* Gm, int per_scenario,
                             const double* Z, const double* W, double* Zout, cudaStream_t st) {
  constexpr int NNP = NN + (NN & 1);
  const size_t smem = (size_t)(N + 1) * PP * NNP * sizeof(double);
  TZ_REQUIRE(smem <= 200 * 1024, "matrix zonotope too large for shared memory");
  if (smem + 8192 > 48 * 1024)
    TZ_CUDA(cudaFuncSetAttribute(reach_kernel_fast<NN, PP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int jthreads = 32;
  while (jthreads < 256 && jthreads < 1 + g) jthreads *= 2;       // a power of two >= 1+g (capped): column threads
  reach_kernel_fast<NN, PP><<<(unsigned)S, 256, smem, st>>>(N, g, gW, C, Gm, per_scenario, Z, W, Zout, jthreads);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

// ---------------------------------------------------------------------------------------
// Girard reduction: one CTA per zonotope, generator block in shared memory.
//   metric per column -> 64-bit radix select of the nReduced smallest (ties: lowest index)
//   -> box of the selected columns -> stable compaction of the kept columns + diag(d).
// ---------------------------------------------------------------------------------------
constexpr int kGirardThreads = 256;
constexpr int kGirardMaxDim = 128;    // vectorised matrix zonotopes reach n*(n+m) = 96

__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_tot, int& total) {
  // blockDim.x == kGirardThreads; returns the exclusive prefix of v, total = block sum
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  int base = 0, tot = 0;
  for (int w = 0; w < kGirardThreads / 32; ++w) {
    const int t = warp_tot[w];
    if (w < wid) base += t;
    tot += t;
  }
  __syncthreads();
  total = tot;
  return base + inc - v;
}

// Column source of girard_block: G(r, j) is entry r of generator j.  ResidentCols reads a block held in memory;
// ProductCols (below, tube_rollout_recompute_kernel) evaluates the entry from the factors of the block instead.
// kCountFromRegisters: loc[d] with a run-time d puts loc[] in 32 bytes of local memory; ProductCols selects the count
// from registers instead.  ResidentCols keeps the indexed read, so girard_kernel and tube_rollout_kernel compile as before.
struct ResidentCols {
  static constexpr bool kCountFromRegisters = false;
  const double* __restrict__ G;
  int64_t ldg;
  __device__ __forceinline__ double operator()(int r, int j) const { return G[(int64_t)r * ldg + j]; }
};

// Girard reduction of the generator block G (n x g; a ResidentCols block in shared memory, or in global memory that
// stays in L2 between the metric pass and the box / compaction passes, or a ProductCols block) of one zonotope by one CTA.
// The metric pass reads every column once, the box pass the reduced ones and the compaction the kept ones.
// Writes the reduced generators to out[r * ldo + j] (global or shared), zero-pads up to gout_cap, returns the
// number of generators written (negative: gout_cap too small).  key / flag: g-element scratch in shared memory.
//   metric per column -> MSB-first radix select of the n_red-th smallest key (stops as soon as a digit bucket is
//   consumed whole) -> ties by lowest index -> box of the selected columns -> stable compaction of the kept ones.
// Every thread owns a CONTIGUOUS range of columns, so that ranks (ties, output positions) need one block scan each.
template <class Cols>
__device__ int girard_block(int n, int g, double order, int metric, const Cols G, unsigned long long* __restrict__ key,
                            unsigned char* __restrict__ flag, double* __restrict__ out, int64_t ldo, int gout_cap) {
  __shared__ int hist[256];
  __shared__ int warp_tot[kGirardThreads / 32];
  __shared__ unsigned long long sel_prefix;
  __shared__ int sel_remaining, sel_done;
  __shared__ double dbox[kGirardMaxDim];
  __shared__ double red[kGirardThreads / 32][8];
  __shared__ unsigned bits[kGirardThreads / 32][4];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int per = (g + kGirardThreads - 1) / kGirardThreads;       // columns per thread (contiguous range)
  const int j0 = min(tid * per, g), j1 = min(j0 + per, g);
  // metric (rows accumulated r = 0..n-1, exactly as oracle/zono.py:_girard_metric) and zero filter
  // Two columns x eight rows of loads are issued before any of them is consumed: with one dependent load per thread in
  // flight the pass was latency-bound at ~1.5 TB/s (Little's law: 1,024 threads x 8 bytes per SM; profiles/r2_reach_girard_ncu.txt).
  // Rows beyond n read as 0, which changes neither the sums nor the maximum (bit-exact against the row-by-row loop).
  int nnz_local = 0;
  unsigned long long kand = ~0ull, kor = 0ull;
  for (int ja = tid; ja < g; ja += 2 * kGirardThreads) {
    const int jc = ja + kGirardThreads;
    const bool hc = jc < g;
    double sumA = 0.0, mxA = 0.0, sumC = 0.0, mxC = 0.0;
    bool nzA = false, nzC = false;
    for (int r0 = 0; r0 < n; r0 += 8) {
      double a[8], c[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool in = r0 + i < n;
        a[i] = in ? fabs(G(r0 + i, ja)) : 0.0;
        c[i] = (in && hc) ? fabs(G(r0 + i, jc)) : 0.0;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        nzA = nzA || (a[i] != 0.0);
        nzC = nzC || (c[i] != 0.0);
        if (metric == 2) {       // no FMA contraction: selection must match the oracle bit for bit
          sumA = __dadd_rn(sumA, __dmul_rn(a[i], a[i]));
          sumC = __dadd_rn(sumC, __dmul_rn(c[i], c[i]));
        } else {
          sumA += a[i];
          sumC += c[i];
        }
        mxA = fmax(mxA, a[i]);
        mxC = fmax(mxC, c[i]);
      }
    }
    const double hA = (metric == 0) ? (sumA - mxA) : sumA;
    const unsigned long long kA = (unsigned long long)__double_as_longlong(hA);    // h >= 0: bit pattern is order-preserving
    key[ja] = kA;
    flag[ja] = nzA ? 1 : 0;
    if (nzA) { ++nnz_local; kand &= kA; kor |= kA; }
    if (hc) {
      const double hC = (metric == 0) ? (sumC - mxC) : sumC;
      const unsigned long long kC = (unsigned long long)__double_as_longlong(hC);
      key[jc] = kC;
      flag[jc] = nzC ? 1 : 0;
      if (nzC) { ++nnz_local; kand &= kC; kor |= kC; }
    }
  }
  {  // bits shared by all active keys of the zonotope (block-wide AND / OR): the select skips the passes over them
    const unsigned ah = __reduce_and_sync(0xffffffffu, (unsigned)(kand >> 32)), al = __reduce_and_sync(0xffffffffu, (unsigned)kand);
    const unsigned oh = __reduce_or_sync(0xffffffffu, (unsigned)(kor >> 32)), ol = __reduce_or_sync(0xffffffffu, (unsigned)kor);
    if (lane == 0) { bits[wid][0] = ah; bits[wid][1] = al; bits[wid][2] = oh; bits[wid][3] = ol; }
  }
  int gnz;
  (void)block_exclusive_scan(nnz_local, warp_tot, gnz);
  const bool do_reduce = (double)gnz > order * (double)n;
  int n_unred = gnz, n_red = 0;
  if (do_reduce) {
    n_unred = (int)floor((double)n * (order - 1.0));
    if (n_unred < 0) n_unred = 0;
    n_red = gnz - n_unred;
    // ---- radix select (MSB first, 8 bits per pass) of the n_red-th smallest key among non-zero columns
    // The generator norms of one zonotope share their sign / exponent bits: the passes over the bytes in which ALL active
    // keys agree would put every key into one bin.  Start at the byte of the highest differing bit instead.
    // (bits[][] was written before the barriers of the block scan above)
    unsigned long long all_and = ~0ull, all_or = 0ull;
#pragma unroll
    for (int w = 0; w < kGirardThreads / 32; ++w) {
      all_and &= ((unsigned long long)bits[w][0] << 32) | bits[w][1];
      all_or |= ((unsigned long long)bits[w][2] << 32) | bits[w][3];
    }
    const unsigned long long kdiff = all_and ^ all_or;
    int pass = kdiff == 0ull ? -1 : ((63 - __clzll((long long)kdiff)) >> 3);       // -1: all keys equal, only ties to rank
    if (tid == 0) {
      sel_prefix = pass >= 7 ? 0ull : (pass < 0 ? all_or : (all_or & (~0ull << ((pass + 1) * 8))));
      sel_remaining = n_red;
      sel_done = 0;
    }
    __syncthreads();
    for (; pass >= 0; --pass) {
      hist[tid] = 0;                                           // kGirardThreads == 256 bins
      __syncthreads();
      const unsigned long long prefix = sel_prefix;
      const unsigned long long himask = (pass == 7) ? 0ull : (~0ull << ((pass + 1) * 8));
      // (a warp-aggregated histogram via __match_any_sync was slower than these plain shared-memory atomics: DESIGN.md 5d)
      for (int j = tid; j < g; j += kGirardThreads)
        if (flag[j] && ((key[j] & himask) == prefix)) atomicAdd(&hist[(int)((key[j] >> (pass * 8)) & 0xffull)], 1);
      __syncthreads();
      if (wid == 0) {        // warp 0 finds the digit: lane l owns bins 8l .. 8l+7
        int loc[8], tot = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { loc[i] = hist[lane * 8 + i]; tot += loc[i]; }
        int inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += t;
        }
        const int rem = sel_remaining;
        const int before = inc - tot;                          // keys in lower bins of other lanes
        const bool mine = before < rem && rem <= inc;          // the rem-th smallest lies in one of my bins
        if (mine) {
          int acc = before, d = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (acc + loc[i] >= rem) { d = i; break; }
            acc += loc[i];
          }
          int cnt;
          if constexpr (Cols::kCountFromRegisters) {
            cnt = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) cnt = i == d ? loc[i] : cnt;
          } else {
            cnt = loc[d];
          }
          const unsigned long long digit = (unsigned long long)(lane * 8 + d);
          if (acc + cnt == rem) {
            // the bucket is consumed whole: every key with this prefix and digit is reduced, no need to refine
            const unsigned long long low = pass == 0 ? 0ull : ((1ull << (pass * 8)) - 1ull);
            sel_prefix = prefix | (digit << (pass * 8)) | low;
            sel_remaining = 0;                                 // no ties at the threshold are left out
            sel_done = 1;
          } else {
            sel_prefix = prefix | (digit << (pass * 8));
            sel_remaining = rem - acc;
          }
        }
      }
      __syncthreads();
      if (sel_done) break;
    }
    // keys < thr are reduced; among keys == thr the first `ties_needed` (lowest index) are reduced.
    // (early stop: thr is the largest key of the consumed bucket's range and all keys <= thr are reduced)
    const unsigned long long thr = sel_prefix;
    const bool whole = sel_done != 0;
    const int ties_needed = sel_remaining;
    int my_ties = 0;
    if (!whole)
      for (int j = j0; j < j1; ++j) my_ties += (flag[j] && key[j] == thr) ? 1 : 0;
    int tot;
    int rank = whole ? 0 : block_exclusive_scan(my_ties, warp_tot, tot);
    for (int j = j0; j < j1; ++j) {
      if (!flag[j]) continue;
      if (whole) { if (key[j] <= thr) flag[j] = 2; }
      else if (key[j] < thr) flag[j] = 2;
      else if (key[j] == thr) { if (rank < ties_needed) flag[j] = 2; ++rank; }
    }
    __syncthreads();
    // ---- box of the reduced columns: 8 rows per sweep, fixed-order block reduction (deterministic)
    for (int r0 = 0; r0 < n; r0 += 8) {
      double acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.0;
      for (int ja = tid; ja < g; ja += 2 * kGirardThreads) {       // two columns of loads in flight, same summation order
        const int jc = ja + kGirardThreads;
        const bool fa = flag[ja] == 2, fc = jc < g && flag[jc] == 2;
        double a[8], c[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const bool in = r0 + i < n;
          a[i] = (fa && in) ? fabs(G(r0 + i, ja)) : 0.0;
          c[i] = (fc && in) ? fabs(G(r0 + i, jc)) : 0.0;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) { acc[i] += a[i]; acc[i] += c[i]; }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const double v = warp_sum(acc[i]);
        if (lane == 0) red[wid][i] = v;
      }
      __syncthreads();
      if (tid < 8 && r0 + tid < n) {
        double t = 0.0;
        for (int w = 0; w < kGirardThreads / 32; ++w) t += red[w][tid];
        dbox[r0 + tid] = t;
      }
      __syncthreads();
    }
  }
  // ---- output: kept columns in original order, then diag(d), zero padding
  int my_keep = 0;
  for (int j = j0; j < j1; ++j) my_keep += flag[j] == 1 ? 1 : 0;
  int kept;
  int pos = block_exclusive_scan(my_keep, warp_tot, kept);
  for (int j = j0; j < j1; ++j) {
    if (flag[j] != 1) continue;
    if (pos < gout_cap)
      for (int r = 0; r < n; ++r) out[(int64_t)r * ldo + pos] = G(r, j);
    ++pos;
  }
  int written = kept;
  if (do_reduce) {
    for (int i = tid; i < n * n; i += kGirardThreads) {
      const int r = i / n, c = i - r * n;
      if (written + c < gout_cap) out[(int64_t)r * ldo + written + c] = (r == c) ? dbox[r] : 0.0;
    }
    written += n;
  }
  if (written > gout_cap) written = -written;          // signals "gout_cap too small"
  const int wpos = written < 0 ? gout_cap : written;
  for (int i = tid; i < n * (gout_cap - wpos); i += kGirardThreads) {
    const int r = i / (gout_cap - wpos), c = i - r * (gout_cap - wpos);
    out[(int64_t)r * ldo + wpos + c] = 0.0;
  }
  __syncthreads();
  return written;
}

// Stand-alone reduction: only the keys and flags live in shared memory (9 bytes per generator), so several CTAs share an
// SM; the generator block is read from HBM once (metric pass) and a second time from L2 (box and compaction).
__global__ void __launch_bounds__(kGirardThreads) girard_kernel(int n, int g, double order, int metric,
                                                                const double* __restrict__ Z, int gout_cap,
                                                                double* __restrict__ Zout, int32_t* __restrict__ gout) {
  extern __shared__ unsigned char smraw[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(smraw);    // g
  unsigned char* flag = reinterpret_cast<unsigned char*>(key + g);           // g: 0 zero, 1 keep, 2 reduce
  const int64_t s = blockIdx.x;
  const int tid = threadIdx.x;
  const int ldz = 1 + g, ldo = 1 + gout_cap;
  const double* Zs = Z + s * (int64_t)n * ldz;
  double* Os = Zout + s * (int64_t)n * ldo;
  for (int r = tid; r < n; r += kGirardThreads) Os[(int64_t)r * ldo] = Zs[(int64_t)r * ldz];
  const int written = girard_block(n, g, order, metric, ResidentCols{Zs + 1, ldz}, key, flag, Os + 1, ldo, gout_cap);
  if (tid == 0) gout[s] = written;
}

// ---------------------------------------------------------------------------------------
// Girard reduction, ONE WARP PER ZONOTOPE (north_star: "a warp-per-zonotope segmented sort/top-k kernel does the order
// reduction").  Same semantics as girard_block, but nothing in it is a CTA barrier: the CTA version spent 26 % of its
// samples at barriers and serialised its phases (metric -> select -> box -> output), so that only the CTAs that happened to
// be in the metric phase had loads in flight (profiles/r1_reach_girard_ncu.txt).  Here up to 32 independent warps per SM
// are each in their own phase.  Lanes stride the columns (j = 32 i + lane: every access a 256-byte run), the keys, flags
// and the 256-bin histogram live in the warp's slice of shared memory, ranks in column order come from ballots.
//   metric -> [common leading bytes of the keys skipped] -> 8-bit MSB-first radix select of the n_red-th smallest key ->
//   ties by lowest index -> box of the selected columns -> kept columns in original order, diag(d), zero padding.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// (hi, lo) += x with the rounding error of the addition kept in lo (Neumaier): the box is computed as
// "sum over all columns minus sum over the kept columns", so that the generator block is read from HBM exactly once;
// the compensation keeps the difference accurate to an ulp of the reduced sum even when the kept columns carry
// almost all of a row's mass, and when the reduced entries of a row are all zero both sums go through the same
// additions in the same order and cancel exactly.
__device__ __forceinline__ void csum(double& hi, double& lo, double x) {
  const double s = hi + x;
  const double bb = s - hi;
  lo += (hi - (s - bb)) + (x - bb);
  hi = s;
}
__device__ __forceinline__ void cwarp(double& hi, double& lo) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oh = __shfl_xor_sync(0xffffffffu, hi, o), ol = __shfl_xor_sync(0xffffffffu, lo, o);
    // (both partners must arrive at the same bits: add the smaller-lane value to the larger-lane one in a fixed order)
    const bool low = (threadIdx.x & o) == 0;
    double h = low ? hi : oh, l = low ? lo : ol;
    const double xh = low ? oh : hi, xl = low ? ol : lo;
    csum(h, l, xh);
    l += xl;
    hi = h; lo = l;
  }
}

__global__ void __launch_bounds__(32) girard_warp_kernel(int n, int g, double order, int metric, const double* __restrict__ Z,
                                                         int gout_cap, double* __restrict__ Zout, int32_t* __restrict__ gout) {
  extern __shared__ __align__(16) unsigned char smw[];
  unsigned long long* key = reinterpret_cast<unsigned long long*>(smw);      // g
  int* hist = reinterpret_cast<int*>(key + g);                                // 256
  unsigned char* flag = reinterpret_cast<unsigned char*>(hist + 256);         // g: 0 zero, 1 keep, 2 reduce
  const int lane = threadIdx.x;
  const int64_t s = blockIdx.x;
  const int ldz = 1 + g, ldo = 1 + gout_cap;
  const double* G = Z + s * (int64_t)n * ldz + 1;
  double* Os = Zout + s * (int64_t)n * ldo;
  double* out = Os + 1;
  const int64_t ldg = ldz;
  for (int r = lane; r < n; r += 32) Os[(int64_t)r * ldo] = G[(int64_t)r * ldg - 1];      // centre
  // ---- metric (rows accumulated r = 0..n-1, exactly as oracle/zono.py:_girard_metric), zero filter, row sums of |G|
  int nnz_local = 0;
  unsigned long long kand = ~0ull, kor = 0ull;
  double bh[8], bl[8];                                         // n <= 8: sum_j |G[r][j]| over this lane's columns
#pragma unroll
  for (int i = 0; i < 8; ++i) { bh[i] = 0.0; bl[i] = 0.0; }
  for (int ja = lane; ja < g; ja += 64) {
    const int jc = ja + 32;
    const bool hc = jc < g;
    double a[8], c[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const bool in = i < n;
      a[i] = in ? fabs(__ldcs(G + (int64_t)i * ldg + ja)) : 0.0;
      c[i] = (in && hc) ? fabs(__ldcs(G + (int64_t)i * ldg + jc)) : 0.0;
    }
    double sumA = 0.0, mxA = 0.0, sumC = 0.0, mxC = 0.0;
    bool nzA = false, nzC = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      nzA = nzA || (a[i] != 0.0);
      nzC = nzC || (c[i] != 0.0);
      if (metric == 2) {       // no FMA contraction: selection must match the oracle bit for bit
        sumA = __dadd_rn(sumA, __dmul_rn(a[i], a[i]));
        sumC = __dadd_rn(sumC, __dmul_rn(c[i], c[i]));
      } else {
        sumA += a[i];
        sumC += c[i];
      }
      mxA = fmax(mxA, a[i]);
      mxC = fmax(mxC, c[i]);
      csum(bh[i], bl[i], a[i]);
      csum(bh[i], bl[i], c[i]);
    }
    const unsigned long long kA = (unsigned long long)__double_as_longlong((metric == 0) ? (sumA - mxA) : sumA);
    key[ja] = kA;                                              // h >= 0: the bit pattern is order-preserving
    flag[ja] = nzA ? 1 : 0;
    if (nzA) { ++nnz_local; kand &= kA; kor |= kA; }
    if (hc) {
      const unsigned long long kC = (unsigned long long)__double_as_longlong((metric == 0) ? (sumC - mxC) : sumC);
      key[jc] = kC;
      flag[jc] = nzC ? 1 : 0;
      if (nzC) { ++nnz_local; kand &= kC; kor |= kC; }
    }
  }
  const int gnz = __reduce_add_sync(0xffffffffu, nnz_local);
  __syncwarp();
  const bool do_reduce = (double)gnz > order * (double)n;
  if (do_reduce) {
    int n_unred = (int)floor((double)n * (order - 1.0));
    if (n_unred < 0) n_unred = 0;
    const int n_red = gnz - n_unred;
    // bits shared by every active key need no pass: start at the byte of the highest differing bit
    const unsigned and_hi = __reduce_and_sync(0xffffffffu, (unsigned)(kand >> 32)), and_lo = __reduce_and_sync(0xffffffffu, (unsigned)kand);
    const unsigned or_hi = __reduce_or_sync(0xffffffffu, (unsigned)(kor >> 32)), or_lo = __reduce_or_sync(0xffffffffu, (unsigned)kor);
    const unsigned long long all_and = ((unsigned long long)and_hi << 32) | and_lo, all_or = ((unsigned long long)or_hi << 32) | or_lo;
    const unsigned long long diff = all_and ^ all_or;
    unsigned long long thr;
    bool whole = false;
    int ties_needed = n_red;
    if (diff == 0ull) {
      thr = all_or;                                            // all active keys are equal: the first n_red of them are reduced
    } else {
      int pass = (63 - __clzll((long long)diff)) >> 3;
      unsigned long long prefix = pass == 7 ? 0ull : (all_or & (~0ull << ((pass + 1) * 8)));
      int remaining = n_red;
      for (; pass >= 0; --pass) {
#pragma unroll
        for (int i = 0; i < 8; ++i) hist[lane * 8 + i] = 0;
        __syncwarp();
        const unsigned long long himask = (pass == 7) ? 0ull : (~0ull << ((pass + 1) * 8));
        for (int j = lane; j < g; j += 32)
          if (flag[j] && ((key[j] & himask) == prefix)) atomicAdd(&hist[(int)((key[j] >> (pass * 8)) & 0xffull)], 1);
        __syncwarp();
        int tot = 0;                                           // lane l owns bins 8l .. 8l+7
        int loc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { loc[i] = hist[lane * 8 + i]; tot += loc[i]; }
        int inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += t;
        }
        const int before = inc - tot;                          // keys in the bins of lower lanes
        const bool mine = before < remaining && remaining <= inc;      // the remaining-th smallest lies in one of my bins
        int acc = before, d = 0, cnt = 0;
        bool found = false;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (!found) {
            if (acc + loc[i] >= remaining) { d = i; cnt = loc[i]; found = true; }
            else acc += loc[i];
          }
        }
        const int owner = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;      // exactly one lane
        const int o_acc = __shfl_sync(0xffffffffu, acc, owner), o_d = __shfl_sync(0xffffffffu, d, owner);
        const int o_cnt = __shfl_sync(0xffffffffu, cnt, owner);
        const unsigned long long digit = (unsigned long long)(owner * 8 + o_d);
        __syncwarp();
        if (o_acc + o_cnt == remaining) {
          // the bucket is consumed whole: every key with this prefix and digit is reduced, no need to refine
          const unsigned long long low = pass == 0 ? 0ull : ((1ull << (pass * 8)) - 1ull);
          prefix = prefix | (digit << (pass * 8)) | low;
          remaining = 0;
          whole = true;
          break;
        }
        prefix = prefix | (digit << (pass * 8));
        remaining -= o_acc;
      }
      thr = prefix;
      ties_needed = remaining;
    }
    // keys < thr are reduced; among keys == thr the first `ties_needed` in column order (whole: all keys <= thr)
    int taken = 0;
    for (int j0 = 0; j0 < g; j0 += 32) {
      const int j = j0 + lane;
      const bool act = j < g && flag[j] != 0;
      const unsigned long long k = act ? key[j] : 0ull;
      const bool tie = act && !whole && k == thr;
      const unsigned tb = __ballot_sync(0xffffffffu, tie);
      const int rank = taken + __popc(tb & lanemask_lt());
      if (act) {
        if (whole) { if (k <= thr) flag[j] = 2; }
        else if (k < thr) flag[j] = 2;
        else if (tie && rank < ties_needed) flag[j] = 2;
      }
      taken += __popc(tb);
    }
    __syncwarp();
  }
  // ---- output: kept columns in original order (their |.| row sums are taken off the totals), then diag(d), zero padding
  double kh[8], kl[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { kh[i] = 0.0; kl[i] = 0.0; }
  int written = 0;
  for (int j0 = 0; j0 < g; j0 += 32) {
    const int j = j0 + lane;
    const bool keep = j < g && flag[j] == 1;
    const unsigned kb = __ballot_sync(0xffffffffu, keep);
    const int pos = written + __popc(kb & lanemask_lt());
    if (keep) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i < n) {
          const double v = G[(int64_t)i * ldg + j];
          if (pos < gout_cap) out[(int64_t)i * ldo + pos] = v;
          csum(kh[i], kl[i], fabs(v));
        }
      }
    }
    written += __popc(kb);
  }
  if (do_reduce) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      cwarp(bh[i], bl[i]);
      cwarp(kh[i], kl[i]);
      // d_r = (total - kept), never negative
      const double dh = bh[i] - kh[i];
      const double bb = dh - bh[i];
      const double err = (bh[i] - (dh - bb)) + (-kh[i] - bb);
      bh[i] = fmax(dh + (err + (bl[i] - kl[i])), 0.0);
    }
    for (int i = lane; i < n * n; i += 32) {
      const int r = i / n, c = i - r * n;
      double dv = 0.0;
#pragma unroll
      for (int q = 0; q < 8; ++q) dv = (q == r) ? bh[q] : dv;
      if (written + c < gout_cap) out[(int64_t)r * ldo + written + c] = (r == c) ? dv : 0.0;
    }
    written += n;
  }
  if (written > gout_cap) written = -written;          // signals "gout_cap too small"
  const int wpos = written < 0 ? gout_cap : written;
  const int padc = gout_cap - wpos;
  for (int i = lane; i < n * padc; i += 32) {
    const int r = i / padc, c = i - r * padc;
    out[(int64_t)r * ldo + wpos + c] = 0.0;
  }
  if (lane == 0) gout[s] = written;
}

// Column col of a tube step's pre-reduction block  [C_K G | G^K_1 c, G^K_1 G | ... | G^D_1 z .. G^D_ND z | G_W]
// (pyzonotope column order, g generators in the current zonotope Zc = [c, G]): the product M v of a staged matrix and a
// column of Zc or z_k, an FMA chain from 0.0 in q order, or a column of W.  The same map and chain as the loop that fills
// Gp in tube_rollout_kernel (left as written there, so that kernel compiles as before): tube_rollout_recompute_kernel
// evaluates an entry wherever girard_block reads the block, and gets the resident kernel's bits.
struct ProductCols {
  static constexpr bool kCountFromRegisters = true;
  const double* MK;             // (NK + 1) x n x n : C_K, G^K_i
  const double* MD;             // ND x n x p : G^D_i
  const double* Zc;             // n x (1 + g), row pitch ldc
  const double* zk;             // p
  const double* W;              // n x (1 + gW), global
  int n, p, NK, ND, gW, g, ldc;
  struct Col {
    const double* M;            // nullptr: a column of W
    const double* v;            // the vector multiplied: a column of Zc (stride ldc) or z_k (stride 1)
    int vstride, len;
  };
  __device__ __forceinline__ Col column(int col) const {
    Col c;
    if (col < g) { c.M = MK; c.v = Zc + 1 + col; c.vstride = ldc; c.len = n; }
    else if (col < g + NK * (1 + g)) {
      const int t = col - g, b = t / (1 + g), j = t - b * (1 + g);
      c.M = MK + (size_t)(1 + b) * n * n; c.v = Zc + j; c.vstride = ldc; c.len = n;
    } else if (col < g + NK * (1 + g) + ND) {
      const int b = col - g - NK * (1 + g);
      c.M = MD + (size_t)b * n * p; c.v = zk; c.vstride = 1; c.len = p;
    } else {
      c.M = nullptr; c.v = W + 1 + (col - g - NK * (1 + g) - ND); c.vstride = 1 + gW; c.len = 0;
    }
    return c;
  }
  __device__ __forceinline__ double entry(const Col& c, int r) const {
    if (c.M == nullptr) return c.v[(int64_t)r * c.vstride];
    double acc = 0.0;
    for (int q = 0; q < c.len; ++q) acc = fma(c.M[r * c.len + q], c.v[(int64_t)q * c.vstride], acc);
    return acc;
  }
  __device__ __forceinline__ double operator()(int r, int col) const { return entry(column(col), r); }
};

// ---------------------------------------------------------------------------------------
// Tube rollout: `steps` reach-set steps of one scenario by one CTA, the zonotope never leaving shared memory:
//   Z_{k+1} = reduce( M_K (x) Z_k  (+)  M_Delta (x) <z_k, 0>  (+)  W ,  order )          z_k = [xbar_k; v_k]
// i.e. tzddpc/tzddpc.py:175-186,205 evaluated numerically with the Girard reduction of
// examples/1.double_integrator_sim.py:170 applied after every step (BASELINE.json configs[4]: long horizons need
// it, the un-reduced generator count grows like (N_K + 1)^k).  Per step the pre-reduction block
//   [C_K G | G^K_1 c, G^K_1 G | ... | G^D_1 z .. G^D_ND z | G_W]   (n x ((N_K+1) g + N_K + N_D + g_W), pyzonotope order)
// is built in shared memory, reduced in place (girard_block) and its interval hull (tzddpc/tzddpc.py:191-197)
// written out: HBM traffic per scenario-step is the hull (2n doubles) + z_k, not the 100 KB generator block.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGirardThreads) tube_rollout_kernel(
    int n, int m, int NK, int ND, int gW, int g0, int steps, double order, int metric, int gcap, int gpre_cap,
    const double* __restrict__ CK, const double* __restrict__ GK, const double* __restrict__ GD, int per_scenario,
    const double* __restrict__ Z0, const double* __restrict__ XU, const double* __restrict__ W,
    double* __restrict__ Zfinal, int32_t* __restrict__ gfinal, double* __restrict__ hull_lo, double* __restrict__ hull_hi) {
  extern __shared__ unsigned char smraw[];
  const int p = n + m, tid = threadIdx.x;
  const int64_t s = blockIdx.x;
  double* Zc = reinterpret_cast<double*>(smraw);                 // n x (1 + gcap): current zonotope [c, G]
  double* Gp = Zc + (size_t)n * (1 + gcap);                      // n x gpre_cap: pre-reduction generator block
  double* MK = Gp + (size_t)n * gpre_cap;                        // (NK + 1) x n x n : C_K, G^K_i
  double* MD = MK + (size_t)(NK + 1) * n * n;                    // ND x n x p
  double* zk = MD + (size_t)ND * n * p;                          // p
  double* cnew = zk + p;                                         // n
  unsigned long long* key = reinterpret_cast<unsigned long long*>(cnew + n + ((n + p) & 1));
  unsigned char* flag = reinterpret_cast<unsigned char*>(key + gpre_cap);
  __shared__ int g_cur, overflow;
  const double* CKs = CK + (per_scenario ? s * (int64_t)n * n : 0);
  const double* GKs = GK + (per_scenario ? s * (int64_t)NK * n * n : 0);
  const double* GDs = GD + (per_scenario ? s * (int64_t)ND * n * p : 0);
  for (int i = tid; i < n * n; i += kGirardThreads) MK[i] = CKs[i];
  for (int i = tid; i < NK * n * n; i += kGirardThreads) MK[n * n + i] = GKs[i];
  for (int i = tid; i < ND * n * p; i += kGirardThreads) MD[i] = GDs[i];
  const int ldc = 1 + gcap;
  for (int i = tid; i < n * (1 + g0); i += kGirardThreads) {
    const int r = i / (1 + g0), j = i - r * (1 + g0);
    Zc[r * ldc + j] = Z0[s * (int64_t)n * (1 + g0) + i];
  }
  if (tid == 0) { g_cur = g0; overflow = 0; }
  __syncthreads();
  for (int k = 0; k < steps; ++k) {
    const int g = g_cur;
    const int gpre = (NK + 1) * g + NK + ND + gW;
    if (tid < p) zk[tid] = XU[(s * (int64_t)steps + k) * p + tid];
    __syncthreads();
    // ---- centre: C_K c + c_W   (M_Delta has a zero centre, tzddpc/tzddpc.py:122-123)
    if (tid < n) {
      double acc = W ? W[(int64_t)tid * (1 + gW)] : 0.0;
      for (int q = 0; q < n; ++q) acc = fma(MK[tid * n + q], Zc[q * ldc], acc);
      cnew[tid] = acc;
    }
    // ---- generator block, pyzonotope column order
    for (int col = tid; col < gpre; col += kGirardThreads) {
      const double* M;
      const double* v;        // the vector multiplied: a column of Zc (stride ldc) or z_k (stride 1)
      int vstride, len;
      if (col < g) { M = MK; v = Zc + 1 + col; vstride = ldc; len = n; }
      else if (col < g + NK * (1 + g)) {
        const int t = col - g, b = t / (1 + g), j = t - b * (1 + g);
        M = MK + (size_t)(1 + b) * n * n; v = Zc + j; vstride = ldc; len = n;
      } else if (col < g + NK * (1 + g) + ND) {
        const int b = col - g - NK * (1 + g);
        M = MD + (size_t)b * n * p; v = zk; vstride = 1; len = p;
      } else {
        M = nullptr; v = W + 1 + (col - g - NK * (1 + g) - ND); vstride = 1 + gW; len = 0;
      }
      for (int r = 0; r < n; ++r) {
        double acc;
        if (M == nullptr) acc = v[(int64_t)r * vstride];
        else {
          acc = 0.0;
          for (int q = 0; q < len; ++q) acc = fma(M[r * len + q], v[(int64_t)q * vstride], acc);
        }
        Gp[(size_t)r * gpre + col] = acc;
      }
    }
    __syncthreads();
    if (tid < n) Zc[tid * ldc] = cnew[tid];
    const int written = girard_block(n, gpre, order, metric, ResidentCols{Gp, gpre}, key, flag, Zc + 1, ldc, gcap);
    if (tid == 0) { g_cur = written < 0 ? gcap : written; if (written < 0) overflow = 1; }
    __syncthreads();
    // ---- interval hull of Z_{k+1}: warp r handles row r
    {
      const int gg = g_cur, lane = tid & 31;
      for (int r = tid >> 5; r < n; r += kGirardThreads / 32) {
        double acc = 0.0;
        for (int j = 1 + lane; j <= gg; j += 32) acc += fabs(Zc[r * ldc + j]);
        acc = warp_sum(acc);
        if (lane == 0) {
          const double c = Zc[r * ldc];
          hull_lo[(s * (int64_t)steps + k) * n + r] = c - acc;
          hull_hi[(s * (int64_t)steps + k) * n + r] = c + acc;
        }
      }
    }
    __syncthreads();
  }
  for (int i = tid; i < n * ldc; i += kGirardThreads) Zfinal[s * (int64_t)n * ldc + i] = Zc[i];
  if (tid == 0) gfinal[s] = overflow ? -g_cur : g_cur;       // negative: gcap was too small at some step (truncated)
}

// The same rollout without the pre-reduction block in shared memory: girard_block reads it through ProductCols, which
// evaluates each entry from the current zonotope, z_k and the staged matrices (at most n + m FMAs) every time a pass
// reads it, so the metric pass computes every column once and the box and compaction passes each column once more.
// Shared memory per scenario is two zonotopes (the reduced one cannot overwrite the one its columns are computed from),
// the matrices and 9 bytes of key and flag per pre-reduction column: 74 KiB at n = 5, order 40, where the resident
// kernel needs 272 KiB.  Results are the resident kernel's bit for bit.
__global__ void __launch_bounds__(kGirardThreads) tube_rollout_recompute_kernel(
    int n, int m, int NK, int ND, int gW, int g0, int steps, double order, int metric, int gcap, int gpre_cap,
    const double* __restrict__ CK, const double* __restrict__ GK, const double* __restrict__ GD, int per_scenario,
    const double* __restrict__ Z0, const double* __restrict__ XU, const double* __restrict__ W,
    double* __restrict__ Zfinal, int32_t* __restrict__ gfinal, double* __restrict__ hull_lo, double* __restrict__ hull_hi) {
  extern __shared__ unsigned char smraw[];
  const int p = n + m, tid = threadIdx.x;
  const int64_t s = blockIdx.x;
  const int ldc = 1 + gcap;
  double* Zc = reinterpret_cast<double*>(smraw);                 // n x (1 + gcap): current zonotope [c, G]
  double* Zn = Zc + (size_t)n * ldc;                             // n x (1 + gcap): the next one
  double* MK = Zn + (size_t)n * ldc;                             // (NK + 1) x n x n : C_K, G^K_i
  double* MD = MK + (size_t)(NK + 1) * n * n;                    // ND x n x p
  double* zk = MD + (size_t)ND * n * p;                          // p
  unsigned long long* key = reinterpret_cast<unsigned long long*>(zk + p + (p & 1));
  unsigned char* flag = reinterpret_cast<unsigned char*>(key + gpre_cap);
  __shared__ int g_cur, overflow;
  const double* CKs = CK + (per_scenario ? s * (int64_t)n * n : 0);
  const double* GKs = GK + (per_scenario ? s * (int64_t)NK * n * n : 0);
  const double* GDs = GD + (per_scenario ? s * (int64_t)ND * n * p : 0);
  for (int i = tid; i < n * n; i += kGirardThreads) MK[i] = CKs[i];
  for (int i = tid; i < NK * n * n; i += kGirardThreads) MK[n * n + i] = GKs[i];
  for (int i = tid; i < ND * n * p; i += kGirardThreads) MD[i] = GDs[i];
  for (int i = tid; i < n * ldc; i += kGirardThreads) {        // zero padding: Zfinal is defined for steps = 0 too
    const int r = i / ldc, j = i - r * ldc;
    Zc[i] = j <= g0 ? Z0[s * (int64_t)n * (1 + g0) + (int64_t)r * (1 + g0) + j] : 0.0;
  }
  if (tid == 0) { g_cur = g0; overflow = 0; }
  __syncthreads();
  for (int k = 0; k < steps; ++k) {
    const int g = g_cur;
    const int gpre = (NK + 1) * g + NK + ND + gW;
    if (tid < p) zk[tid] = XU[(s * (int64_t)steps + k) * p + tid];
    __syncthreads();
    // ---- centre: C_K c + c_W, as in tube_rollout_kernel
    if (tid < n) {
      double acc = W ? W[(int64_t)tid * (1 + gW)] : 0.0;
      for (int q = 0; q < n; ++q) acc = fma(MK[tid * n + q], Zc[q * ldc], acc);
      Zn[tid * ldc] = acc;
    }
    const ProductCols P{MK, MD, Zc, zk, W, n, p, NK, ND, gW, g, ldc};
    const int written = girard_block(n, gpre, order, metric, P, key, flag, Zn + 1, ldc, gcap);
    if (tid == 0) { g_cur = written < 0 ? gcap : written; if (written < 0) overflow = 1; }
    __syncthreads();
    // ---- interval hull of Z_{k+1}: warp r handles row r
    {
      const int gg = g_cur, lane = tid & 31;
      for (int r = tid >> 5; r < n; r += kGirardThreads / 32) {
        double acc = 0.0;
        for (int j = 1 + lane; j <= gg; j += 32) acc += fabs(Zn[r * ldc + j]);
        acc = warp_sum(acc);
        if (lane == 0) {
          const double c = Zn[r * ldc];
          hull_lo[(s * (int64_t)steps + k) * n + r] = c - acc;
          hull_hi[(s * (int64_t)steps + k) * n + r] = c + acc;
        }
      }
    }
    double* t = Zc; Zc = Zn; Zn = t;
    __syncthreads();
  }
  for (int i = tid; i < n * ldc; i += kGirardThreads) Zfinal[s * (int64_t)n * ldc + i] = Zc[i];
  if (tid == 0) gfinal[s] = overflow ? -g_cur : g_cur;       // negative: gcap was too small at some step (truncated)
}

}  // namespace tz

using namespace tz;

extern "C" int tz_interval_hull(int64_t S, int32_t n, int32_t g, const double* Z, double* lo, double* hi, void* stream) {
  TZ_REQUIRE(S >= 0 && n >= 1 && g >= 0, "bad shape");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(Z && lo && hi, "null pointer");
  const int wpb = 8;
  hull_kernel<<<(unsigned)((S + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(S, n, g, Z, lo, hi);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_reach_step(int64_t S, int32_t n, int32_t p, int32_t N, int32_t g, int32_t gW, const double* C,
                             const double* Gm, int32_t per_scenario_model, const double* Z, const double* W,
                             double* Zout, void* stream) {
  TZ_REQUIRE(S >= 0 && n >= 1 && n <= 16 && p >= 1 && N >= 0 && g >= 0 && gW >= 0, "bad shape (n <= 16)");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(C && Z && Zout && (N == 0 || Gm) && (gW == 0 || W), "null pointer");
  const size_t smem = (size_t)(N + 1) * n * p * sizeof(double);
  TZ_REQUIRE(smem <= 200 * 1024, "matrix zonotope too large for shared memory");
  cudaStream_t st = (cudaStream_t)stream;
  // exact-dimension fast paths: M_K (p = n) and M_Delta (p = n + 1) of the double integrator, the pulley and the 5-dim system
#define TZ_FAST(NN, PP) \
  if (n == NN && p == PP) return launch_reach_fast<NN, PP>(S, N, g, gW, C, Gm, per_scenario_model, Z, W, Zout, st);
  TZ_FAST(2, 2) TZ_FAST(2, 3) TZ_FAST(4, 4) TZ_FAST(4, 5) TZ_FAST(5, 5) TZ_FAST(5, 6)
#undef TZ_FAST
  if (n <= 8) {
    if (smem + 8192 > 48 * 1024) TZ_CUDA(cudaFuncSetAttribute(reach_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reach_kernel<8><<<(unsigned)S, 256, smem, st>>>(n, p, N, g, gW, C, Gm, per_scenario_model, Z, W, Zout);
  } else {
    if (smem + 8192 > 48 * 1024) TZ_CUDA(cudaFuncSetAttribute(reach_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    reach_kernel<16><<<(unsigned)S, 256, smem, st>>>(n, p, N, g, gW, C, Gm, per_scenario_model, Z, W, Zout);
  }
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_girard_reduce(int64_t S, int32_t n, int32_t g, double order, int32_t metric, const double* Z,
                                int32_t gout_cap, double* Zout, int32_t* gout, void* stream) {
  TZ_REQUIRE(S >= 0 && n >= 1 && n <= kGirardMaxDim && g >= 0 && gout_cap >= 0 && order > 0, "bad shape (n <= 128)");
  TZ_REQUIRE(metric >= 0 && metric <= 2, "metric must be 0 (l1-linf), 1 (l1) or 2 (l2)");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(Z && Zout && gout, "null pointer");
  {  // Short zonotopes (the tubes Ze[1] of the examples: 24 / 75 / 113 generators): one warp per zonotope, a 256-thread CTA
     // would idle.  Measured on B200 (n = 5, order 3, scratch/girard_small.py): warp kernel 2.0x / 1.7x / 1.1x faster at
     // g = 32 / 64 / 113, CTA kernel 1.2x / 1.6x / 1.7x faster at g = 256 / 512 / 1024 and 1.4-2.6x at the stress sizes.
    const size_t smw = (size_t)g * 9 + 256 * sizeof(int) + 32;
    if (g <= 128 && n <= 8 && smw <= 56 * 1024) {
      if (smw + 8192 > 48 * 1024)
        TZ_CUDA(cudaFuncSetAttribute(girard_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
      girard_warp_kernel<<<(unsigned)S, 32, smw, (cudaStream_t)stream>>>(n, g, order, metric, Z, gout_cap, Zout, gout);
      TZ_CUDA(cudaGetLastError());
      return TZ_OK;
    }
  }
  const size_t smem = (size_t)g * sizeof(unsigned long long) + (size_t)g + 16;
  TZ_REQUIRE(smem <= 200 * 1024, "too many generators (g=%d) for the shared-memory key table", g);
  if (smem + 8192 > 48 * 1024) TZ_CUDA(cudaFuncSetAttribute(girard_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  girard_kernel<<<(unsigned)S, kGirardThreads, smem, (cudaStream_t)stream>>>(n, g, order, metric, Z, gout_cap, Zout, gout);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_tube_rollout(int64_t S, int32_t n, int32_t m, int32_t NK, int32_t ND, int32_t gW, int32_t g0, int32_t steps,
                               double order, int32_t metric, const double* CK, const double* GK, const double* GD,
                               int32_t per_scenario_model, const double* Z0, const double* XU, const double* W, int32_t gcap,
                               double* Zfinal, int32_t* gfinal, double* hull_lo, double* hull_hi, void* stream) {
  TZ_REQUIRE(S >= 0 && n >= 1 && n <= 16 && m >= 1 && NK >= 0 && ND >= 0 && gW >= 0 && g0 >= 0 && steps >= 0 && order >= 1.0,
             "bad shape (n <= 16, order >= 1)");
  TZ_REQUIRE(metric >= 0 && metric <= 2, "metric must be 0 (l1-linf), 1 (l1) or 2 (l2)");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(CK && Z0 && XU && Zfinal && gfinal && hull_lo && hull_hi && (NK == 0 || GK) && (ND == 0 || GD) && (gW == 0 || W),
             "null pointer");
  // generators after a reduction: floor(n (order - 1)) kept + n boxed; before the first one there may be g0
  const int gred = (int)floor((double)n * (order - 1.0)) + n;
  const int gmax = g0 > gred ? g0 : gred;
  TZ_REQUIRE(gcap >= gmax, "gcap must be at least max(g0, floor(n (order - 1)) + n) = %d", gmax);
  // A step keeps up to floor(n * order) generators unreduced (girard_block reduces only when more than order * n are
  // non-zero), which rounding can put above gred (order 1.2, n = 5: 6 against 5); a larger gcap then lets them through.
  const int gkeep = (int)floor((double)n * order);
  const int gstep = gkeep > gmax ? (gkeep < gcap ? gkeep : gcap) : gmax;      // bound on the generators entering a step
  const int64_t gpre_cap = (int64_t)(NK + 1) * gstep + NK + ND + gW;
  const int p = n + m;
  const size_t smem = ((size_t)n * (1 + gcap) + (size_t)n * gpre_cap + (size_t)(NK + 1) * n * n + (size_t)ND * n * p + p + n + 2) *
                          sizeof(double) + (size_t)gpre_cap * sizeof(unsigned long long) + (size_t)gpre_cap + 16;
  // without the n x gpre_cap block, with a second zonotope: about a third of the resident size at n = 5
  const size_t smem_rc = ((size_t)2 * n * (1 + gcap) + (size_t)(NK + 1) * n * n + (size_t)ND * n * p + p + 1) * sizeof(double) +
                         (size_t)gpre_cap * sizeof(unsigned long long) + (size_t)gpre_cap + 16;
  const size_t limit = 220 * 1024;
  // The resident kernel wherever it fits; TZDDPC_ROLLOUT = resident / recompute (read per launch) forces one of the two,
  // for comparisons of the two kernels.
  bool recompute = smem > limit;
  if (const char* e = getenv("TZDDPC_ROLLOUT")) {
    TZ_REQUIRE(!strcmp(e, "resident") || !strcmp(e, "recompute"), "TZDDPC_ROLLOUT must be resident or recompute, not '%s'", e);
    recompute = !strcmp(e, "recompute");
  }
  const size_t need = recompute ? smem_rc : smem;
  TZ_REQUIRE(need <= limit,
             "tube step (n=%d, %lld generators before reduction) needs %zu bytes of shared memory with the block resident and "
             "%zu with it recomputed; at most %zu fit",
             n, (long long)gpre_cap, smem, smem_rc, limit);
  auto kernel = recompute ? tube_rollout_recompute_kernel : tube_rollout_kernel;
  if (need + 8192 > 48 * 1024) TZ_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
  kernel<<<(unsigned)S, kGirardThreads, need, (cudaStream_t)stream>>>(
      n, m, NK, ND, gW, g0, steps, order, metric, gcap, (int)gpre_cap, CK, GK, GD, per_scenario_model, Z0, XU, W,
      Zfinal, gfinal, hull_lo, hull_hi);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}
