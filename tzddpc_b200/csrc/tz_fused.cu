// Fused per-step kernel of the TZDDPC hot path: bounds of the parametric program from
// (xbar0, e0)  ->  ADMM + polish  ->  nominal trajectory, cost, Ze[1].Z  ->  closed-loop update.
//
// Persistent kernel: one wave of CTAs, each staging the (scaled, padded) program into shared
// memory once and then looping over tiles of SPB = 128/G scenarios.  Inside a tile
//   * solve phase : G adjacent lanes per scenario (tz_admm.cuh);
//   * output phase: threads are re-mapped to (scenario, slice) so that every warp writes full
//     128-byte lines of the scenario-fastest (SoA) output arrays; Ze[1].Z -- 88 % structural
//     zeros, but dense by contract -- is written from a zero-entry list and a one-term-per-entry
//     table with streaming stores.
// Replaces, per closed-loop step,
//   tzddpc/tzddpc.py:357-377  (TZDDPC.solve: parameter update + cvxpy solve + Ze[1])
//   examples/2.pulley_sim.py:90-96 (nominal/plant/error update, Zek.Z.value)
// Algorithmic HBM bytes per scenario-step (SURVEY.md 8d):
//   8*[6n + N*m + (N+1)n + 1 + n(1+g1)] + 4.
#include "tz_step.cuh"
#include "tz_big.h"

namespace tz {

// the larger buckets are compiled in tz_bucket1.cu / tz_bucket2.cu / tz_bucket3.cu
// fast_step_kernel (tz_fast.cuh) is compiled in tz_fast.cu
template <class BK>
int launch_fast(const TzProgram* p, const SolverParams& sp, const StepArgs& a, cudaStream_t st);
extern template int launch_fast<B0>(const TzProgram*, const SolverParams&, const StepArgs&, cudaStream_t);
template <class BK>
int launch_fast_set(const TzProgram* p0, const SolverParams& sp, const StepArgs& a, const SetEntry* entries, const int32_t* tile_prog,
                    int block, cudaStream_t st);
extern template int launch_fast_set<B0>(const TzProgram*, const SolverParams&, const StepArgs&, const SetEntry*, const int32_t*, int,
                                        cudaStream_t);
extern template int launch_bucket<B1>(const TzProgram*, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket<B2>(const TzProgram*, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket<B3>(const TzProgram*, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set<B1>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set<B2>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set<B3>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set_run<B1>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set_run<B2>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
extern template int launch_bucket_set_run<B3>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);

constexpr int64_t kHotMinBatch = 256;

struct RowClasses { int n2 = 0, nu = 0, nl = 0; };

static RowClasses classify(const TzProgramDesc& d, std::vector<int>* cls) {
  RowClasses rc;
  for (int i = 0; i < d.nc; ++i) {
    const bool lf = std::isfinite(d.l0[i]), uf = std::isfinite(d.u0[i]);
    int c = 0;                                       // 0: two-sided / kink / free, 1: upper only, 2: lower only
    if (d.wabs[i] > 0.0 || (lf && uf) || (!lf && !uf)) c = 0;
    else if (uf) c = 1;
    else c = 2;
    if (cls) (*cls)[i] = c;
    (c == 0 ? rc.n2 : c == 1 ? rc.nu : rc.nl)++;
  }
  return rc;
}

// unit atoms |p_c| are implicit columns; everything else is a "general" atom
static int general_atoms(const TzProgramDesc& d, std::vector<int>* colmap) {
  const int npar = d.npar;
  int nag = 0;
  for (int i = 0; i < d.na; ++i) {
    int nnz = 0, where = -1;
    for (int k = 0; k < npar; ++k)
      if (d.Bt[i * npar + k] != 0.0) { ++nnz; where = k; }
    const bool unit = (nnz == 1 && d.gam[i] == 0.0 && std::fabs(std::fabs(d.Bt[i * npar + where]) - 1.0) < 1e-15);
    if (colmap) (*colmap)[i] = unit ? -(where + 1) : nag;      // negative: unit atom of parameter `where`
    if (!unit) ++nag;
  }
  return nag;
}

template <class BK>
bool fits(const TzProgramDesc& d) {
  const RowClasses rc = classify(d, nullptr);
  return d.nz <= BK::NZ && rc.n2 <= BK::N2 * BK::G && rc.nu <= BK::NU * BK::G && rc.nl <= BK::NL * BK::G &&
         2 * d.n <= BK::NPAR && general_atoms(d, nullptr) <= BK::NAG && d.nchk <= BK::NCHK;
}

template <class BK>
void pack(const TzProgramDesc& d, QpProg<BK>& g) {
  std::memset(&g, 0, sizeof(g));
  const int nz = d.nz, nc = d.nc, npar = d.npar, na = d.na, ncol = 1 + npar + na;
  std::vector<int> cls(nc), amap(na);
  classify(d, &cls);
  const int nag = general_atoms(d, &amap);
  // parameter k of the caller's p = [xbar0 (n); e0 (n)] -> slot of the padded p = [xbar0 (NPAR/2) | e0 (NPAR/2)]
  const int nx = d.n;
  auto pk = [&](int k) { return k < nx ? k : BK::NPAR / 2 + (k - nx); };
  // column j of the caller's [1 | p | alpha] layout -> column of the padded [1 | p | |p| | general] layout
  auto colmap = [&](int j) {
    if (j == 0) return 0;
    if (j <= npar) return 1 + pk(j - 1);
    const int am = amap[j - 1 - npar];
    return am < 0 ? 1 + BK::NPAR + pk(-am - 1) : 1 + 2 * BK::NPAR + am;
  };
  for (int a = 0; a < BK::NZ; ++a) g.D[a] = 1.0;
  for (int i = 0; i < BK::NC; ++i) {
    g.l0[i] = -INFINITY; g.u0[i] = INFINITY; g.Einv[i] = 1.0; g.row_of_slot[i] = -1; g.sing_var[i] = -1; g.sing_inv[i] = 0.0;
  }
  for (int a = 0; a < nz; ++a) {
    g.D[a] = d.D[a];
    g.q0[a] = d.c * d.D[a] * d.q0[a];
    for (int b = 0; b < nz; ++b) g.P[a][b] = d.c * d.D[a] * d.P[a * nz + b] * d.D[b];
    for (int k = 0; k < npar; ++k) {
      g.Qp[a][pk(k)] = d.c * d.D[a] * d.Qp[a * npar + k];
      if (d.Qp[a * npar + k] != 0.0) g.has_qp = 1;
    }
  }
  int next[3] = {0, BK::N2 * BK::G, (BK::N2 + BK::NU) * BK::G};
  for (int i = 0; i < nc; ++i) {
    const int s = next[cls[i]]++;
    const double E = d.E[i];
    g.row_of_slot[s] = i;
    g.Einv[s] = 1.0 / E;
    int nnz = 0, where = -1;
    for (int a = 0; a < nz; ++a) {
      g.A[s][a] = E * d.A[i * nz + a] * d.D[a];
      if (g.A[s][a] != 0.0) { ++nnz; where = a; }
    }
    if (nnz == 1) { g.sing_var[s] = where; g.sing_inv[s] = 1.0 / g.A[s][where]; }     // a bound on one variable
    g.l0[s] = E * d.l0[i];
    g.u0[s] = E * d.u0[i];
    g.Rs[s] = E;
    for (int j = 0; j < ncol; ++j) g.R[s][colmap(j)] += d.R[i * ncol + j];
    if (cls[i] == 0) {
      g.kink0[s] = E * d.kink0[i];
      g.wabs[s] = d.wabs[i] > 0.0 ? d.c * d.wabs[i] / E : 0.0;
    }
  }
  for (int i = 0; i < na; ++i) {
    if (amap[i] < 0) continue;
    g.gam[amap[i]] = d.gam[i];
    for (int k = 0; k < npar; ++k) g.Bt[amap[i]][pk(k)] = d.Bt[i * npar + k];
  }
  for (int i = 0; i < d.nchk; ++i) {
    for (int j = 0; j < ncol; ++j) g.Rchk[i][colmap(j)] += d.Rchk[i * ncol + j];
    g.chk_tol[i] = 1e-9 * std::fmax(1.0, std::fabs(d.Rchk[i * ncol]));
  }
  for (int j = 0; j < ncol; ++j) g.cc[colmap(j)] += d.cc[j];
  for (int a = 0; a < npar; ++a)
    for (int b = 0; b < npar; ++b) g.CC2[pk(a)][pk(b)] = d.CC2[a * npar + b];
  // ---- groups of rows that share their shift row up to the sign of its constant / |.| part (see QpProg::grp_*)
  {
    auto in_L = [&](int c) { return c >= 1 && c <= BK::NPAR; };
    std::vector<int> rep_of;                         // group -> slot of its first row
    std::vector<std::vector<std::pair<int, double>>> members;
    for (int s = 0; s < BK::NC; ++s) {
      if (g.row_of_slot[s] < 0) continue;            // padding
      int found = -1;
      double sgn = 1.0;
      for (size_t q = 0; q < rep_of.size() && found < 0; ++q) {
        const int r0 = rep_of[q];
        bool same_L = true, same_A = true, neg_A = true;
        for (int c = 0; c < BK::NCOLP; ++c) {
          const double a = g.R[s][c], b = g.R[r0][c];
          if (in_L(c)) same_L = same_L && (a == b);
          else { same_A = same_A && (a == b); neg_A = neg_A && (a == -b); }
        }
        if (same_L && (same_A || neg_A)) { found = (int)q; sgn = same_A ? 1.0 : -1.0; }
      }
      if (found < 0) { rep_of.push_back(s); members.emplace_back(); found = (int)rep_of.size() - 1; }
      members[found].push_back({s, sgn});
    }
    int t = 0, gi = 0;
    for (auto& mem : members) {
      g.grp_first[gi++] = t;
      for (size_t k = 0; k < mem.size(); ++k, ++t) {
        g.grp_order[t] = mem[k].first;
        g.grp_new[t] = k == 0 ? 1 : 0;
        g.grp_sgn[t] = mem[k].second;
      }
    }
    g.ngrp = gi;
    for (; gi < BK::NC + 4; ++gi) g.grp_first[gi] = t;
    for (; t < BK::NC; ++t) { g.grp_order[t] = 0; g.grp_new[t] = 0; g.grp_sgn[t] = 1.0; }
  }
  g.cinv = 1.0 / d.c;
  g.nz = nz; g.nc = nc; g.npar = npar; g.nag = nag; g.nchk = d.nchk;
  g.has_cc2 = 0;
  for (int a = 0; a < npar * npar; ++a) g.has_cc2 |= (d.CC2[a] != 0.0) ? 1 : 0;
}

}  // namespace tz

using namespace tz;

// host images of one program: the packed QpProg<bucket> and the run-time sized tables
struct HostImage {
  std::vector<unsigned char> packed, aux;
};

template <class BK>
static int create_bucket(const TzProgramDesc& d, TzProgram* p, int id, HostImage& img) {
  p->bucket = id;
  img.packed.assign(sizeof(QpProg<BK>), 0);
  pack<BK>(d, *reinterpret_cast<QpProg<BK>*>(img.packed.data()));
  p->NZ = BK::NZ;
  p->NC = BK::NC;
  p->G = BK::G;
  p->NW = BK::NW; p->OM_V = BK::OM_V; p->OM_P = BK::OM_P; p->OM_C = BK::OM_C; p->HP = BK::NPAR / 2;
  return TZ_OK;
}

// the generic warp-per-scenario path (tz_big.cu) for a program no register-resident bucket serves; no packed image, no tables
static int use_big_path(const TzProgramDesc* d, TzProgram* p) {
  p->bucket = 4;
  p->NZ = d->nz; p->NC = d->nc; p->G = 32;
  p->nz = d->nz; p->nc = d->nc; p->n = d->n; p->m = d->m; p->N = d->horizon; p->nv = d->nv; p->g1 = d->g1; p->npar = d->npar;
  for (int e = 0; e < d->n * (1 + d->g1); ++e)
    if (d->ze1_ptr[e + 1] > d->ze1_ptr[e]) p->tube_ent.push_back(e);
  p->aux.n_nz = (int)p->tube_ent.size();
  p->aux.n = d->n; p->aux.m = d->m; p->aux.N = d->horizon; p->aux.nv = d->nv; p->aux.g1 = d->g1;
  return TZ_OK;
}

// Everything of tz_program_create that runs on the host: validation, bucket choice, packing, tables.  No CUDA call.
static int build_program_host(const TzProgramDesc* d, TzProgram* p, HostImage& img) {
  TZ_REQUIRE(d != nullptr, "null argument");
  TZ_REQUIRE(d->n >= 1 && d->n <= kMaxN && d->m >= 1 && d->m <= kMaxM, "dim_x must be 1..%d and dim_u 1..%d", kMaxN, kMaxM);
  TZ_REQUIRE(d->npar == 2 * d->n, "npar must be 2*dim_x");
  TZ_REQUIRE(d->nv == d->horizon * d->m && d->nv <= 16 && d->nz >= d->nv, "bad nv/nz");
  TZ_REQUIRE(d->nc >= 0 && d->na >= 0 && d->nchk >= 0 && d->g1 >= 0 && d->nterms >= 0 && d->nkink >= 0 && d->nkink <= d->nc,
             "negative size in the program descriptor");
  TZ_REQUIRE(d->ze1_ptr && d->ze1_ptr[0] == 0, "ze1_ptr[0] must be 0");
  for (int e = 0; e < d->n * (1 + d->g1); ++e)
    TZ_REQUIRE(d->ze1_ptr[e + 1] >= d->ze1_ptr[e], "ze1_ptr must be non-decreasing (entry %d)", e);
  TZ_REQUIRE(d->ze1_ptr[d->n * (1 + d->g1)] == d->nterms, "ze1_ptr[n(1+g1)] must equal nterms");
  int rc = TZ_ERANGE;
#define TZ_TRY(BK, ID) \
  if (rc == TZ_ERANGE && fits<BK>(*d)) rc = create_bucket<BK>(*d, p, ID, img);
  TZ_TRY(B0, 0) TZ_TRY(B1, 1) TZ_TRY(B2, 2) TZ_TRY(B3, 3)
#undef TZ_TRY
  if (rc == TZ_ERANGE && big_fits(*d)) return use_big_path(d, p);
  if (rc != TZ_OK) {
    if (rc == TZ_ERANGE) {
      const RowClasses c = classify(*d, nullptr);
      return fail(TZ_ERANGE, "program (nz=%d rows: %d two-sided, %d upper, %d lower; npar=%d general atoms=%d nchk=%d) "
                  "exceeds every compiled bucket", d->nz, c.n2, c.nu, c.nl, d->npar, general_atoms(*d, nullptr), d->nchk);
    }
    return rc;
  }
  p->nz = d->nz; p->nc = d->nc; p->n = d->n; p->m = d->m; p->N = d->horizon; p->nv = d->nv; p->g1 = d->g1; p->npar = d->npar;
  // ---- run-time sized tables: XB, centre map of Ze[1], K, and the non-zero entries of Ze[1].Z.  Columns / indices
  // of the caller's w = [1; v (nv); xbar0 (n); e0 (n)] are remapped to the kernel's padded vector om (Bucket::OM_*).
  const int n = d->n, nwc = 1 + d->nv + d->npar, ld1 = 1 + d->g1, nent = n * ld1, NW = p->NW;
  auto omidx = [&](int j) {
    if (j == 0) return 0;
    if (j <= d->nv) return p->OM_V + (j - 1);
    const int k = j - 1 - d->nv;
    return k < n ? p->OM_P + k : p->OM_P + p->HP + (k - n);
  };
  const int nrows = (d->horizon + 1) * n;
  std::vector<double> XB((size_t)nrows * NW, 0.0), CZ((size_t)n * NW, 0.0), coef;
  std::vector<int32_t> ent, idx;
  for (int i = 0; i < nrows; ++i)
    for (int j = 0; j < nwc; ++j) XB[(size_t)i * NW + omidx(j)] = d->XB[(size_t)i * nwc + j];
  for (int e = 0; e < nent; ++e) {
    const int t0 = d->ze1_ptr[e], t1 = d->ze1_ptr[e + 1];
    for (int t = t0; t < t1; ++t)
      if (d->ze1_idx[t] < 0 || d->ze1_idx[t] >= nwc) return fail(TZ_EINVAL, "ze1_idx[%d] out of range", t);
    const int r = e / ld1, j = e % ld1;
    if (j == 0) {                        // centre column: its (possibly many) terms become om[OM_C + r]
      for (int t = t0; t < t1; ++t) CZ[(size_t)r * NW + omidx(d->ze1_idx[t])] += d->ze1_val[t];
      ent.push_back(e); idx.push_back(p->OM_C + r); coef.push_back(1.0);
    } else if (t1 - t0 == 1) {
      ent.push_back(e); idx.push_back(omidx(d->ze1_idx[t0])); coef.push_back(d->ze1_val[t0]);
    } else if (t1 - t0 > 1) {
      return fail(TZ_EINVAL, "generator entry %d of Ze[1] has %d terms: only single-term generator entries are supported "
                  "(boxed M_K / M_Delta)", e, t1 - t0);
    }
  }
  // zero runs of the dense Ze[1].Z: the rows between consecutive non-zero entries (fast_step_kernel writes each row once)
  std::vector<int32_t> zstart, zlen;
  {
    int next = 0;
    for (size_t i = 0; i <= ent.size(); ++i) {
      const int stop = i < ent.size() ? ent[i] : nent;
      if (stop > next) { zstart.push_back(next); zlen.push_back(stop - next); }
      next = stop + 1;
    }
  }
  const size_t nXB = XB.size(), nCZ = CZ.size(), nK = (size_t)d->m * n, nco = coef.size();
  // fast_step_kernel's tables, in the double part: the term table as 16-byte pairs (coef, idx | ent << 32) on an even offset,
  // then the zero runs as int32 pairs
  const size_t o_tt = (nXB + nCZ + nK + nco + 1) & ~(size_t)1;
  const size_t o_zrun = o_tt + 2 * nco;
  int zrun_split = 0;
  {
    int total = 0, acc = 0;
    for (int v : zlen) total += v;
    while (zrun_split < (int)zlen.size() && 2 * acc < total) acc += zlen[zrun_split++];
  }
  // ... and once more as a flat list of rows in two halves (fast_step_kernel: the two halves of a CTA, 16-byte index loads)
  std::vector<int32_t> zrow;
  int n_zrow_half = 0;
  {
    std::vector<int32_t> all;
    for (size_t i = 0; i < zstart.size(); ++i)
      for (int c = 0; c < zlen[i]; ++c) all.push_back(zstart[i] + c);
    const size_t h0 = (all.size() + 1) / 2, h1 = all.size() - h0;
    n_zrow_half = (int)((std::max(h0, h1) + 3) & ~(size_t)3);
    if (h1 == 0) n_zrow_half = all.empty() ? 0 : n_zrow_half;
    zrow.assign((size_t)2 * n_zrow_half, 0);
    for (int half = 0; half < 2 && !all.empty(); ++half) {
      const size_t b = half == 0 ? 0 : h0, cnt = half == 0 ? h0 : h1;
      for (int k = 0; k < n_zrow_half; ++k) {
        // (an empty second half repeats the first half's last row: storing a zero twice is harmless)
        const size_t src = cnt == 0 ? h0 - 1 : b + std::min((size_t)k, cnt - 1);
        zrow[(size_t)half * n_zrow_half + k] = all[src];
      }
    }
  }
  const size_t o_zrow = (o_zrun + zstart.size() + 1) & ~(size_t)1;
  const size_t ndbl = o_zrow + (size_t)n_zrow_half, nint = ent.size() + idx.size();
  const size_t smem_tab = (ndbl + (size_t)n * n + (size_t)n * d->m) * sizeof(double) + nint * sizeof(int32_t);
  if (smem_tab > kMaxTabBytes) {
    // the rows fit a register bucket but its tables do not fit the shared memory staged for them (n = 8, m = 4, N = 2 needs
    // 25 KiB): the generic path serves the program instead
    if (big_fits(*d)) {
      *p = TzProgram();
      img = HostImage();
      return use_big_path(d, p);
    }
    return fail(TZ_ERANGE, "program tables need %zu bytes of shared memory (limit %d)", smem_tab, kMaxTabBytes);
  }
  std::vector<unsigned char>& host = img.aux;
  host.assign(ndbl * sizeof(double) + nint * sizeof(int32_t) + 16, 0);
  double* hd = reinterpret_cast<double*>(host.data());
  std::memcpy(hd, XB.data(), nXB * sizeof(double));
  std::memcpy(hd + nXB, CZ.data(), nCZ * sizeof(double));
  std::memcpy(hd + nXB + nCZ, d->K, nK * sizeof(double));
  if (nco) std::memcpy(hd + nXB + nCZ + nK, coef.data(), nco * sizeof(double));
  int32_t* hi = reinterpret_cast<int32_t*>(hd + ndbl);
  if (!ent.empty()) std::memcpy(hi, ent.data(), ent.size() * sizeof(int32_t));
  if (!idx.empty()) std::memcpy(hi + ent.size(), idx.data(), idx.size() * sizeof(int32_t));
  for (size_t i = 0; i < nco; ++i) {
    hd[o_tt + 2 * i] = coef[i];
    const long long bits = (long long)(uint32_t)idx[i] | ((long long)ent[i] << 32);
    std::memcpy(&hd[o_tt + 2 * i + 1], &bits, sizeof(bits));
  }
  for (size_t i = 0; i < zstart.size(); ++i) {
    const int32_t pr[2] = {zstart[i], zlen[i]};
    std::memcpy(&hd[o_zrun + i], pr, sizeof(pr));
  }
  if (!zrow.empty()) std::memcpy(&hd[o_zrow], zrow.data(), zrow.size() * sizeof(int32_t));
  Aux& ax = p->aux;
  ax.tab = nullptr;                      // (set when the tables are uploaded)
  ax.n_dbl = (int)ndbl; ax.n_int = (int)nint;
  ax.o_XB = 0; ax.o_CZ = (int)nXB; ax.o_K = (int)(nXB + nCZ); ax.o_coef = (int)(nXB + nCZ + nK);
  ax.o_ent = 0; ax.o_idx = (int)ent.size();
  ax.o_tt = (int)o_tt; ax.o_zrun = (int)o_zrun; ax.n_zrun = (int)zstart.size();
  ax.zrun_split = zrun_split;
  ax.o_zrow = (int)o_zrow; ax.n_zrow_half = n_zrow_half;
  ax.n_nz = (int)ent.size();
  p->tube_ent = ent;
  ax.n = n; ax.m = d->m; ax.N = d->horizon; ax.nv = d->nv; ax.g1 = d->g1;
  p->smem_tab = (smem_tab + 15) & ~(size_t)15;
  return TZ_OK;
}

static int device_info(TzProgram* p) {
  int dev = 0;
  TZ_CUDA(cudaGetDevice(&dev));
  p->device = dev;
  TZ_CUDA(cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, dev));
  return TZ_OK;
}

extern "C" int tz_program_create(const TzProgramDesc* d, TzProgram** out) {
  TZ_REQUIRE(d && out, "null argument");
  TzProgram* p = new (std::nothrow) TzProgram();
  if (!p) return fail(TZ_ENOMEM, "out of host memory");
  HostImage img;
  int rc = build_program_host(d, p, img);
  if (rc == TZ_OK) rc = device_info(p);
  if (rc == TZ_OK && p->bucket == 4) rc = big_create(*d, &p->big);
  if (rc != TZ_OK) {
    delete p;
    return rc;
  }
  if (p->bucket == 4) {
    *out = p;
    return TZ_OK;
  }
  cudaError_t err = cudaMalloc(&p->packed_dev, img.packed.size());
  if (err == cudaSuccess) err = cudaMemcpy(p->packed_dev, img.packed.data(), img.packed.size(), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMalloc(&p->aux_dev, img.aux.size());
  if (err == cudaSuccess) err = cudaMemcpy(p->aux_dev, img.aux.data(), img.aux.size(), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    tz_program_destroy(p);              // (frees whatever was allocated before the failure)
    return fail(TZ_ECUDA, "program upload: %s", cudaGetErrorString(err));
  }
  p->aux.tab = reinterpret_cast<const double*>(p->aux_dev);
  *out = p;
  return TZ_OK;
}

extern "C" void tz_program_destroy(TzProgram* p) {
  if (!p) return;
  if (p->owns_device) {
    if (p->packed_dev) cudaFree(p->packed_dev);
    if (p->aux_dev) cudaFree(p->aux_dev);
  }
  if (p->big) big_destroy(p->big);
  delete p;
}

// ---- D programs of one structure created at once (the data-set axis: one program per data set): packed on the host,
// ONE device allocation and ONE copy for all images, one for all tables
struct TzProgramBatch {
  std::vector<TzProgram*> progs;          // views into the two allocations below (owns_device = false)
  void* packed_all = nullptr;
  void* aux_all = nullptr;
};

extern "C" void tz_program_batch_destroy(TzProgramBatch* b) {
  if (!b) return;
  for (TzProgram* p : b->progs) delete p;
  if (b->packed_all) cudaFree(b->packed_all);
  if (b->aux_all) cudaFree(b->aux_all);
  delete b;
}

extern "C" int tz_program_create_batch(const TzProgramDesc* descs, int32_t D, TzProgramBatch** out) {
  TZ_REQUIRE(descs && out && D >= 1, "null argument / empty batch");
  TzProgramBatch* b = new (std::nothrow) TzProgramBatch();
  if (!b) return fail(TZ_ENOMEM, "out of host memory");
  std::vector<unsigned char> packed_h, aux_h;
  size_t pstride = 0, astride = 0;
  int rc = TZ_OK;
  for (int d = 0; d < D && rc == TZ_OK; ++d) {
    TzProgram* p = new (std::nothrow) TzProgram();
    if (!p) { rc = fail(TZ_ENOMEM, "out of host memory"); break; }
    p->owns_device = false;
    b->progs.push_back(p);
    HostImage img;
    rc = build_program_host(&descs[d], p, img);
    if (rc == TZ_OK && p->bucket == 4) rc = fail(TZ_ERANGE, "programs of the generic large-program path cannot be batched");
    if (rc != TZ_OK) break;
    if (d == 0) {
      pstride = (img.packed.size() + 255) & ~(size_t)255;
      astride = (img.aux.size() + 255) & ~(size_t)255;
      packed_h.assign(pstride * (size_t)D, 0);
      aux_h.assign(astride * (size_t)D, 0);
    }
    const TzProgram* p0 = b->progs[0];
    if (p->bucket != p0->bucket || img.packed.size() > pstride || img.aux.size() > astride || p->smem_tab != p0->smem_tab) {
      rc = fail(TZ_EINVAL, "program %d of the batch does not have the structure of program 0", d);
      break;
    }
    std::memcpy(packed_h.data() + pstride * (size_t)d, img.packed.data(), img.packed.size());
    std::memcpy(aux_h.data() + astride * (size_t)d, img.aux.data(), img.aux.size());
  }
  if (rc == TZ_OK) {
    cudaError_t err = cudaMalloc(&b->packed_all, packed_h.size());
    if (err == cudaSuccess) err = cudaMemcpy(b->packed_all, packed_h.data(), packed_h.size(), cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMalloc(&b->aux_all, aux_h.size());
    if (err == cudaSuccess) err = cudaMemcpy(b->aux_all, aux_h.data(), aux_h.size(), cudaMemcpyHostToDevice);
    if (err != cudaSuccess) rc = fail(TZ_ECUDA, "program batch upload: %s", cudaGetErrorString(err));
  }
  for (int d = 0; d < D && rc == TZ_OK; ++d) {
    TzProgram* p = b->progs[d];
    rc = device_info(p);
    p->packed_dev = static_cast<unsigned char*>(b->packed_all) + pstride * (size_t)d;
    p->aux_dev = static_cast<unsigned char*>(b->aux_all) + astride * (size_t)d;
    p->aux.tab = reinterpret_cast<const double*>(p->aux_dev);
  }
  if (rc != TZ_OK) {
    tz_program_batch_destroy(b);
    return rc;
  }
  *out = b;
  return TZ_OK;
}

extern "C" const TzProgram* tz_program_batch_get(const TzProgramBatch* b, int32_t d) {
  if (!b || d < 0 || d >= (int32_t)b->progs.size()) return nullptr;
  return b->progs[d];
}

extern "C" int tz_program_bucket(const TzProgram* p, char* buf, size_t cap) {
  TZ_REQUIRE(p && buf && cap > 0, "null argument");
  snprintf(buf, cap, "B%d(NZ=%d,NC=%d,G=%d)", p->bucket, p->NZ, p->NC, p->G);
  return p->bucket;
}

extern "C" int tz_program_warm_rows(const TzProgram* p) {
  if (!p) return fail(TZ_EINVAL, "null program");
  if (p->bucket == 4) return 1;           // (the generic large-program path starts cold: no warm-start rows)
  return p->NZ + p->NC + p->G + 1;        // x | y | activity words | valid flag
}

static void program_dims(const TzProgram* p, int32_t* out) {
  out[0] = p->n; out[1] = p->m; out[2] = p->nv; out[3] = (p->N + 1) * p->n; out[4] = p->n * (1 + p->g1); out[5] = p->aux.n_nz;
  out[6] = tz_program_warm_rows(p); out[7] = p->device;
}

extern "C" int tz_program_dims(const TzProgram* p, int32_t* out8) {
  TZ_REQUIRE(p && out8, "null argument");
  program_dims(p, out8);
  return TZ_OK;
}

extern "C" void tz_solver_opts_default(TzSolverOpts* o) {
  if (!o) return;
  o->rho = 0.1; o->rho_active = 100.0; o->rho_inactive = 0.1; o->sigma = 1e-6; o->alpha = 1.6;
  o->eps_abs = 1e-6; o->eps_rel = 1e-6; o->max_iter = 4000; o->check_every = 8; o->polish = 3; o->warm_start = 0;
  o->cert_first = 3;
  o->tube_packed = 0;
  o->hot_path = 1;
}

static SolverParams to_params(const TzSolverOpts* o) {
  TzSolverOpts d;
  tz_solver_opts_default(&d);
  if (o) d = *o;
  return SolverParams{d.rho, d.rho_active, d.rho_inactive, d.sigma, d.alpha, d.eps_abs, d.eps_rel,
                      d.max_iter, d.check_every, d.polish, d.warm_start, d.cert_first, d.tube_packed != 0 ? 1 : 0,
                      d.hot_path != 0 ? 1 : 0};
}

// two scenarios per lane in the output phase need 16-byte aligned rows: S, ld even and aligned base pointers
static int vec2_ok(const StepArgs& a) {
  const void* ptrs[] = {a.x, a.xbar, a.e, a.noise, a.x_restart, a.cost, a.v, a.xbar_traj, a.ze1, a.u_out, a.xbar0, a.e0, a.x_hist, a.xbar_hist, a.e_hist,
                        a.AB_true};
  bool ok = (a.S % 2 == 0) && (a.ld % 2 == 0);
  for (const void* q : ptrs) ok = ok && ((reinterpret_cast<uintptr_t>(q) & 15u) == 0);
  ok = ok && ((reinterpret_cast<uintptr_t>(a.status) & 7u) == 0) && ((reinterpret_cast<uintptr_t>(a.iters) & 7u) == 0);
  return ok ? 1 : 0;
}

// What a launch over one program and over a program set (program p the first of the set) do before choosing the kernels:
// the device check, the output layout (vec2), the solver options, and whether to take the hot path.  The hot path is the hint
// mode of the two-variable programs: fast_step_kernel (one thread per scenario, closed-form certificate) decides every
// scenario whose hint still holds; the 16-scenario tiles it defers are listed in the warm-start scratch (rows 2G: counters,
// 2G + 1: list) and solved by the step kernel right behind it.  Batches below kHotMinBatch scenarios and fused runs stay on
// the step kernel: one launch instead of two -- batch-1 latency.
static int prepare(const TzProgram* p, const char* what, const TzSolverOpts* o, const StepArgs& a_in, StepArgs* a, SolverParams* sp,
                   bool* hot) {
  int cur = -1;
  TZ_CUDA(cudaGetDevice(&cur));
  TZ_REQUIRE(cur == p->device, "the %s was created on CUDA device %d, the current device is %d", what, p->device, cur);
  *a = a_in;
  a->vec2 = vec2_ok(*a);
  *sp = to_params(o);
  TZ_REQUIRE(sp->max_iter >= 1 && sp->rho > 0 && sp->rho_act > 0 && sp->rho_inact > 0 && sp->alpha > 0 && sp->alpha < 2,
             "bad solver options");
  *hot = p->bucket == 0 && sp->hot && sp->warm == 2 && a->warm != nullptr && a->q_in == nullptr && a->S >= kHotMinBatch &&
         a->nsteps <= 1;
  if (*hot) {
    a->defer = reinterpret_cast<int32_t*>(a->warm + (int64_t)(2 * B0::G) * a->ld);
    a->defer_list = reinterpret_cast<int32_t*>(a->warm + (int64_t)(2 * B0::G + 1) * a->ld);
    a->list_mode = 0;
  }
  return TZ_OK;
}

static int launch(const TzProgram* p, const TzSolverOpts* o, const StepArgs& a_in, void* stream) {
  TZ_REQUIRE(p != nullptr, "null program");
  TZ_REQUIRE(a_in.S >= 0, "negative batch");
  if (a_in.S == 0) return TZ_OK;
  StepArgs a;
  SolverParams sp;
  bool hot;
  if (const int rc = prepare(p, "program", o, a_in, &a, &sp, &hot)) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (hot) {
    if (const int rc = launch_fast<B0>(p, sp, a, st)) return rc;
    a.list_mode = 1;
    return launch_bucket<B0>(p, sp, a, st);
  }
  switch (p->bucket) {
    case 4:
      TZ_REQUIRE(a.q_in == nullptr, "tz_qp_solve is not available for programs of the generic large-program path");
      return big_launch(p->big, sp, a, st);
    case 0: return launch_bucket<B0>(p, sp, a, st);
    case 1: return launch_bucket<B1>(p, sp, a, st);
    case 2: return launch_bucket<B2>(p, sp, a, st);
    case 3: return launch_bucket<B3>(p, sp, a, st);
  }
  return fail(TZ_EINVAL, "corrupt program handle");
}

extern "C" int tz_solve(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, const double* xbar0,
                        const double* e0, double* cost, double* v, double* xbar_traj, double* ze1, int32_t* status,
                        int32_t* iters, double* warm, void* stream) {
  TZ_REQUIRE(S == 0 || (xbar0 && e0 && status), "xbar0, e0 and status are required");
  StepArgs a{};
  a.S = S; a.ld = S; a.xbar0 = xbar0; a.e0 = e0; a.cost = cost; a.v = v; a.xbar_traj = xbar_traj; a.ze1 = ze1;
  a.status = status; a.iters = iters; a.warm = warm;
  return launch(prog, opts, a, stream);
}

// The arguments of one closed-loop step.  The plant is either shared (A_true, B_true) or, with `plants` (the _plants entry
// points), per scenario (AB_true); the arguments are checked before any CUDA call.
static int closed_loop_args(int64_t S, double* x, double* xbar, double* e, const double* noise, const double* x_restart, bool plants,
                            const double* A_true, const double* B_true, const double* AB_true, double* cost, double* v,
                            double* xbar_traj, double* ze1, double* u_out, int32_t* status, int32_t* iters, double* warm,
                            double* stats, StepArgs* out) {
  if (plants)
    TZ_REQUIRE(S == 0 || (x && xbar && e && AB_true && status), "x, xbar, e, AB_true, status are required");
  else
    TZ_REQUIRE(S == 0 || (x && xbar && e && A_true && B_true && status), "x, xbar, e, A_true, B_true, status are required");
  StepArgs a{};
  a.S = S; a.ld = S; a.xbar0 = xbar; a.e0 = e; a.x = x; a.xbar = xbar; a.e = e; a.noise = noise; a.x_restart = x_restart; a.A_true = A_true; a.B_true = B_true;
  a.cost = cost; a.v = v; a.xbar_traj = xbar_traj; a.ze1 = ze1; a.u_out = u_out; a.status = status; a.iters = iters;
  a.warm = warm; a.stats = stats;
  a.AB_true = AB_true;
  *out = a;
  return TZ_OK;
}

extern "C" int tz_closed_loop_step(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, double* x, double* xbar,
                                   double* e, const double* noise, const double* x_restart, const double* A_true,
                                   const double* B_true,
                                   double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                   int32_t* status, int32_t* iters, double* warm, double* stats, void* stream) {
  StepArgs a;
  if (const int rc = closed_loop_args(S, x, xbar, e, noise, x_restart, false, A_true, B_true, nullptr, cost, v, xbar_traj, ze1, u_out,
                                      status, iters, warm, stats, &a)) return rc;
  return launch(prog, opts, a, stream);
}

extern "C" int tz_closed_loop_step_plants(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, double* x, double* xbar,
                                          double* e, const double* noise, const double* x_restart, const double* AB_true,
                                          double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                          int32_t* status, int32_t* iters, double* warm, double* stats, void* stream) {
  StepArgs a;
  if (const int rc = closed_loop_args(S, x, xbar, e, noise, x_restart, true, nullptr, nullptr, AB_true, cost, v, xbar_traj, ze1, u_out,
                                      status, iters, warm, stats, &a)) return rc;
  return launch(prog, opts, a, stream);
}

// ---- fused run: K closed-loop steps in one launch (small batches: the launch per step is what the step costs) -----------
// Of one program (prog, tz_closed_loop_run*) or of a program set (set, tz_closed_loop_run_set*, which check it; prog is then NULL).
static int launch_set(const TzProgramSet* s, const TzSolverOpts* o, const StepArgs& a_in, void* stream);

static int closed_loop_run(const TzProgram* prog, const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, int32_t nsteps,
                           double* x, double* xbar, double* e, const double* noise, const double* x_restart, bool plants,
                           const double* A_true, const double* B_true, const double* AB_true, double* cost, double* v,
                           double* xbar_traj, double* ze1, double* u_out, double* x_hist, double* xbar_hist, double* e_hist,
                           int32_t* status, int32_t* iters, double* warm, double* stats, void* stream) {
  TZ_REQUIRE(prog != nullptr || set != nullptr, "null program");
  TZ_REQUIRE(nsteps >= 1, "nsteps must be >= 1");
  StepArgs a;
  if (const int rc = closed_loop_args(S, x, xbar, e, noise, x_restart, plants, A_true, B_true, AB_true, cost, v, xbar_traj, ze1, u_out,
                                      status, iters, warm, stats, &a)) return rc;
  a.nsteps = nsteps; a.x_hist = x_hist; a.xbar_hist = xbar_hist; a.e_hist = e_hist;
  // (two-scenarios-per-lane output: vec2_ok wants an even batch, and then every per-step block starts 16-byte aligned too)
  if (set != nullptr) return launch_set(set, opts, a, stream);   // (a set holds register-bucket programs only)
  TZ_REQUIRE(prog->bucket >= 0 && prog->bucket <= 3, "tz_closed_loop_run serves the register-bucket programs (up to 12 variables)");
  return launch(prog, opts, a, stream);
}

extern "C" int tz_closed_loop_run(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x, double* xbar,
                                  double* e, const double* noise, const double* x_restart, const double* A_true,
                                  const double* B_true, double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                  double* x_hist, double* xbar_hist, double* e_hist, int32_t* status, int32_t* iters, double* warm,
                                  double* stats, void* stream) {
  return closed_loop_run(prog, nullptr, opts, S, nsteps, x, xbar, e, noise, x_restart, false, A_true, B_true, nullptr, cost, v,
                         xbar_traj, ze1, u_out, x_hist, xbar_hist, e_hist, status, iters, warm, stats, stream);
}

extern "C" int tz_closed_loop_run_plants(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x,
                                         double* xbar, double* e, const double* noise, const double* x_restart, const double* AB_true,
                                         double* cost, double* v, double* xbar_traj, double* ze1, double* u_out, double* x_hist,
                                         double* xbar_hist, double* e_hist, int32_t* status, int32_t* iters, double* warm,
                                         double* stats, void* stream) {
  return closed_loop_run(prog, nullptr, opts, S, nsteps, x, xbar, e, noise, x_restart, true, nullptr, nullptr, AB_true, cost, v,
                         xbar_traj, ze1, u_out, x_hist, xbar_hist, e_hist, status, iters, warm, stats, stream);
}

// ---- tube pattern (packed Ze[1].Z) ------------------------------------------------------------------
extern "C" int tz_program_tube_pattern(const TzProgram* p, int32_t* entries_host, int32_t cap) {
  if (!p) return fail(TZ_EINVAL, "null program");
  const int nnz = p->aux.n_nz;
  if (entries_host) {
    TZ_REQUIRE(cap >= nnz, "tube pattern needs %d entries (cap %d)", nnz, cap);
    std::memcpy(entries_host, p->tube_ent.data(), (size_t)nnz * sizeof(int32_t));
  }
  return nnz;
}

// ---- data-set axis: program sets ----------------------------------------------------------------------
struct TzProgramSet {
  std::vector<const TzProgram*> progs;
  std::vector<int64_t> begin;          // nprog + 1
  tz::SetEntry* entries_dev = nullptr;
  int32_t* tile_prog_dev = nullptr;    // program of every global 16-scenario tile (the hot path: fast_step_kernel over a set)
  int block = 16;                      // largest of 128 / 64 / 32 / 16 that divides every program's first scenario
  int64_t max_scen = 0, total_tiles = 0;
};

extern "C" int tz_program_set_create(const TzProgram* const* progs, int32_t nprog, const int64_t* begin, TzProgramSet** out) {
  TZ_REQUIRE(progs && begin && out && nprog >= 1, "null argument / empty set");
  const TzProgram* p0 = progs[0];
  TZ_REQUIRE(p0 != nullptr, "null program 0");
  TZ_REQUIRE(begin[0] == 0, "begin[0] must be 0");
  std::vector<tz::SetEntry> ent((size_t)nprog);
  int64_t mx = 0, tiles = 0;
  for (int j = 0; j < nprog; ++j) {
    const TzProgram* p = progs[j];
    TZ_REQUIRE(p != nullptr, "null program %d", j);
    const Aux &a = p->aux, &b = p0->aux;
    // one kernel instance and one table layout serve the whole set: the programs must be the same problem (dimensions,
    // horizon, cost and constraint structure) built from different data
    TZ_REQUIRE(p->bucket != 4, "programs of the generic large-program path cannot be combined into a set");
    TZ_REQUIRE(p->bucket == p0->bucket && p->smem_tab == p0->smem_tab && a.n_dbl == b.n_dbl && a.n_int == b.n_int &&
               a.o_XB == b.o_XB && a.o_CZ == b.o_CZ && a.o_K == b.o_K && a.o_coef == b.o_coef && a.o_ent == b.o_ent &&
               a.o_idx == b.o_idx && a.o_tt == b.o_tt && a.o_zrun == b.o_zrun && a.n_zrun == b.n_zrun && a.zrun_split == b.zrun_split && a.o_zrow == b.o_zrow && a.n_zrow_half == b.n_zrow_half && a.n_nz == b.n_nz && a.n == b.n && a.m == b.m && a.N == b.N && a.nv == b.nv && a.g1 == b.g1,
               "program %d does not have the structure of program 0 (bucket / table sizes differ)", j);
    TZ_REQUIRE(p->tube_ent == p0->tube_ent, "program %d: Ze[1] has a different sparsity pattern than program 0", j);
    const int64_t cnt = begin[j + 1] - begin[j];
    TZ_REQUIRE(cnt >= 0, "begin[] must be non-decreasing");
    TZ_REQUIRE(begin[j] % 16 == 0, "begin[%d] = %lld: the scenarios of a program must start on a multiple of 16", j,
               (long long)begin[j]);
    ent[j] = tz::SetEntry{p->packed_dev, a.tab, begin[j], begin[j + 1], tiles};
    tiles += (cnt + TZ_SPO_MIN - 1) / TZ_SPO_MIN;             // (every bucket has output tiles of TZ_SPO_MIN scenarios)
    if (cnt > mx) mx = cnt;
  }
  TzProgramSet* s = new (std::nothrow) TzProgramSet();
  if (!s) return fail(TZ_ENOMEM, "out of host memory");
  s->progs.assign(progs, progs + nprog);
  s->begin.assign(begin, begin + nprog + 1);
  s->max_scen = mx;
  s->total_tiles = tiles;
  // tile -> program (programs start on whole tiles; an empty program owns no tile)
  std::vector<int32_t> tile_prog((size_t)((begin[nprog] + TZ_SPO_MIN - 1) / TZ_SPO_MIN) + 1, nprog - 1);
  s->block = 128;
  for (int j = 0; j < nprog; ++j) {
    for (int64_t t = begin[j] / TZ_SPO_MIN; t < (begin[j + 1] + TZ_SPO_MIN - 1) / TZ_SPO_MIN; ++t) tile_prog[(size_t)t] = j;
    if (begin[j + 1] > begin[j])
      while (s->block > 16 && begin[j] % s->block != 0) s->block /= 2;
  }
  cudaError_t err = cudaMalloc(&s->entries_dev, ent.size() * sizeof(tz::SetEntry));
  if (err == cudaSuccess) err = cudaMemcpy(s->entries_dev, ent.data(), ent.size() * sizeof(tz::SetEntry), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMalloc(&s->tile_prog_dev, tile_prog.size() * sizeof(int32_t));
  if (err == cudaSuccess)
    err = cudaMemcpy(s->tile_prog_dev, tile_prog.data(), tile_prog.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    if (s->entries_dev) cudaFree(s->entries_dev);
    if (s->tile_prog_dev) cudaFree(s->tile_prog_dev);
    delete s;
    return fail(TZ_ECUDA, "program set upload: %s", cudaGetErrorString(err));
  }
  *out = s;
  return TZ_OK;
}

extern "C" void tz_program_set_destroy(TzProgramSet* s) {
  if (!s) return;
  if (s->entries_dev) cudaFree(s->entries_dev);
  if (s->tile_prog_dev) cudaFree(s->tile_prog_dev);
  delete s;
}

extern "C" int64_t tz_program_set_scenarios(const TzProgramSet* s) { return s ? s->begin.back() : -1; }

extern "C" int tz_program_set_dims(const TzProgramSet* s, int32_t* out8) {
  TZ_REQUIRE(s && out8 && !s->progs.empty(), "null argument");
  program_dims(s->progs[0], out8);
  return TZ_OK;
}

static int launch_set(const TzProgramSet* s, const TzSolverOpts* o, const StepArgs& a_in, void* stream) {
  TZ_REQUIRE(s != nullptr, "null program set");
  TZ_REQUIRE(a_in.S == s->begin.back(), "batch of %lld scenarios, the set was created for %lld", (long long)a_in.S,
             (long long)s->begin.back());
  if (a_in.S == 0) return TZ_OK;
  const TzProgram* p0 = s->progs[0];
  const int np = (int)s->progs.size();
  // a fused run (tz_closed_loop_run_set, nsteps >= 1) takes step_kernel_set_run whatever the set and the batch: it is the
  // kernel that places the histories of every program, and prepare keeps a run of more than one step off the hot path
  const bool run = a_in.nsteps >= 1;
  if (np == 1 && !run) return launch(p0, o, a_in, stream);       // one program: exactly step_kernel (tiles strided over the grid)
  StepArgs a;
  SolverParams sp;
  bool hot;
  if (const int rc = prepare(p0, "program set", o, a_in, &a, &sp, &hot)) return rc;
  for (size_t j = 0; j + 1 < s->begin.size(); ++j)       // (every program starts on a multiple of 16 scenarios: alignment carries over)
    if ((s->begin[j + 1] - s->begin[j]) % 2 != 0) a.vec2 = 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (hot && !run) {
    // the hot path over a set: fast_step_kernel looks the program of every 16-scenario tile up, the tiles it defers are
    // solved by step_kernel_set_list
    if (const int rc = launch_fast_set<B0>(p0, sp, a, s->entries_dev, s->tile_prog_dev, s->block, st)) return rc;
    a.list_mode = 1;
    return launch_bucket_set_list<B0>(p0, s->entries_dev, s->tile_prog_dev, sp, a, st);
  }
#define TZ_SET(BK) (run ? launch_bucket_set_run<BK> : launch_bucket_set<BK>)(p0, s->entries_dev, np, s->total_tiles, sp, a, st)
  switch (p0->bucket) {
    case 0: return TZ_SET(B0);
    case 1: return TZ_SET(B1);
    case 2: return TZ_SET(B2);
    case 3: return TZ_SET(B3);
  }
#undef TZ_SET
  return fail(TZ_EINVAL, "corrupt program handle");
}

extern "C" int tz_solve_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, const double* xbar0,
                            const double* e0, double* cost, double* v, double* xbar_traj, double* ze1, int32_t* status,
                            int32_t* iters, double* warm, void* stream) {
  TZ_REQUIRE(S == 0 || (xbar0 && e0 && status), "xbar0, e0 and status are required");
  StepArgs a{};
  a.S = S; a.ld = S; a.xbar0 = xbar0; a.e0 = e0; a.cost = cost; a.v = v; a.xbar_traj = xbar_traj; a.ze1 = ze1;
  a.status = status; a.iters = iters; a.warm = warm;
  return launch_set(set, opts, a, stream);
}

extern "C" int tz_closed_loop_step_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, double* x, double* xbar,
                                       double* e, const double* noise, const double* x_restart, const double* A_true,
                                       const double* B_true, double* cost, double* v, double* xbar_traj, double* ze1,
                                       double* u_out, int32_t* status, int32_t* iters, double* warm, double* stats,
                                       void* stream) {
  StepArgs a;
  if (const int rc = closed_loop_args(S, x, xbar, e, noise, x_restart, false, A_true, B_true, nullptr, cost, v, xbar_traj, ze1, u_out,
                                      status, iters, warm, stats, &a)) return rc;
  return launch_set(set, opts, a, stream);
}

extern "C" int tz_closed_loop_step_set_plants(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, double* x, double* xbar,
                                              double* e, const double* noise, const double* x_restart, const double* AB_true,
                                              double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                              int32_t* status, int32_t* iters, double* warm, double* stats, void* stream) {
  StepArgs a;
  if (const int rc = closed_loop_args(S, x, xbar, e, noise, x_restart, true, nullptr, nullptr, AB_true, cost, v, xbar_traj, ze1, u_out,
                                      status, iters, warm, stats, &a)) return rc;
  return launch_set(set, opts, a, stream);
}

extern "C" int tz_closed_loop_run_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x,
                                      double* xbar, double* e, const double* noise, const double* x_restart, const double* A_true,
                                      const double* B_true, double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                      double* x_hist, double* xbar_hist, double* e_hist, int32_t* status, int32_t* iters, double* warm,
                                      double* stats, void* stream) {
  TZ_REQUIRE(set != nullptr, "null program set");
  return closed_loop_run(nullptr, set, opts, S, nsteps, x, xbar, e, noise, x_restart, false, A_true, B_true, nullptr, cost, v,
                         xbar_traj, ze1, u_out, x_hist, xbar_hist, e_hist, status, iters, warm, stats, stream);
}

extern "C" int tz_closed_loop_run_set_plants(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x,
                                             double* xbar, double* e, const double* noise, const double* x_restart,
                                             const double* AB_true, double* cost, double* v, double* xbar_traj, double* ze1,
                                             double* u_out, double* x_hist, double* xbar_hist, double* e_hist, int32_t* status,
                                             int32_t* iters, double* warm, double* stats, void* stream) {
  TZ_REQUIRE(set != nullptr, "null program set");
  return closed_loop_run(nullptr, set, opts, S, nsteps, x, xbar, e, noise, x_restart, true, nullptr, nullptr, AB_true, cost, v,
                         xbar_traj, ze1, u_out, x_hist, xbar_hist, e_hist, status, iters, warm, stats, stream);
}

extern "C" int tz_qp_solve(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, const double* q, const double* l,
                           const double* u, double* z, double* y, int32_t* status, int32_t* iters, void* stream) {
  TZ_REQUIRE(S == 0 || (q && l && u && z && status), "q, l, u, z, status are required");
  StepArgs a{};
  a.S = S; a.ld = S; a.q_in = q; a.l_in = l; a.u_in = u; a.z_out = z; a.y_out = y; a.status = status; a.iters = iters;
  TzSolverOpts o;
  tz_solver_opts_default(&o);
  if (opts) o = *opts;
  o.warm_start = 0;
  return launch(prog, &o, a, stream);
}

// ---- host-buffer variants: chunked H2D -> kernels -> D2H pipeline ---------------------------------
static size_t host_scratch_doubles(const TzProgram* p, int64_t S) {
  const size_t n = p->n, nent = (size_t)p->n * (1 + p->g1), nt = (size_t)(p->N + 1) * p->n;
  // A, B | x, xbar, e, noise | cost | v | xbar_traj | ze1 | status (as int32, rounded up) | warm rows (active-set hints /
  // ADMM iterate carried between calls when opts->warm_start != 0) | x_restart | u   (the last two: tz_closed_loop_run_host)
  return (size_t)S * (4 * n + 1 + p->nv + nt + nent + 1 + (size_t)tz_program_warm_rows(p) + n + p->m) + (size_t)(n * n + n * p->m) + 16;
}

extern "C" size_t tz_closed_loop_step_host_scratch_bytes(const TzProgram* prog, int64_t S) {
  if (!prog || S < 0) return 0;
  return host_scratch_doubles(prog, S) * sizeof(double);
}

namespace {
// the chunk streams are created once per host thread and device and reused by later calls (creating and destroying them
// cost tens of microseconds of every call); a thread that moves to another device gets that device's own pool
struct StreamPool {
  cudaStream_t s[16];
  cudaEvent_t ready = nullptr;      // plant matrices (and, resident mode, the state) uploaded on s[0]; the other chunk streams wait for it
  int n = 0;
};
constexpr int kMaxPoolDevices = 64;

StreamPool* stream_pool(int device, int nchunks) {
  static thread_local StreamPool pools[kMaxPoolDevices];
  if (device < 0 || device >= kMaxPoolDevices) return nullptr;
  StreamPool& pool = pools[device];
  if (!pool.ready && cudaEventCreateWithFlags(&pool.ready, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  while (pool.n < nchunks) {
    if (cudaStreamCreateWithFlags(&pool.s[pool.n], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    ++pool.n;
  }
  return &pool;
}

struct HostStep {
  int upload_state = 1;      // copy x, xbar, e (and x_restart) up before the step
  int download_state = 1;    // copy xbar and e down after the step (x always comes down)
  double *x, *xbar, *e;
  const double *x_restart, *noise, *A_true, *B_true;
  double *cost, *v, *traj, *ze1, *u;
  int32_t* status;
};

int closed_loop_host(const TzProgram* p, const TzSolverOpts* opts, int64_t S, const HostStep& hs, void* dev_scratch, int32_t nchunks) {
  const int64_t n = p->n, m = p->m, nent = (int64_t)p->n * (1 + p->g1), nt = (int64_t)(p->N + 1) * p->n, nv = p->nv;
  // packed tube (opts->tube_packed): only the entries of Ze[1].Z that are not structurally zero cross the bus
  const int64_t tube_rows = (opts && opts->tube_packed) ? (int64_t)p->aux.n_nz : nent;
  if (nchunks < 1) nchunks = 1;
  if (nchunks > 16) nchunks = 16;
  if ((int64_t)nchunks > S) nchunks = (int)S;
  double* d = reinterpret_cast<double*>(dev_scratch);
  double* dA = d; d += n * n;
  double* dB = d; d += n * m;
  d += (16 - ((n * n + n * m) % 16)) % 16;
  double *dx = d, *dxb = dx + n * S, *de = dxb + n * S, *dw = de + n * S, *dcost = dw + n * S, *dv = dcost + S,
         *dtraj = dv + nv * S, *dze = dtraj + nt * S;
  int32_t* dst = reinterpret_cast<int32_t*>(dze + nent * S);
  double* dwarm = dze + nent * S + S;      // behind the status words (S int32 <= S doubles)
  double* dxr = dwarm + (int64_t)tz_program_warm_rows(p) * S;
  double* du = dxr + n * S;
  const bool use_warm = opts && opts->warm_start != 0;
  int cur_dev = 0;
  TZ_CUDA(cudaGetDevice(&cur_dev));
  StreamPool* pool = stream_pool(cur_dev, nchunks);
  if (!pool) return fail(TZ_ECUDA, "closed_loop_host: cannot create the chunk streams on device %d", cur_dev);
  cudaStream_t* streams = pool->s;
  int rc = TZ_OK;
  cudaError_t err = cudaSuccess;
  if (hs.upload_state) {
    err = cudaMemcpyAsync(dA, hs.A_true, n * n * sizeof(double), cudaMemcpyHostToDevice, streams[0]);
    if (err == cudaSuccess) err = cudaMemcpyAsync(dB, hs.B_true, n * m * sizeof(double), cudaMemcpyHostToDevice, streams[0]);
  }
  if (err == cudaSuccess) err = cudaEventRecord(pool->ready, streams[0]);
  for (int c = 1; c < nchunks && err == cudaSuccess; ++c) err = cudaStreamWaitEvent(streams[c], pool->ready, 0);
  int64_t per = (S + nchunks - 1) / nchunks;
  per = (per + 15) & ~(int64_t)15;          // whole tiles, 16-byte aligned chunk starts
  // The device arrays are SoA with leading dimension S; a chunk [s0, s1) of a d x S array is d strided
  // segments, moved with one 2-D copy per array.
  auto h2d = [&](double* dev, const double* host, int64_t rows, int64_t s0, int64_t cnt, cudaStream_t st) {
    return cudaMemcpy2DAsync(dev + s0, S * sizeof(double), host + s0, S * sizeof(double), cnt * sizeof(double), rows,
                             cudaMemcpyHostToDevice, st);
  };
  auto d2h = [&](double* host, const double* dev, int64_t rows, int64_t s0, int64_t cnt, cudaStream_t st) {
    return cudaMemcpy2DAsync(host + s0, S * sizeof(double), dev + s0, S * sizeof(double), cnt * sizeof(double), rows,
                             cudaMemcpyDeviceToHost, st);
  };
  for (int c = 0; c < nchunks && err == cudaSuccess && rc == TZ_OK; ++c) {
    const int64_t s0 = (int64_t)c * per, cnt = (s0 + per <= S ? per : S - s0);
    if (cnt <= 0) break;
    cudaStream_t st = streams[c];
    if (hs.upload_state) {
      err = h2d(dx, hs.x, n, s0, cnt, st);
      if (err == cudaSuccess) err = h2d(dxb, hs.xbar, n, s0, cnt, st);
      if (err == cudaSuccess) err = h2d(de, hs.e, n, s0, cnt, st);
      if (err == cudaSuccess && hs.x_restart) err = h2d(dxr, hs.x_restart, n, s0, cnt, st);
    }
    if (err == cudaSuccess) err = h2d(dw, hs.noise, n, s0, cnt, st);
    if (err != cudaSuccess) break;
    // the chunk is its own batch of `cnt` scenarios inside arrays of leading dimension S
    StepArgs a{};
    a.S = cnt; a.ld = S;
    a.xbar0 = dxb + s0; a.e0 = de + s0; a.x = dx + s0; a.xbar = dxb + s0; a.e = de + s0; a.noise = dw + s0;
    a.x_restart = hs.x_restart ? dxr + s0 : nullptr;
    a.A_true = dA; a.B_true = dB;
    a.cost = hs.cost ? dcost + s0 : nullptr;
    a.v = hs.v ? dv + s0 : nullptr;
    a.xbar_traj = hs.traj ? dtraj + s0 : nullptr;
    a.ze1 = hs.ze1 ? dze + s0 : nullptr;
    a.u_out = hs.u ? du + s0 : nullptr;
    a.status = dst + s0;
    a.warm = use_warm ? dwarm + s0 : nullptr;
    rc = launch(p, opts, a, st);
    if (rc != TZ_OK) break;
    err = d2h(hs.x, dx, n, s0, cnt, st);
    if (err == cudaSuccess && hs.download_state) err = d2h(hs.xbar, dxb, n, s0, cnt, st);
    if (err == cudaSuccess && hs.download_state) err = d2h(hs.e, de, n, s0, cnt, st);
    if (err == cudaSuccess && hs.cost) err = d2h(hs.cost, dcost, 1, s0, cnt, st);
    if (err == cudaSuccess && hs.v) err = d2h(hs.v, dv, nv, s0, cnt, st);
    if (err == cudaSuccess && hs.traj) err = d2h(hs.traj, dtraj, nt, s0, cnt, st);
    if (err == cudaSuccess && hs.ze1) err = d2h(hs.ze1, dze, tube_rows, s0, cnt, st);
    if (err == cudaSuccess && hs.u) err = d2h(hs.u, du, m, s0, cnt, st);
    if (err == cudaSuccess)
      err = cudaMemcpyAsync(hs.status + s0, dst + s0, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
  }
  for (int c = 0; c < nchunks; ++c) {
    cudaError_t e2 = cudaStreamSynchronize(streams[c]);
    if (err == cudaSuccess) err = e2;
  }
  if (rc != TZ_OK) return rc;
  if (err != cudaSuccess) return fail(TZ_ECUDA, "closed_loop_host: %s", cudaGetErrorString(err));
  return TZ_OK;
}
}  // namespace

extern "C" int tz_closed_loop_step_host(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, double* x_host,
                                        double* xbar_host, double* e_host, const double* noise_host,
                                        const double* A_true_host, const double* B_true_host, double* cost_host,
                                        double* v_host, double* xbar_traj_host, double* ze1_host, int32_t* status_host,
                                        void* dev_scratch, int32_t nchunks) {
  TZ_REQUIRE(prog && dev_scratch, "null argument");
  TZ_REQUIRE(S == 0 || (x_host && xbar_host && e_host && noise_host && A_true_host && B_true_host && status_host),
             "x, xbar, e, noise, A_true, B_true, status are required");
  // the resident path with the state uploaded before and downloaded after the step (flags 3), no restart state, no u
  return tz_closed_loop_run_host(prog, opts, S, 3, x_host, xbar_host, e_host, nullptr, noise_host, A_true_host, B_true_host, cost_host,
                                 v_host, xbar_traj_host, ze1_host, nullptr, status_host, dev_scratch, nchunks);
}

extern "C" int tz_closed_loop_run_host(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t flags, double* x_host,
                                       double* xbar_host, double* e_host, const double* x_restart_host, const double* noise_host,
                                       const double* A_true_host, const double* B_true_host, double* cost_host, double* v_host,
                                       double* xbar_traj_host, double* ze1_host, double* u_host, int32_t* status_host,
                                       void* dev_scratch, int32_t nchunks) {
  TZ_REQUIRE(prog && dev_scratch, "null argument");
  const bool up = (flags & 1) != 0, down = (flags & 2) != 0;
  TZ_REQUIRE(S == 0 || (x_host && noise_host && status_host), "x, noise, status are required");
  TZ_REQUIRE(S == 0 || !up || (xbar_host && e_host && A_true_host && B_true_host),
             "flags & 1 (upload the state): xbar, e, A_true, B_true are required");
  TZ_REQUIRE(S == 0 || !down || (xbar_host && e_host), "flags & 2 (download xbar and e): xbar, e are required");
  if (S == 0) return TZ_OK;
  HostStep hs;
  hs.upload_state = up ? 1 : 0; hs.download_state = down ? 1 : 0;
  hs.x = x_host; hs.xbar = xbar_host; hs.e = e_host; hs.x_restart = x_restart_host; hs.noise = noise_host; hs.A_true = A_true_host;
  hs.B_true = B_true_host; hs.cost = cost_host; hs.v = v_host; hs.traj = xbar_traj_host; hs.ze1 = ze1_host; hs.u = u_host;
  hs.status = status_host;
  return closed_loop_host(prog, opts, S, hs, dev_scratch, nchunks);
}
