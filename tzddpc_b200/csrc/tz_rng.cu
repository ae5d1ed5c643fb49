// Counter-based random numbers for the scenario axes of the batched closed loop (SURVEY.md 8d: "all draws come from a
// documented Philox4x32 stream so that the CPU oracle and the GPU consume identical numbers").
//
//   Philox4x32-10 (Salmon et al., SC'11), key = (seed lo, seed hi),
//   counter = (scenario lo, scenario hi, t, (purpose << 16) | block)        -> 4 x 32 random bits = 2 draws
//   uniform draw  beta = 2 * (u64 >> 11) * 2^-53 - 1  in [-1, 1)            (Zonotope.sample, examples/2.pulley_sim.py:92)
//   vertex draw   beta = +-1 from the top bit of the same 64 bits           (random vertex of W, examples/utils.py:37)
// The scenario index is GLOBAL (scenario_offset + local index), so results do not depend on how scenarios are sharded
// over GPUs.  purposes: 0 closed-loop noise w_t, 1 data-set inputs u_t, 2 data-set noise, 3 initial state of the data set,
// 4 starting points of the gain-synthesis adversary, 5 samples of its robustness check (tz_gain.cu), 6 plants drawn from M_Sigma
// (tz_sample_plants: t = 0, draw g = k (T-1) + j for generator g of M_Sigma).
//
//   tz_sample_noise          w_t = c_W + G_W beta_t          for S scenarios, SoA n x S   (examples/2.pulley_sim.py:92)
//   tz_generate_trajectories examples/utils.py:6-45 batched over S data sets (quirk Q9 kept: the first returned state row
//                            is the origin), output AoS S x T x dim as tz_identify reads it; the _plants variant takes a
//                            plant per data set
//   tz_sample_plants         [A B] ~ U(M_Sigma) per scenario, SoA n(n+m) x S as tz_closed_loop_step_plants reads it
#include "tz_philox.cuh"

namespace tz {

__global__ void __launch_bounds__(256) noise_kernel(int64_t S, int64_t ld, int n, int gW, const double* __restrict__ WZ, int vertex,
                                                    uint64_t seed, int64_t scenario_offset, uint32_t t, double* __restrict__ out) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  double w[kMaxN];
  for (int r = 0; r < n; ++r) w[r] = WZ[(int64_t)r * (1 + gW)];
  for (int j = 0; j < gW; ++j) {
    const double b = draw(seed, (uint64_t)(scenario_offset + s), t, 0u, j, vertex != 0);
    for (int r = 0; r < n; ++r) w[r] = fma(WZ[(int64_t)r * (1 + gW) + 1 + j], b, w[r]);
  }
  for (int r = 0; r < n; ++r) out[(int64_t)r * ld + s] = w[r];
}

// PER: a plant per data set, A at A + s n n and B at B + s n m
template <bool PER = false>
__global__ void __launch_bounds__(128) gen_traj_kernel(int64_t S, int T, int n, int m, int g0, int gU, int gW,
                                                       const double* __restrict__ A, const double* __restrict__ B,
                                                       const double* __restrict__ X0Z, const double* __restrict__ UZ,
                                                       const double* __restrict__ WZ, uint64_t seed, int64_t scenario_offset,
                                                       double* __restrict__ U, double* __restrict__ X) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  if constexpr (PER) {
    A += s * n * n;
    B += s * n * m;
  }
  const uint64_t sid = (uint64_t)(scenario_offset + s);
  double x[kMaxN], xn[kMaxN], u[kMaxM];
  for (int r = 0; r < n; ++r) {                       // X[j, 0] = X0.sample()     (examples/utils.py:32)
    double acc = X0Z[(int64_t)r * (1 + g0)];
    for (int j = 0; j < g0; ++j) acc = fma(X0Z[(int64_t)r * (1 + g0) + 1 + j], draw(seed, sid, 0u, 3u, j, false), acc);
    x[r] = acc;
  }
  double* Us = U + s * (int64_t)T * m;
  double* Xs = X + s * (int64_t)T * n;
  for (int r = 0; r < n; ++r) Xs[r] = 0.0;            // quirk Q9: the returned Y[j, 0] stays zero (:32-40)
  for (int t = 0; t < T; ++t) {
    for (int k = 0; k < m; ++k) {                     // u = U.sample()           (:27)
      double acc = UZ[(int64_t)k * (1 + gU)];
      for (int j = 0; j < gU; ++j) acc = fma(UZ[(int64_t)k * (1 + gU) + 1 + j], draw(seed, sid, (uint32_t)t, 1u, j, false), acc);
      u[k] = acc;
      Us[(int64_t)t * m + k] = acc;
    }
    if (t + 1 < T) {                                  // x+ = A x + B u + (random vertex of W)   (:35-40)
      for (int r = 0; r < n; ++r) {
        double acc = WZ[(int64_t)r * (1 + gW)];
        for (int j = 0; j < gW; ++j) acc = fma(WZ[(int64_t)r * (1 + gW) + 1 + j], draw(seed, sid, (uint32_t)t, 2u, j, true), acc);
        for (int k = 0; k < n; ++k) acc = fma(A[r * n + k], x[k], acc);
        for (int k = 0; k < m; ++k) acc = fma(B[r * m + k], u[k], acc);
        xn[r] = acc;
      }
      for (int r = 0; r < n; ++r) { x[r] = xn[r]; Xs[(int64_t)(t + 1) * n + r] = xn[r]; }
    }
  }
}

// One thread per scenario: [A B] = AB_d - G_W R,  R[k, :] = sum_j beta_kj Pinv_d[j, :],  beta ~ U[-1, 1) -- a uniform point of the
// generator box of M_Sigma = (X1 - M_w) pinv([X0; U0]), whose generator g = k (T-1) + j is -G_W[:, k] Pinv_d[j, :] (SURVEY.md
// App. A.7; the rank-one structure of tz_gain.cu's robustness check).  A data-set index outside [0, D) gives a NaN plant.
__global__ void __launch_bounds__(128) sample_plants_kernel(int64_t S, int D, int T, int n, int m, int gW,
                                                            const double* __restrict__ AB, const double* __restrict__ Pinv,
                                                            const double* __restrict__ WZ, const int32_t* __restrict__ dataset,
                                                            uint64_t seed, int64_t scenario_offset, double* __restrict__ out) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const int d = dataset ? dataset[s] : 0;
  const int nm = n + m, Tm = T - 1;
  if (d < 0 || d >= D) {
    for (int i = 0; i < n * nm; ++i) out[(int64_t)i * S + s] = NAN;
    return;
  }
  const double* ABd = AB + (int64_t)d * n * nm;
  const double* Pd = Pinv + (int64_t)d * Tm * nm;
  const uint64_t sid = (uint64_t)(scenario_offset + s);
  double ab[kMaxN * (kMaxN + kMaxM)];
  for (int i = 0; i < n * nm; ++i) ab[i] = ABd[i];
  for (int k = 0; k < gW; ++k) {
    double r[kMaxN + kMaxM];
    for (int c = 0; c < nm; ++c) r[c] = 0.0;
    for (int j = 0; j < Tm; ++j) {
      const double b = draw(seed, sid, 0u, 6u, k * Tm + j, false);
      for (int c = 0; c < nm; ++c) r[c] = fma(b, Pd[(int64_t)j * nm + c], r[c]);
    }
    for (int i = 0; i < n; ++i) {
      const double g = WZ[(int64_t)i * (1 + gW) + 1 + k];
      for (int c = 0; c < nm; ++c) ab[i * nm + c] = fma(-g, r[c], ab[i * nm + c]);
    }
  }
  for (int i = 0; i < n * nm; ++i) out[(int64_t)i * S + s] = ab[i];
}

}  // namespace tz

using namespace tz;

extern "C" void tz_philox4x32_10_host(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out4) {
  uint32_t o[4];
  philox4x32_10(k0, k1, c0, c1, c2, c3, o);
  for (int i = 0; i < 4; ++i) out4[i] = o[i];
}

extern "C" int tz_sample_noise(int64_t S, int64_t ld, int32_t n, int32_t gW, const double* WZ, int32_t vertex, uint64_t seed,
                               int64_t scenario_offset, uint32_t t, double* out, void* stream) {
  TZ_REQUIRE(S >= 0 && ld >= S && n >= 1 && n <= kMaxN && gW >= 0 && gW <= 65535 * 2, "bad shape");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(WZ && out, "null pointer");
  noise_kernel<<<(unsigned)((S + 255) / 256), 256, 0, (cudaStream_t)stream>>>(S, ld, n, gW, WZ, vertex, seed, scenario_offset, t, out);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_generate_trajectories(int64_t S, int32_t T, int32_t n, int32_t m, int32_t g0, int32_t gU, int32_t gW,
                                        const double* A, const double* B, const double* X0Z, const double* UZ, const double* WZ,
                                        uint64_t seed, int64_t scenario_offset, double* U, double* X, void* stream) {
  TZ_REQUIRE(S >= 0 && T >= 2 && n >= 1 && n <= kMaxN && m >= 1 && m <= kMaxM && g0 >= 0 && gU >= 0 && gW >= 0, "bad shape");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(A && B && X0Z && UZ && WZ && U && X, "null pointer");
  gen_traj_kernel<false><<<(unsigned)((S + 127) / 128), 128, 0, (cudaStream_t)stream>>>(S, T, n, m, g0, gU, gW, A, B, X0Z, UZ, WZ, seed,
                                                                               scenario_offset, U, X);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_generate_trajectories_plants(int64_t S, int32_t T, int32_t n, int32_t m, int32_t g0, int32_t gU, int32_t gW,
                                               const double* A, const double* B, const double* X0Z, const double* UZ, const double* WZ,
                                               uint64_t seed, int64_t scenario_offset, double* U, double* X, void* stream) {
  TZ_REQUIRE(S >= 0 && T >= 2 && n >= 1 && n <= kMaxN && m >= 1 && m <= kMaxM && g0 >= 0 && gU >= 0 && gW >= 0, "bad shape");
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(A && B && X0Z && UZ && WZ && U && X, "null pointer");
  gen_traj_kernel<true><<<(unsigned)((S + 127) / 128), 128, 0, (cudaStream_t)stream>>>(S, T, n, m, g0, gU, gW, A, B, X0Z, UZ, WZ,
                                                                                      seed, scenario_offset, U, X);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}

extern "C" int tz_sample_plants(int64_t S, int32_t D, int32_t T, int32_t n, int32_t m, int32_t gW, const double* AB, const double* Pinv,
                                const double* WZ, const int32_t* dataset, uint64_t seed, int64_t scenario_offset, double* AB_out,
                                void* stream) {
  TZ_REQUIRE(S >= 0 && D >= 1 && T >= 2 && n >= 1 && n <= kMaxN && m >= 1 && m <= kMaxM && gW >= 0, "bad shape");
  // (draw g of a scenario is half g % 2 of counter block g / 2, and the block is 16 bits of the counter)
  TZ_REQUIRE((int64_t)gW * (T - 1) <= 2 * 65536, "gW (T-1) = %lld generators: at most 131072", (long long)gW * (T - 1));
  if (S == 0) return TZ_OK;
  TZ_REQUIRE(AB && Pinv && WZ && AB_out, "null pointer");
  sample_plants_kernel<<<(unsigned)((S + 127) / 128), 128, 0, (cudaStream_t)stream>>>(S, D, T, n, m, gW, AB, Pinv, WZ, dataset, seed,
                                                                                    scenario_offset, AB_out);
  TZ_CUDA(cudaGetLastError());
  return TZ_OK;
}
