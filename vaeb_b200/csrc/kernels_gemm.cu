// Instantiations + launch heuristics of the fp32 FFMA GEMM (gemm_simt.cuh).
#include "gemm_simt.cuh"
#include "launchers.h"

namespace {

// 64x64 tiles when they already fill the chip; 32x32 tiles for the skinny (M = 100) shapes so
// that more of the 148 SMs get a CTA.
inline bool use_big_tiles(int M, int N) {
  const long t = (long)((M + 63) / 64) * ((N + 63) / 64);
  return t >= 120;
}

template <bool TA, bool TB, bool ONES, bool DUAL, bool TWO, class Epi>
cudaError_t run_gemm(cudaStream_t st, int64_t* launches, const GemmOperands& g, const Epi& epi, float* partial,
                     int* n_col_tiles, bool force_big = false) {
  if (g.M <= 0 || g.N <= 0) return cudaSuccess;
  if (force_big || use_big_tiles(g.M, g.N)) {
    dim3 grid((g.N + 63) / 64, (g.M + 63) / 64);
    if (n_col_tiles) *n_col_tiles = grid.x;
    gemm_f32_kernel<64, 64, 4, 4, TA, TB, ONES, DUAL, TWO, Epi><<<grid, 256, 0, st>>>(g, epi, partial);
  } else {
    dim3 grid((g.N + 31) / 32, (g.M + 31) / 32);
    if (n_col_tiles) *n_col_tiles = grid.x;
    gemm_f32_kernel<32, 32, 2, 2, TA, TB, ONES, DUAL, TWO, Epi><<<grid, 256, 0, st>>>(g, epi, partial);
  }
  ++*launches;
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_dense_act(cudaStream_t st, int64_t* launches, const float* in, int rows, int K, const float* W,
                             const float* b, int N, int act, float* out) {
  GemmOperands g{in, W, nullptr, nullptr, K, N, rows, N, K};
  EpiBiasAct epi{b, out, N, act};
  return run_gemm<false, false, false, false, false>(st, launches, g, epi, nullptr, nullptr);
}

cudaError_t launch_dec2_loglik(cudaStream_t st, int64_t* launches, bool continuous, const float* h_d, int rows,
                               int H, const float* W2, const float* b2, const float* W6, const float* b6, int D,
                               const float* x, int x_div, int x_mod, float scale, float* da, float* dlv,
                               float* partial, int* n_col_tiles, bool fixed_tiles) {
  // fixed_tiles: the row sums must not depend on how many rows share the launch (the
  // importance-sampling estimator is bit-identical for any sharding of the test points)
  GemmOperands g{h_d, W2, nullptr, W6, H, D, rows, D, H};
  if (continuous) {
    EpiGaussian epi{b2, b6, x, D, x_div, x_mod, scale, da, dlv, D};
    return run_gemm<false, false, false, true, false>(st, launches, g, epi, partial, n_col_tiles, fixed_tiles);
  }
  EpiBernoulli epi{b2, x, D, x_div, x_mod, scale, da, D};
  return run_gemm<false, false, false, false, false>(st, launches, g, epi, partial, n_col_tiles, fixed_tiles);
}

cudaError_t launch_dec2_ae(cudaStream_t st, int64_t* launches, int mode, const float* h_d, int rows, int H,
                           const float* W2, const float* b2, int D, const float* x, float* da, float* partial,
                           int* n_col_tiles) {
  GemmOperands g{h_d, W2, nullptr, nullptr, H, D, rows, D, H};
  if (mode == 1) {
    EpiSquaredError epi{b2, x, D, da, D};
    return run_gemm<false, false, false, false, false>(st, launches, g, epi, partial, n_col_tiles);
  }
  EpiBernoulliClamp epi{b2, x, D, da, D};
  return run_gemm<false, false, false, false, false>(st, launches, g, epi, partial, n_col_tiles);
}

cudaError_t launch_dec2_recon(cudaStream_t st, int64_t* launches, bool continuous, const float* h_d, int rows,
                              int H, const float* W2, const float* b2, const float* W6, const float* b6, int D,
                              float* y, float* lv, float inv_n, int first) {
  GemmOperands g{h_d, W2, nullptr, W6, H, D, rows, D, H};
  EpiReconAccum epi{b2, b6, y, continuous ? lv : nullptr, D, inv_n, first};
  if (continuous) return run_gemm<false, false, false, true, false>(st, launches, g, epi, nullptr, nullptr);
  return run_gemm<false, false, false, false, false>(st, launches, g, epi, nullptr, nullptr);
}

cudaError_t launch_wgrad(cudaStream_t st, int64_t* launches, const float* in, int rows, int K, const float* d,
                         int N, float* gW, float* gb) {
  // C[K+1, N] = [in | 1]^T . d ; contraction over the rows
  GemmOperands g{in, d, nullptr, nullptr, K, N, K + 1, N, rows};
  EpiWgrad epi{gW, gb, K, N};
  return run_gemm<true, false, true, false, false>(st, launches, g, epi, nullptr, nullptr);
}

cudaError_t launch_dgrad_tanh(cudaStream_t st, int64_t* launches, const float* d, const float* W, const float* d2,
                              const float* W2, int rows, int N, int K, const float* h, float* out, int act) {
  // out[rows,K] = d[rows,N] . W[K,N]^T : B(k'=n, n'=k) = W[k*N + n] -> TB with ldb = N
  GemmOperands g{d, W, d2, W2, N, N, rows, K, N};
  EpiMulOneMinusSq epi{h, out, K, act};
  if (d2) return run_gemm<false, true, false, false, true>(st, launches, g, epi, nullptr, nullptr);
  return run_gemm<false, true, false, false, false>(st, launches, g, epi, nullptr, nullptr);
}

cudaError_t launch_dgrad(cudaStream_t st, int64_t* launches, const float* d, const float* W, int rows, int N, int K,
                         float* out) {
  GemmOperands g{d, W, nullptr, nullptr, N, N, rows, K, N};
  EpiStore epi{out, K};
  return run_gemm<false, true, false, false, false>(st, launches, g, epi, nullptr, nullptr);
}
