// Host-side launchers of the fp32 kernels (implemented in kernels_gemm.cu / kernels_small.cu).
// Every launcher enqueues on `st`, bumps *launches by the kernels it started and returns a
// cudaError_t from cudaGetLastError().
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

// ---- dense layers (kernels_gemm.cu) ---------------------------------------------------
// out[rows,N] = act(in[rows,K] . W[K,N] + b)          VAEB.py:246,254 ; mlp.py:66-74
cudaError_t launch_dense_act(cudaStream_t st, int64_t* launches, const float* in, int rows, int K,
                             const float* W, const float* b, int N, int act, float* out);
// Decoder output layer fused with the log-likelihood (VAEB.py:257-263,302-313).
// partial[rows, *n_col_tiles] receives per-tile row sums.  da (and dlv) == nullptr: eval.
cudaError_t launch_dec2_loglik(cudaStream_t st, int64_t* launches, bool continuous, const float* h_d, int rows,
                               int H, const float* W2, const float* b2, const float* W6, const float* b6, int D,
                               const float* x, int x_div, int x_mod, float scale, float* da, float* dlv,
                               float* partial, int* n_col_tiles, bool fixed_tiles = false);
// AE baselines: decoder output layer fused with logpdf.bernoulli (mode 0, 1e-7 clamp; logpdf.py:85-86) or the
// squared error of vanilla-ae/ae.py:66 (mode 1, row sums = -se); da == nullptr: evaluation only
cudaError_t launch_dec2_ae(cudaStream_t st, int64_t* launches, int mode, const float* h_d, int rows, int H,
                           const float* W2, const float* b2, int D, const float* x, float* da, float* partial,
                           int* n_col_tiles);
// reconstruct accumulation (VAEB.py:282-292)
cudaError_t launch_dec2_recon(cudaStream_t st, int64_t* launches, bool continuous, const float* h_d, int rows,
                              int H, const float* W2, const float* b2, const float* W6, const float* b6, int D,
                              float* y, float* lv, float inv_n, int first);
// gW[K,N] = in[rows,K]^T . d[rows,N], gb[N] = colsum(d)   (weight + bias gradient in one GEMM)
cudaError_t launch_wgrad(cudaStream_t st, int64_t* launches, const float* in, int rows, int K, const float* d,
                         int N, float* gW, float* gb);
// out[rows,K] = (d[rows,N] . W[K,N]^T (+ d2 . W2^T)) * (1 - h^2)
cudaError_t launch_dgrad_tanh(cudaStream_t st, int64_t* launches, const float* d, const float* W,
                              const float* d2, const float* W2, int rows, int N, int K, const float* h, float* out,
                              int act = 1);   // act: the hidden activation whose derivative multiplies (VAEB_ACT_*)
// out[rows,K] = d[rows,N] . W[K,N]^T
cudaError_t launch_dgrad(cudaStream_t st, int64_t* launches, const float* d, const float* W, int rows, int N,
                         int K, float* out);

// ---- small fused kernels (kernels_small.cu) -----------------------------------------
struct EpsSource {
  const float* injected;   // device eps or nullptr
  uint64_t seed; uint32_t stream; uint32_t step; int64_t row_offset;
};
// mu, ls = h_e.W4+b4, h_e.W5+b5 (VAEB.py:248-249); if L>0 also eps, z = mu+exp(.5 ls) eps
// (VAEB.py:41-47) for l<L with rows laid out [L,rows,Z]; row_aux[rows] = KL row (VAEB.py:343)
// for LB or (1/L) sum_l (log p(z) - log q(z|x)) (VAEB.py:322-325) for LA.  row_aux == nullptr: no row terms (encoding
// only, with L = 0).
cudaError_t launch_enc2(cudaStream_t st, int64_t* launches, const float* h_e, int rows, int H, const float* W4,
                        const float* b4, const float* W5, const float* b5, int Z, int L, int la, EpsSource src,
                        float* mu, float* ls, float* eps, float* z, float* row_aux);
// importance-sampling rows r = i*L + l: eps, z and aux[r] = log p(z) - log q(z|x)
cudaError_t launch_is_sample(cudaStream_t st, int64_t* launches, const float* mu, const float* ls, int n, int L,
                             int Z, EpsSource src, float* z, float* aux);
// reconstruct: z[rows,Z] = mu + exp(.5 ls) * eps(sample)
cudaError_t launch_recon_sample(cudaStream_t st, int64_t* launches, const float* mu, const float* ls, int rows,
                                int Z, EpsSource src, int sample, int n_rows_total, float* z);
// encoder-side gradient assembly: dz[L,rows,Z] -> dmu, dls (SURVEY 8a backward formulas)
cudaError_t launch_dprep(cudaStream_t st, int64_t* launches, const float* dz, const float* z, const float* eps,
                         const float* mu, const float* ls, int rows, int Z, int L, int la, float w,
                         float* dmu, float* dls);
// per_row[m] = (1/L) sum_l sum_t partial[(l*rows+m), t] + row_aux[m]; base = sum_m per_row;
// scalar_out (nullable) = (mult*base + sum(tprior[0..n_tprior)))/div.  loglik / aux (both or neither): the two terms
// of per_row, loglik[m] = (1/L) sum_l sum_t partial (one rounding) and aux[m] = row_aux[m]
cudaError_t launch_finalize(cudaStream_t st, int64_t* launches, const float* partial, int n_tiles,
                            const float* row_aux, int rows, int L, float* per_row, float* base_out,
                            float mult, const float* tprior, int n_tprior, float div, float* scalar_out,
                            unsigned int* counter = nullptr,   // rows >= 2048 with a ticket counter and room for
                            float* block_part = nullptr,       // rows/256 block sums: one launch
                            float* loglik = nullptr, float* aux = nullptr);
// vaeb_sample: x[rows, D] drawn from p(x|z) given the decoder outputs (lv == nullptr: Bernoulli with means `mean`)
cudaError_t launch_sample_x(cudaStream_t st, int64_t* launches, const float* mean, const float* lv, int rows, int D,
                            uint64_t seed, uint32_t step, int64_t row_offset, float* x);
// logw[r] = sum_t partial[r,t] + aux[r];  logp[i] = logsumexp_l logw[i*L+l] - log L
cudaError_t launch_is_reduce(cudaStream_t st, int64_t* launches, const float* partial, int n_tiles,
                             const float* aux, int n, int L, float* logw, float* logp);
// out[m] = sum_q part[m, q]   (fixed order)
cudaError_t launch_row_partials_sum(cudaStream_t st, int64_t* launches, const float* part, int n_part, int rows,
                                    float* out);
cudaError_t launch_gather_rows(cudaStream_t st, int64_t* launches, const float* src, const int* idx, int n, int D,
                               float* out);
cudaError_t launch_axpy(cudaStream_t st, int64_t* launches, float* y, const float* x, float a, int64_t n);
// g -= prior*p  (VAEB.py:389-390); thread 0 also writes (mult*base)/div to scalar_out if non-null
cudaError_t launch_add_prior(cudaStream_t st, int64_t* launches, float* g, const float* p, int64_t n4, float prior,
                             const float* base, float mult, float div, float* scalar_out);
// Adagrad (VAEB.py:426-444; VAEBfullbayes.py:183-184 with p2 = lr*1e-6) over the flat buffer.
// If scalar_out != nullptr thread 0 also writes (mult*base + tprior)/div.
cudaError_t launch_adadelta(cudaStream_t st, int64_t* launches, float* p, float* gac, float* dxac, const float* g,
                            int64_t n4, float rho, float eps, float prior, const float* base, float mult, float div,
                            float* scalar_out);
// Adam (adam.cuh; alpha_t = lr / (1 - b1^t), s2_t = sqrt(1 - b2^t)) over the flat buffer.
// If scalar_out != nullptr thread 0 also writes (mult*base)/div.
cudaError_t launch_adam(cudaStream_t st, int64_t* launches, float* p, float* m, float* v, const float* g, int64_t n4,
                        float alpha_t, float s2_t, float b1, float b2, float eps, float prior, const float* base,
                        float mult, float div, float* scalar_out);
cudaError_t launch_adagrad(cudaStream_t st, int64_t* launches, float* p, float* acc, const float* g, int64_t n4,
                           float lr, float eps, float prior, float p2, const float* base, float mult, float div,
                           float* scalar_out);
#define VAEB_TP_BLOCKS 128
// thetaPrior partials (VAEB.py:359-363) over n real elements
cudaError_t launch_theta_prior(cudaStream_t st, int64_t* launches, const float* vmu, const float* vsig, int64_t n,
                               float* partials);
// theta = mu + |sigma| * zeta  (VAEB.py:127-129); zeta injected or Philox; zeta_out always written
cudaError_t launch_sample_theta(cudaStream_t st, int64_t* launches, const float* vmu, const float* vsig,
                                const float* zeta_in, uint64_t seed, uint32_t step, int64_t n, float* theta,
                                float* zeta_out);
// Adagrad on the variational parameters (VAEB.py:391-393,399,436-442)
cudaError_t launch_fvb_adagrad(cudaStream_t st, int64_t* launches, float* vmu, float* vsig, float* ada_mu,
                               float* ada_sig, const float* gtheta, const float* zeta, int sampled, int64_t n,
                               float lr, float eps, float prior, float* gmu, float* gsig, int apply);
cudaError_t launch_philox_fill(cudaStream_t st, int64_t* launches, uint64_t seed, uint32_t stream, uint32_t step,
                               uint32_t sample, int64_t first, int64_t n, float* out);

// ---- latent-layer kernels (kernels_latent.cu) ------------------------------------------
// w45t[2Z, H] = [W4^T ; W5^T]: head weights with the hidden index contiguous
cudaError_t launch_transpose_heads(cudaStream_t st, int64_t* launches, const float* W4, const float* W5, int H, int Z,
                                   float* w45t);
// enc2 + reparameterisation + row terms + decoder hidden layer.
// hd_hi/hd_lo: optional bf16 mirrors [L*rows, ld_mirror] of h_d for the tcgen05 GEMMs.
cudaError_t launch_latent_fwd(cudaStream_t st, int64_t* launches, const float* h_e, int rows, int H,
                              const float* w45t, const float* b4, const float* b5, const float* W1, const float* b1,
                              int Z, int L, int la, EpsSource src, float* mu, float* ls, float* eps, float* z,
                              float* row_aux, float* h_d, void* hd_hi, void* hd_lo, int ld_mirror, int act = 1);
// true when the 64-row large-batch kernels serve this shape
bool latent_large_batch(int rows, int H, int Z, int L);
// dz, dmu/dls, da3 and the bound (per row + deterministic total by the last block to finish).
// da3_hi/da3_lo: optional bf16 mirrors of da3, written only below latent_large_batch (the tensor-core path of the
// large-batch shapes computes da3 on tcgen05).  w_aux: weight of the latent term's gradient (the data weight times the
// KL weight of vaeb_set_kl_weight); the data term arrives in da1 already weighted.
cudaError_t launch_latent_bwd(cudaStream_t st, int64_t* launches, const float* da1, const float* W1,
                              const float* w45t, const float* h_e, const float* z, const float* eps, const float* mu,
                              const float* ls, int rows, int H, int Z, int L, int la, float w_aux, float* dmu, float* dls,
                              float* da3, void* da3_hi, void* da3_lo, int ld_mirror, const float* partial,
                              int n_tiles, const float* row_aux, float* per_row, unsigned int* counter,
                              float* base_out, float mult, const float* tprior, int n_tprior, float div,
                              float* scalar_out, int act = 1);
size_t small_wgrad_scratch_elems(int rows, int H, int Z);
// gW1,gb1,gW4,gb4,gW5,gb5 in one launch (two for large batches: row chunks + deterministic reduce)
cudaError_t launch_small_wgrad(cudaStream_t st, int64_t* launches, const float* z, const float* da1, int R,
                               const float* h_e, const float* dmu, const float* dls, int rows, int H, int Z,
                               float* gW1, float* gb1, float* gW4, float* gb4, float* gW5, float* gb5,
                               float* scratch);
// byte-valued host inputs of vaeb_update_host_async_u8: out = (float)in * scale
cudaError_t launch_expand_u8(cudaStream_t st, const uint8_t* in, float* out, int64_t n, float scale);
