// Host interface of the tcgen05 layer kernels (tc_layers.cu).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#define TC_LAYER_MAPS_BYTES 512   // four CUtensorMap (hi/lo of A and B)

struct TcBuffers {   // bf16 mirrors; *l == nullptr in plain-bf16 mode
  void *xh = nullptr, *xl = nullptr;       // data rows          [rows_data, ldx], ones column at D
  void *w3h = nullptr, *w3l = nullptr;     // W3                 [D, ldh]
  void *w2h = nullptr, *w2l = nullptr;     // W2                 [H, ldd]
  void *hdh = nullptr, *hdl = nullptr;     // h_d                [R, ldh], ones column at H
  void *da2h = nullptr, *da2l = nullptr;   // d bound / d a      [R, ldd]
  void *da3h = nullptr, *da3l = nullptr;   // d bound / d a3     [rows, ldh]
  // large-batch latent layers (rows >= 1024, L = 1): operands of the thin weight-gradient GEMMs
  void *heh = nullptr, *hel = nullptr;     // h_e                [rows, ldh], ones column at H
  void *d1h = nullptr, *d1l = nullptr;     // d bound / d a1     [R, ldh]
  void *zh = nullptr, *zl = nullptr;       // z                  [R, ldz], ones column at Z
  void *ddh = nullptr, *ddl = nullptr;     // [dmu | dls]        [rows, ldq]
  void *w45h = nullptr, *w45l = nullptr;   // [W4^T ; W5^T]      [2Z, ldh]
  void *w1h = nullptr, *w1l = nullptr;     // W1                 [Z, ldh]
  void *whh = nullptr, *whl = nullptr;     // heads, interleaved [H, ldq]: column 2j = W4[:,j], 2j+1 = W5[:,j]
  int ldz = 64, ldq = 64;                   // MN-major operands: row strides are multiples of 64 elements (3-D TMA boxes)
  int ldx = 0, ldh = 0, ldd = 0;
  float* wg_scratch = nullptr;             // split-K slices of the wide weight gradients
};

struct TcMaps {
  alignas(64) unsigned char enc1[TC_LAYER_MAPS_BYTES];
  alignas(64) unsigned char dec2[TC_LAYER_MAPS_BYTES];
  alignas(64) unsigned char dgrad[TC_LAYER_MAPS_BYTES];
  alignas(64) unsigned char wgrad2[TC_LAYER_MAPS_BYTES];
  alignas(64) unsigned char wgrad3[TC_LAYER_MAPS_BYTES];
  alignas(64) unsigned char wgrad1[TC_LAYER_MAPS_BYTES];    // gW1|gb1 = [z|1]^T . da1
  alignas(64) unsigned char wgrad45w[TC_LAYER_MAPS_BYTES];  // gW4|gW5 (+ bias row) = [h_e|1]^T . [dmu|dls], B boxes as wide
                                                            // as the other weight gradients'
  alignas(64) unsigned char dhe[TC_LAYER_MAPS_BYTES];       // da3 = ([dmu|dls] . [W4^T;W5^T]) * (1 - h_e^2)
  alignas(64) unsigned char dz[TC_LAYER_MAPS_BYTES];        // dz = da1 . W1^T (+ dmu, dls in the epilogue)
  alignas(64) unsigned char enc2[TC_LAYER_MAPS_BYTES];      // (mu, ls) = h_e . [W4|W5] (+ reparameterisation in the epilogue)
  alignas(64) unsigned char dec1[TC_LAYER_MAPS_BYTES];      // h_d = tanh(z . W1 + b1)
};

// programmatic dependent launch of the layer kernels (their prologues overlap the previous kernel's tail): for steps
// whose kernels are all about one wave
void tc_set_pdl(bool on);
// UMMA N of the activation layers (A K-major) for `rows` rows and outputs at least n_min wide: 256 selects the
// persistent kernel (large batches), else 128 / 64 with one tile per CTA
int tc_act_bn(int rows, int n_min);
// bn: UMMA N of the H-wide activation layers (enc1, dec1, both dgrads); bn_d (0: = bn): of dec2 (D wide)
// Dd (0: = D): width of the decoder output layer -- 2 D for the Gaussian head's interleaved columns [W2|W6]'
int tc_build_maps(TcMaps* m, const TcBuffers& b, int rows_data, int R, int rows, int D, int H, int bn, int Z, int bn_w,
                  int bn_d = 0, int Dd = 0);
// Gaussian decoder (VAEB.py:257-258, 306-307): a|lv = h_d.[W2|W6]' + b, log-density and both deltas in the epilogue
cudaError_t tc_dec2_gaussian(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                             const float* b2, const float* b6, const float* x, int x_div, int x_mod, float scale, void* da_hi,
                             void* da_lo, int ldda, float* partial, int* n_tiles, const void* xm_hi = nullptr,
                             const void* xm_lo = nullptr, int ldxm = 0, int xm_off = 0);

cudaError_t tc_split_matrix(cudaStream_t st, int64_t* launches, const float* src, int64_t rows, int cols, int ld_src,
                            void* hi, void* lo, int ld_dst, int ones_col);
cudaError_t tc_mirror_weights(cudaStream_t st, int64_t* launches, const float* w3, void* w3h, void* w3l, int D, int H,
                              int ldh, const float* w2, void* w2h, void* w2l, int ldd, const float* w6 = nullptr);
cudaError_t tc_enc1(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int D, int H,
                    int x_row_off, const float* b3, float* h_e, void* he_hi, void* he_lo, int ldm);
cudaError_t tc_dec2_bernoulli(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                              const float* b2, const float* x, int x_div, int x_mod, float scale, void* da_hi,
                              void* da_lo, int ldda, float* partial, int* n_tiles, const void* xm_hi = nullptr,
                              const void* xm_lo = nullptr, int ldxm = 0, int xm_off = 0);   // x == nullptr: x from its mirror
cudaError_t tc_dgrad_hd(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int D, int H,
                        const float* h_d, float* da1, void* d1_hi, void* d1_lo, int ldm, const void* h_hi = nullptr,
                        const void* h_lo = nullptr);   // h_d == nullptr: h is read from its mirror; da1 == nullptr: mirror only
// Deferred reduction of split-K slices: the weight-gradient GEMMs of a step append their job, one launch sums all
constexpr int TC_MAX_REDUCE_JOBS = 4;
struct TcReduceJob {
  const float* scratch; int splits; size_t stride; int n_w, n_b;
  float *gW, *gb, *gW2, *gb2; int kind, H, Z;       // kind 1: the interleaved heads slice -> (W4, b4, W5, b5)
};
struct TcReduceJobs { TcReduceJob job[TC_MAX_REDUCE_JOBS]; int n = 0; };
cudaError_t tc_wgrad_reduce_all(cudaStream_t st, int64_t* launches, const TcReduceJobs& jobs);
// all per-step weight mirrors / transposes of the large-batch path in one launch (W3, W2, [W4^T;W5^T] incl. its fp32
// copy w45t, the interleaved heads, W1)
cudaError_t tc_prepare_weights(cudaStream_t st, int64_t* launches, const float* W3, const float* W2, const float* W4,
                               const float* W5, const float* W1, const TcBuffers& b, float* w45t, int D, int H, int Z,
                               const float* W6 = nullptr);
// (mu, ls) = h_e.[W4|W5] + b fused with eps, z = mu + exp(.5 ls) eps, the KL / LA row terms (4 partials per row in
// aux_part) and the z mirror (VAEB.py:248-249, 41-47, 343, 322-325)
struct EpsSource;
cudaError_t tc_enc2_heads(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int rows, int H, int Z, int la,
                          const float* b4, const float* b5, const EpsSource& src, float* mu, float* ls, float* eps,
                          float* z, void* z_hi, void* z_lo, int ldz, float* aux_part, int* n_aux);
// h_d = tanh(z.W1 + b1) with its bf16 mirror (VAEB.py:254)
cudaError_t tc_dec1(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int Z, int H,
                    const float* b1, float* h_d, void* hd_hi, void* hd_lo, int ldm);
// dz = da1.W1^T fused with the encoder-side gradient assembly (SURVEY.md 8a: dmu, dls) and the [dmu|dls] mirror;
// w_aux weights the latent term's gradient
cudaError_t tc_dz_dprep(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int R, int H, int Z, int la, float w_aux,
                        const float* z, const float* eps, const float* mu, const float* ls, float* dmu, float* dls,
                        void* dd_hi, void* dd_lo, int ldq);
cudaError_t tc_dgrad_he(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int Z, int H,
                        const float* h_e, float* da3, void* da3_hi, void* da3_lo, int ldm, const void* h_hi = nullptr,
                        const void* h_lo = nullptr);
// scratch: device floats for the split-K slices of a weight gradient (tc_wgrad_scratch_elems), or nullptr
size_t tc_wgrad_scratch_elems(int D, int H);
cudaError_t tc_wgrad2(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                      float* gW2, float* gb2, float* scratch, float* gW6 = nullptr, float* gb6 = nullptr);
cudaError_t tc_wgrad3(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int D, int H,
                      int x_row_off, float* gW3, float* gb3, float* scratch);

// every weight-gradient GEMM of the step in ONE launch (W2, W1, [W4|W5], W3); the split-K slices stay in `scratch`
// (four regions of `region` floats) and their reductions are appended to `jobs`
cudaError_t tc_wgrad_all(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int rows, int D, int H,
                         int Z, int x_row_off, float* gW2, float* gb2, float* gW1, float* gb1, float* gW4, float* gb4,
                         float* gW5, float* gb5, float* gW3, float* gb3, float* scratch, size_t region, TcReduceJobs* jobs,
                         int n_sm, float* gW6 = nullptr, float* gb6 = nullptr);

// ---- the tail of a large-batch update as one launch (tc_tail.cu) --------------------------------------------------
// split-K slices -> gradient, bound, (N GPUs: reduce-scatter + all-gather over peer memory), prior + Adagrad, weight mirrors
constexpr int TC_MAX_PEERS = 8;
struct TcTailArgs {
  TcReduceJobs jobs;
  float* params; float* ada; float* grads; int64_t padded;
  float lr, eps, prior, p2;
  // bound: partial[rows, n_tiles] + (aux_part[rows, n_aux] or row_aux[rows])
  const float* partial; int n_tiles; const float* aux_part; int n_aux; const float* row_aux; int rows;
  float* per_row; float* block_part; float* base_out; float mult, div; float* scalar_out;
  // weight mirrors (w3h == nullptr: none)
  void *w3h, *w3l, *w2h, *w2l, *w45h, *w45l, *whh, *whl, *w1h, *w1l; float* w45t;
  int D, H, Z, ldh, ldd, ldq; int64_t oW3, oW4, oW5, oW1, oW2, oW6;      // oW6 < 0: Bernoulli decoder
  // grid barrier (monotonic counter; bar_base = arrivals before this launch)
  unsigned int* bar; unsigned int bar_base;
  // data parallel over peer memory (world == 1: unused)
  int world, rank; unsigned int epoch;
  float* gsum[TC_MAX_PEERS]; unsigned int* flags[TC_MAX_PEERS]; float* peer_params[TC_MAX_PEERS]; float* peer_ada[TC_MAX_PEERS];
  // Adam (adam.cuh): `ada` holds m and v holds the second moment; peer_ada / peer_v are every rank's m / v
  float alpha_t, s2_t, b1, b2, adam_eps;
  float* v; float* peer_v[TC_MAX_PEERS];
};
// `adam` selects the instantiation: Adam, or prior + Adagrad (lr, eps, prior, p2)
int tc_tail_grid(int n_sm, bool adam);
cudaError_t tc_tail_launch(cudaStream_t st, int64_t* launches, const TcTailArgs& a, int grid, bool adam);
