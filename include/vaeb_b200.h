/*
 * vaeb_b200.h -- C-ABI of the B200-native AEVB hot path (drop-in boundary).
 *
 * The reference (budzianowski/VAEB) has no native plugin ABI: its hot path is entered
 * through two Theano-compiled Python callables, `update(index)` and `validate(x)`
 * (VAEB.py:408-422), built by `VAEB.getGradient` (VAEB.py:370-424).  This header is the
 * C-ABI that sits directly beneath those callables.  Every entry point names the
 * reference interface it replaces (file:line under the reference root).  The reference-side
 * binding (a ctypes stub in VAEB.py) is shown in INTEGRATION.md; the shipped host mirror
 * is vaeb_b200/model.py.
 *
 * Conventions: plain pointers and sizes, no torch types.  All `float*` arguments are HOST
 * pointers unless named `d_*` / documented as device.  Matrices are row-major fp32.
 * Parameter tensors follow the reference list order
 *   [W3,W4,W5,W1,W2,(W6),b3,b4,b5,b1,b2,(b6)]            (VAEB.py:111-115)
 * with weights stored [in,out].  Every function returns 0 on success or a VAEB_E* code;
 * `vaeb_last_error()` returns a thread-local message.  A handle is bound to one GPU and is
 * not re-entrant.  There is no CPU fallback: without a CUDA device `vaeb_create` fails.
 */
#ifndef VAEB_B200_H_
#define VAEB_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VAEB_OK 0
#define VAEB_EINVAL 1   /* bad argument / unsupported configuration      */
#define VAEB_ECUDA 2    /* CUDA runtime error (message has the details)  */
#define VAEB_ENCCL 3    /* NCCL error or communicator not attached       */
#define VAEB_ESTATE 4   /* call sequence error (e.g. no data uploaded)   */

/* estimator -- which bound `getGradient` builds (VAEB.py:378-383) */
#define VAEB_EST_LB 0           /* getLB   VAEB.py:332-346 */
#define VAEB_EST_LA 1           /* getLA   VAEB.py:315-330 (--generic_estimator) */
#define VAEB_EST_FVB 2          /* getFVBL VAEB.py:349-367 exactly as shipped: weights NOT sampled */
#define VAEB_EST_FVB_SAMPLED 3  /* getFVBL with sample_variational_params (VAEB.py:127-129) live */

/* variant -- which script's objective/update scalars */
#define VAEB_VARIANT_VAEB 0       /* VAEB.py: sum objective, -0.5*sum(p^2) prior, Adagrad        */
#define VAEB_VARIANT_FULLBAYES 1  /* VAEBfullbayes.py:139-145,169-185: mean objective, no prior, */
                                  /* extra -lr*1e-6*p^2 in the update                            */

/* precision -- arithmetic of the dense layers */
#define VAEB_PREC_FP32 0   /* fp32 FFMA tiles (parity tier 1e-4)                          */
#define VAEB_PREC_BF16 1   /* tcgen05 bf16 operands, fp32 TMEM accumulation (1e-2 tier)   */
#define VAEB_PREC_BF16X3 2 /* tcgen05, operands as bf16 hi+lo, 3 MMAs per k-step: fp32-tier */

/* eps source */
#define VAEB_EPS_PHILOX 0    /* on-device Philox4x32-10 + Box-Muller                      */
#define VAEB_EPS_INJECTED 1  /* caller passes eps (the reference's host RNG draws)         */

typedef struct vaeb_handle vaeb_handle;

/* Mirrors the constructor VAEB.__init__ (VAEB.py:132-152). */
typedef struct vaeb_config {
  int32_t input_dim;      /* D  = x_train.shape[1]                      (VAEB.py:135) */
  int32_t hidden_units;   /* H                                          (VAEB.py:136) */
  int32_t latent_size;    /* Z                                          (VAEB.py:137) */
  int32_t batch_size;     /* M  rows per update()                       (VAEB.py:140) */
  int32_t L;              /* samples of z per datapoint                 (VAEB.py:143) */
  int32_t continuous;     /* 1 Gaussian decoder, 0 Bernoulli            (VAEB.py:138) */
  int32_t estimator;      /* VAEB_EST_*                                              */
  int32_t variant;        /* VAEB_VARIANT_*                                          */
  int32_t precision;      /* VAEB_PREC_*                                             */
  int32_t device;         /* CUDA ordinal                                            */
  float learning_rate;    /*                                            (VAEB.py:139) */
  float adagrad_eps;      /* 1e-6                                       (VAEB.py:144) */
  float prior_scale;      /* 1.0: -0.5*scale*sum(p^2)                   (VAEB.py:386) */
  float sigma_vb_init;    /* 1e-3 fullVBSigmaInit                       (VAEB.py:146) */
  uint64_t seed;          /* Philox key (reference: RandomStreams(seed=10), VAEB.py:158) */
  int32_t encoder_hidden_layers;   /* 0 or 1: one hidden layer, as VAEB.py:245-251 builds the encoder; 2..4: the deeper
                                      encoders of Report/replication/replic.tex:46-57 (extra H x H tanh layers between the first
                                      hidden layer and the heads; parameters W3_k, b3_k appended AFTER the reference's list;
                                      fp32 per-layer kernels, L^A / L^B estimators, one GPU) */
  int32_t reserved0;
} vaeb_config;

#define VAEB_OPT_ADAGRAD 0   /* getUpdates          VAEB.py:426-444 (the path the reference runs) */
#define VAEB_OPT_ADADELTA 1  /* getAdaDeltaUpdates  VAEB.py:449-469 (the alternative commented out at :404) */
#define VAEB_OPT_ADAM 2      /* Adam (Kingma & Ba 2015), selected with vaeb_set_adam */

#define VAEB_ACT_TANH 1      /* the reference's hidden layers (VAEB.py:246,254) */
#define VAEB_ACT_SIGMOID 2   /* alternatives compared in Report/replication/replic.tex:73-82 */
#define VAEB_ACT_RELU 3

const char* vaeb_last_error(void);
int vaeb_version(void);      /* 106: adds vaeb_step_counter, the getter of vaeb_set_step_counter (vaeb_config unchanged);
                                105: vaeb_profile_optimizer loses its variant argument (vaeb_config unchanged);
                                104: adds the KL weight (vaeb_set_kl_weight, vaeb_kl_step, vaeb_set_kl_step; vaeb_config
                                unchanged);
                                103: adds Adam (vaeb_set_adam, vaeb_adam_step, vaeb_set_adam_step; vaeb_config unchanged);
                                102: adds the encode, sample and validate_terms entry points (vaeb_config unchanged);
                                101: vaeb_config ends with encoder_hidden_layers, reserved0 (100: it ended with seed) */
/* sizeof(vaeb_config) as this library was compiled: a binding that declares the struct itself (ctypes, cgo) compares it
 * with its own size before the first vaeb_create -- a shorter struct would be read past its end. */
int vaeb_config_size(void);

/* VAEB.__init__ (VAEB.py:132-187): allocates the flat params / ADA / grads buffers
 * (VAEB.py:178-182) and workspaces on cfg->device.  Parameters start at zero: the host
 * mirror draws the reference initialisation (VAEB.py:50-115) and calls vaeb_set_params. */
int vaeb_create(const vaeb_config* cfg, vaeb_handle** out);
int vaeb_destroy(vaeb_handle* h);

/* Use an existing cudaStream_t for all work (NULL: the handle's own stream). */
int vaeb_set_stream(vaeb_handle* h, void* cuda_stream);
int vaeb_synchronize(vaeb_handle* h);

/* self.params / self.ADA / self.full_variational_params access (VAEB.py:111-125,178-182).
 * `which`: 0 params, 1 ADA accumulators (AdaDelta: g_ac; Adam: the first moment m), 2 gradients of the last step
 *          (criterion incl. prior), 3 variational means, 4 variational sigmas, 5 ADA of means, 6 ADA of sigmas,
 *          7 gradients w.r.t. means, 8 gradients w.r.t. sigmas  (3..8: FVB estimators only),
 *          9 AdaDelta's dx_ac or Adam's second moment v (whichever optimizer is selected).
 * `tensors[i]` points at host storage of tensor i in reference order. */
int vaeb_num_tensors(vaeb_handle* h, int32_t* n_tensors, int64_t* n_elements);
int vaeb_tensor_shape(vaeb_handle* h, int32_t i, int32_t* rows, int32_t* cols);
int vaeb_set_tensors(vaeb_handle* h, int32_t which, const float* const* tensors);
int vaeb_get_tensors(vaeb_handle* h, int32_t which, float* const* tensors);
/* Device address of a flat buffer (`which` as above) for zero-copy plumbing (e.g. wrapping as
 * a tensor for torch.distributed).  LIFETIME: the PARAMETER buffer (which = 0) is double-buffered by the
 * single-launch step kernels (they read theta_t from one copy while writing theta_{t+1} into the other), so its
 * address is valid only until the next vaeb_update* / vaeb_collect call on the handle: RE-QUERY it after every
 * update and never cache it across updates (tests/test_gpu_parity.py::test_device_buffer_tracks_updates).  The
 * accumulator and gradient buffers keep their addresses for the life of the handle. */
int vaeb_device_buffer(vaeb_handle* h, int32_t which, void** d_ptr, int64_t* n_elements);

/* ---- AE baselines (SURVEY.md 8f rank 2): ConstructAE of degenerate-vae/ae.py:41-117 and vanilla-ae/ae.py:45-104,
 * one tanh hidden layer per side as LearnFreyFace / LearnMNIST build them.  They share the handle's parameter
 * layout: W3 = Wenc, W4 = Wz, W1 = Wdec, W2 = Wout | Wmu, W6 = Wlogs2 (cfg.continuous = otype 'cont'); W5, b5 unused.
 * cfg.prior_scale = 1/s2 (mlp.ConstructNormalPrior, mlp.py:87-91), cfg.learning_rate = eta of infalg.AdaGrad. */
#define VAEB_AE_DEGENERATE 0  /* Z = Hz.Wz + bz, N(0,1) prior on Z, logpdf.bernoulli (+1e-7) | indep_normal */
#define VAEB_AE_VANILLA 1     /* Z = tanh(Hz.Wz + bz), squared error of sigmoid outputs                      */

/* `train(idx)` (ae.py:79-87): gathers rows idx[0..n) of the resident data (`givens = {X: Xtr[idx]}`), ascends
 * logjoint with AdaGrad (infalg.py:148-164) and returns loglik / n (degenerate) or se / n (vanilla), computed with
 * the pre-update parameters. */
int vaeb_ae_train(vaeb_handle* h, int32_t kind, const int32_t* idx, int32_t n, float* out);

/* `reconstruct(X)` (what = 0, ae.py:90-96), `encode(X)` (1, :99-105), `decode(Z)` (2, :108-114) on host arrays:
 * in[rows, D | Dz] -> out[rows, D | Dz | D]. */
int vaeb_ae_forward(vaeb_handle* h, int32_t kind, int32_t what, const float* in, int64_t rows, float* out);

/* Selects the update rule of the next vaeb_update* calls.  VAEB_OPT_ADADELTA restates
 * getAdaDeltaUpdates (VAEB.py:449-469): g_ac = rho g_ac + (1-rho) g^2; dx = sqrt(dx_ac + eps) g / sqrt(g_ac + eps);
 * p += dx; dx_ac = rho dx_ac + (1-rho) dx^2, with eps = adagrad_eps (VAEB.py:144) and rho = 0.95 (VAEB.py:145).
 * Both accumulators restart at zero.  Not available for the full-VB estimators. */
/* Activation of both hidden layers (encoder VAEB.py:246, decoder :254).  tanh (default) runs everywhere; sigmoid and ReLU
 * (Report/replication/replic.tex:73-82) run on the fp32 per-layer kernels (L^A / L^B estimators, one GPU). */
int vaeb_set_hidden_activation(vaeb_handle* h, int32_t act);
int vaeb_set_optimizer(vaeb_handle* h, int32_t optimizer, float rho);
/* Selects Adam (Kingma & Ba 2015) for the next vaeb_update* calls, in the ascent convention and with the weight prior of
 * getUpdates (VAEB.py:389-390), per element at Adam step t (t = 1 for the first update applied after this call):
 *   g = grad - prior_scale p   (no prior term for the VAEBfullbayes variant);  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
 *   p += alpha_t m / (sqrt(v) / s2_t + eps),  alpha_t = learning_rate / (1 - b1^t),  s2_t = sqrt(1 - b2^t)
 * (alpha_t, s2_t computed in double and rounded to float once per update): torch.optim.Adam(maximize=True).  m, v and
 * t restart at zero; vaeb_set_optimizer switches back to Adagrad or AdaDelta.  t advances once per applied update, when
 * the update is enqueued.  The single-launch step kernels apply Adagrad only: Adam updates of M <= 128 rows run the
 * per-layer kernels.  VAEB_EINVAL: beta1 or beta2 outside [0, 1), eps not positive and finite, or a full-VB estimator;
 * VAEB_ESTATE after vaeb_comm_p2p_export (select the optimizer on every rank before exporting). */
int vaeb_set_adam(vaeb_handle* h, float beta1, float beta2, float eps);
/* Adam step counter t (updates applied since vaeb_set_adam): with m and v (which = 1, 9) it is the optimizer state to
 * save and restore. */
int vaeb_adam_step(vaeb_handle* h, int64_t* t);
int vaeb_set_adam_step(vaeb_handle* h, int64_t t);

/* Weight of the latent term while training: KL warm-up (Bowman et al. 2016; Sonderby et al. 2016) and beta-VAE (Higgins
 * et al. 2017).  Sets the weight and resets the KL step counter t to 0.  The n-th update applied after this call
 * (n = 1, 2, ...) ascends
 *   loglik + beta_n aux,   beta_n = beta * min(1, n / warmup_updates)   (warmup_updates = 0: beta_n = beta)
 * where aux is the term vaeb_validate_terms returns: the analytic -KL for L^B, the Monte-Carlo log p(z) - log q(z|x)
 * for L^A.  beta_n is computed in double and rounded to float once per update.  t advances once per applied update,
 * when the update is enqueued, on every update path (vaeb_update_many advances it by n, each of its updates with its
 * own beta_n); vaeb_apply_update does not advance it.  Only the gradient is weighted: the values vaeb_update,
 * vaeb_update_host, vaeb_update_many and vaeb_collect return stay the unweighted bound SGVB/M.  vaeb_gradients uses
 * beta_{t+1}, the weight the next applied update would use, and does not advance t.  vaeb_validate, vaeb_validate_terms,
 * vaeb_is_logpx, vaeb_encode, vaeb_sample, vaeb_reconstruct and the AE entry points ignore the weight;
 * vaeb_profile_update restores t.  A handle that never calls this, or calls it with (1, 0), computes exactly what it
 * computed before the weight existed.  Any optimizer, variant, L, activation and encoder depth; data-parallel ranks
 * must agree on (beta, warmup_updates, t).  VAEB_EINVAL: beta negative, NaN or infinite, warmup_updates < 0, or a
 * full-VB estimator (its bound has its own weight-prior term). */
int vaeb_set_kl_weight(vaeb_handle* h, float beta, int64_t warmup_updates);
/* The KL step counter t (updates applied since vaeb_set_kl_weight): save and restore it so that a resumed run continues
 * its warm-up. */
int vaeb_kl_step(vaeb_handle* h, int64_t* t);
int vaeb_set_kl_step(vaeb_handle* h, int64_t t);

/* `x_train = th.shared(...)` (VAEB.py:184): copies x[N,D] to the device once. */
int vaeb_upload_data(vaeb_handle* h, const float* x, int64_t n_rows);

/* `update(index)` (VAEB.py:408-415): one AEVB step on rows [index*M,(index+1)*M) of the
 * resident data: forward, bound, backward, prior, Adagrad.  *elbo_out = SGVB/M computed
 * with the PRE-update parameters (VAEBfullbayes variant: the mean objective).  eps: NULL for
 * Philox, else host eps[L,M,Z] (the draws of `srng.normal`, VAEB.py:42).  Synchronous. */
int vaeb_update(vaeb_handle* h, int64_t index, const float* eps, float* elbo_out);

/* As vaeb_update, but the minibatch x[rows,D] comes from HOST memory in this call (the
 * end-to-end path: H2D copy of the inputs + D2H of the result inside the call). */
int vaeb_update_host(vaeb_handle* h, const float* x, int64_t rows, const float* eps, float* elbo_out);

/* Streaming form of vaeb_update_host for a host-side data loader feeding train_model's loop
 * (VAEB.py:577-579): enqueue one update on the minibatch x[rows,D] in PINNED host memory and return at
 * once.  The H2D copy runs on a copy stream into a ring of staging buffers and overlaps the previous
 * update's kernel; the update's bound is copied back D2H (4 bytes, asynchronously) as soon as its kernel
 * ends.  The caller must not modify x until vaeb_collect returns.  Philox eps only. */
int vaeb_update_host_async(vaeb_handle* h, const float* x, int64_t rows);

/* The same for BYTE-VALUED data sets: the reference's two data sets are 8-bit images stored as pixel / 256
 * (mnist.pkl.gz, freyfaces.pkl; loaded at VAEB.py:230-239, 544-555), so a host-side loader can keep them as bytes
 * and send a quarter of the PCIe traffic.  x[rows,D] uint8 in PINNED host memory; the minibatch the update sees is
 * (float)x * scale, one IEEE fp32 product per element computed on the device -- bit-identical to feeding
 * vaeb_update_host_async the host array np.float32(x) * np.float32(scale) (tests/test_gpu_async.py). */
int vaeb_update_host_async_u8(vaeb_handle* h, const uint8_t* x, int64_t rows, float scale);

/* Page-locked host memory for vaeb_update_host_async (plain cudaMallocHost / cudaFreeHost, so that a host
 * without torch can feed the streaming path).  vaeb_update_host_async returns VAEB_EINVAL for pageable memory:
 * such a copy would be staged synchronously by the driver and the overlap would be lost without any sign. */
int vaeb_host_alloc(int64_t bytes, void** out);
int vaeb_host_free(void* p);

/* Waits for every update enqueued by vaeb_update_host_async since the last collect and writes their
 * SGVB/M values, in submission order, to elbo_out[0..n) where n = *n_inout on return
 * (*n_inout on entry = capacity of elbo_out; VAEB_EINVAL if smaller than the number outstanding). */
int vaeb_collect(vaeb_handle* h, int32_t* n_inout, float* elbo_out);

/* The inner loop of train_model (VAEB.py:577-579) as ONE call: `n` updates in the order
 * `batch_order[0..n)` with no host synchronisation between them; elbo_out[n] receives each
 * step's SGVB/M.  Philox eps only. */
int vaeb_update_many(vaeb_handle* h, const int32_t* batch_order, int32_t n, float* elbo_out);

/* `validate(x)` (VAEB.py:418-422): SGVB of x[n,D] (a SUM over rows; the caller divides,
 * VAEB.py:582).  No parameter update.  per_row_out (NULL or float[n]) receives the
 * per-datapoint bound.  eps: NULL for Philox, else host eps[L,n,Z]. */
int vaeb_validate(vaeb_handle* h, const float* x, int64_t n, const float* eps,
                  float* sgvb_out, float* per_row_out);

/* Forward+backward only: fills the gradient buffer (`which`=2 / 7,8) without the Adagrad
 * update; the parity tests read per-tensor gradients through this.  x==NULL: rows of the
 * resident data starting at index*M. */
int vaeb_gradients(vaeb_handle* h, const float* x, int64_t rows, int64_t index, const float* eps,
                   const float* zeta, float* sgvb_out, float* per_row_out);
/* The Adagrad update alone (VAEB.py:426-444) on the current gradient buffer.  VAEB_EINVAL for Adam handles. */
int vaeb_apply_update(vaeb_handle* h);

/* Importance-sampled marginal likelihood (new capability named by the north star; the
 * integrand is getLA's, VAEB.py:319-327): log p^(x_i) = logsumexp_l(log w_il) - log L for
 * x[n,D].  eps: NULL (Philox keyed by (row_offset+i, l, j): results do not depend on how
 * rows are sharded over GPUs) or host eps[n,L,Z].  logw_out: NULL or float[n*L]. */
int vaeb_is_logpx(vaeb_handle* h, const float* x, int64_t n, int32_t L, const float* eps,
                  int64_t row_offset, float* logpx_out, float* logw_out);

/* `reconstruct(x, n_samples)` deterministic part (VAEB.py:267-292): decoder means averaged
 * over n_samples reparameterised z (n_samples<=0: decode mu).  y_out[n,D]; for the Gaussian
 * decoder lv_out[n,D] receives the averaged log-variance output (else may be NULL). */
int vaeb_reconstruct(vaeb_handle* h, const float* x, int64_t n, int32_t n_samples,
                     const float* eps, float* y_out, float* lv_out);

/* The decoder alone on caller-supplied latent points z[n,Z] (VAEB.py:253-265; the compiled `freyFace(z)` function
 * of freyFace.py:237-244 that the manifold renderer :350-369 calls): y_out[n,D] = sigmoid(tanh(z.W1+b1).W2+b2),
 * and for the Gaussian decoder lv_out[n,D] = tanh(z.W1+b1).W6+b6 (else may be NULL). */
int vaeb_decode(vaeb_handle* h, const float* z, int64_t n, float* y_out, float* lv_out);

/* The encoder alone (VAEB.py:245-251): the parameters of q(z|x) for host x[n,D].  mu_out[n,Z] is the mean and
 * logvar_out[n,Z] the second head, a log-VARIANCE although the reference names it log_sigma (VAEB.py:45,343).  Every
 * encoder depth and hidden activation; the fp32 per-layer kernels for every precision, in chunks of 32768 rows. */
int vaeb_encode(vaeb_handle* h, const float* x, int64_t n, float* mu_out, float* logvar_out);

/* Samples from the generative model (AEVB Fig. 5): for rows i < n, z_i ~ N(0, I), the decoder outputs of z_i and a draw
 * x_i ~ p(x|z_i).  z_out[n,Z]; mean_out[n,D] = y (sigmoid outputs, as vaeb_decode); lv_out[n,D] the Gaussian decoder's
 * log-variance output (the Bernoulli decoder: must be NULL); x_out[n,D].  Any output may be NULL.
 * Noise: Philox stream 5 (VAEB_STREAM_SAMPLE), key = cfg.seed, counter step = `step`, global row r = row_offset + i:
 *   z[i,j]   = normal   element r*Z + j of (stream 5, step, sample 0)
 *   x[i,d]:  u / eps  = element r*D + d of (stream 5, step, sample 1)
 *     Bernoulli: x = 1 if u < y else 0, u the uniform ((bits >> 8) + 0.5) * 2^-24 of that element's 32-bit output
 *     Gaussian:  x = y + exp(lv / 2) * eps, eps the normal of that element -- the likelihood's own variance exp(lv)
 *                (VAEB.py:302-313), not the exp(lv)^2 of the reference's reconstruct (VAEB.py:295-297)
 * "normal" / "uniform element e" as in vaeb_philox_normal: group e / 4, output e % 4, Box-Muller pairs (0,1), (2,3).
 * Results do not depend on how rows are split over calls or GPUs.  The step counter of the handle is not used or
 * advanced. */
int vaeb_sample(vaeb_handle* h, int64_t n, uint32_t step, int64_t row_offset, float* z_out, float* mean_out,
                float* lv_out, float* x_out);

/* The two terms of getLB / getLA (VAEB.py:332-346, :315-330) per row of x[n,D], with the inputs, noise and step counter
 * of vaeb_validate: loglik_out[n] = mean over the L samples of log p(x|z); aux_out[n] = the term the estimator adds to
 * it, the analytic -KL for L^B and the Monte-Carlo mean of log p(z) - log q(z|x) for L^A.  Their sum is vaeb_validate's
 * per-row bound, bit for bit when L is a power of two; otherwise the bound is formed with one fused multiply-add and
 * the float sum loglik + aux can differ from it in the last bit.  Full-VB handles return the same two terms under the
 * parameters they evaluate with; the weight-prior term of their bound (VAEB.py:359-363) is not per row and is in
 * neither. */
int vaeb_validate_terms(vaeb_handle* h, const float* x, int64_t n, const float* eps, float* loglik_out,
                        float* aux_out);

/* Dense tanh layers of the AE-side builders (degenerate-vae/mlp.py:66-74 ConstructMLP):
 * out = f(...f(x.W0+b0)...Wk+bk), f = tanh on every layer (act=1) or identity on the last
 * (act_last=0: logpdf.py:72-73 OutToReal; 2: sigmoid, logpdf.py:46-47 OutToProbs). */
int vaeb_mlp_forward(vaeb_handle* h, const float* x, int64_t n, int32_t n_layers,
                     const int32_t* dims /* n_layers+1 */, const float* const* W,
                     const float* const* b, int32_t act_last, float* out);

/* Philox eps exactly as the kernels draw it (for parity tests of the RNG itself):
 * out[n] = N(0,1) for flat elements first_elem.. of (stream, step, sample). */
int vaeb_philox_normal(vaeb_handle* h, int32_t stream, uint32_t step, uint32_t sample,
                       int64_t first_elem, int64_t n, float* out);
/* The Philox step counter: every update, validate and reconstruct draws its noise from (seed, stream, step) and advances
 * it by one.  vaeb_step_counter first launches any streaming updates still pending (as vaeb_get_tensors does). */
int vaeb_set_step_counter(vaeb_handle* h, uint32_t step);
int vaeb_step_counter(vaeb_handle* h, uint32_t* step);

/* ---- The training state of a handle ----------------------------------------------------------------------------
 * What a binding saves between two updates, and restores into a fresh handle, so that the next update -- and every
 * validate, reconstruct and update after it -- computes the same bits as a run that was never interrupted:
 *   buffers (vaeb_get_tensors / vaeb_set_tensors, by `which`):
 *     0             the parameters;
 *     1             Adagrad's accumulators, AdaDelta's g_ac or Adam's m;
 *     9             AdaDelta's dx_ac or Adam's v (those two optimizers only);
 *     3, 4, 5, 6    the variational means and sigmas and their Adagrad accumulators (full-VB estimators only);
 *     10, 11        VAEB_EST_FVB_SAMPLED only: theta and zeta of the next update.  The tensor-core step kernel draws
 *                   them for step t + 1 in the epilogues of step t (MUFU forms), so they are not re-derivable with the
 *                   same bits.  Reading them returns the draw for the current step counter (made then, with the
 *                   accurate forms of the other paths, if nothing has drawn it yet); writing them declares them the
 *                   draw for the current step counter;
 *   counters:
 *     vaeb_step_counter / vaeb_set_step_counter, vaeb_adam_step / vaeb_set_adam_step (Adam),
 *     vaeb_kl_step / vaeb_set_kl_step.
 * Restore in this order: vaeb_create with the same vaeb_config (seed included) and vaeb_upload_data; then the settings
 * that reset counters or accumulators -- vaeb_set_optimizer or vaeb_set_adam, vaeb_set_hidden_activation,
 * vaeb_set_kl_weight; then buffers 0-9; then the three counters; then buffers 10 and 11 (after the step counter, whose
 * draw they are).
 * Not state: the gradient buffers (2, 7, 8), which every update overwrites; buffers 10 and 11 of the other estimators;
 * the operand mirrors of the tensor-core paths and the parameter double buffer of the single-launch kernels, which
 * are rebuilt from the fp32 buffers with the bits the kernels themselves would have written.  Streaming updates
 * (vaeb_update_host_async) must be collected before the state is read.  Data-parallel ranks hold the same state: one
 * rank saves it, every rank restores it before attaching. */

/* Data-parallel training (new; SURVEY 8e): one handle per rank/GPU.  Rank 0 makes an id,
 * the host plumbing broadcasts the 128 bytes, every rank attaches.  After attaching,
 * vaeb_update* all-reduces (sum) the flat gradient and the bound over ranks before the
 * prior and the Adagrad update, so `batch_size` is the PER-RANK share of the global batch.
 * `nccl_library` = path of libnccl.so.2 to dlopen (the one torch bundles). */
int vaeb_comm_unique_id(const char* nccl_library, uint8_t id_out[128]);
int vaeb_comm_attach(vaeb_handle* h, const char* nccl_library, const uint8_t id[128],
                     int32_t rank, int32_t world_size);
int vaeb_comm_detach(vaeb_handle* h);
/* Data parallel over PEER MEMORY (NVLink / NVSwitch, ranks = processes of one box): after vaeb_comm_attach every rank
 * exports three CUDA IPC handles (its gradient staging buffer + flags, its parameters, its accumulators: Adam's m with v
 * right after it in the same allocation, so every rank must have selected the same optimizer before exporting;
 * vaeb_b200.distributed.attach_data_parallel compares the ranks' optimizers and refuses a mix), the
 * host plumbing all-gathers the 192 bytes per rank, every rank attaches all of them.  From then on the tail of a
 * large-batch tensor-core update (tc_tail.cu) IS the collective: each rank sums ITS slice of the flat gradient from
 * every rank's staging buffer with peer loads, applies prior + Adagrad (or Adam), and stores the new parameters (and
 * Adam's m and v) into every rank's buffers -- one launch, no NCCL kernel.  Other update paths keep using ncclAllReduce.  vaeb_comm_detach unmaps. */
int vaeb_comm_p2p_export(vaeb_handle* h, uint8_t handles_out[192]);
int vaeb_comm_p2p_attach(vaeb_handle* h, const uint8_t* all_handles, int32_t world_size);

/* Measurement aid for bench.py: runs the phases of one update on batch `index` one at a time,
 * each launched `iters` times back to back between two CUDA events on the handle's stream.
 * ms[i] = mean duration of phase i, flops[i]/bytes[i] = its ALGORITHMIC work per launch,
 * names + 48*i = its name.  The model state is restored afterwards. */
int vaeb_profile_update(vaeb_handle* h, int64_t index, int32_t iters, int32_t max_phases, int32_t* n_phases,
                        float* ms, double* flops, double* bytes, char* names);

/* Measurement aid for bench.py: the flat Adagrad pass of getUpdates (VAEB.py:426-444) over this handle's parameter,
 * accumulator and gradient buffers, `iters` launches back to back between two CUDA events on the handle's stream.
 * bytes_per_launch = 20 B x the number of parameters (SURVEY.md 8d).  A handle with a large hidden layer gives the
 * stream-sized buffer the HBM roofline needs; parameters and accumulators are restored afterwards. */
int vaeb_profile_optimizer(vaeb_handle* h, int32_t iters, float* ms_per_launch, double* bytes_per_launch);

/* Self-test of the tcgen05/TMA GEMM building block: C[M,N] = bf16(A[M,K]) . bf16(B[K,N]) with fp32
 * TMEM accumulation.  a_mn_major / b_mn_major choose the memory layout handed to TMA (0: the
 * contraction index is contiguous, 1: the M resp. N index is contiguous), block_n the UMMA N. */
int vaeb_tc_gemm_test(int32_t device, int32_t M, int32_t N, int32_t K, int32_t a_mn_major, int32_t b_mn_major,
                      int32_t block_n, const float* A, const float* B, float* C);

/* Counters for the bench: kernels launched by this handle since creation. */
int vaeb_launch_count(vaeb_handle* h, int64_t* n_launches);

/* Which kernel serves update() for a minibatch of `rows` rows with this handle's configuration: 2 = the tensor-core
 * single-launch step kernel (step_tc.cu: M <= 128, L = 1, one GPU), 1 = the fp32 FFMA single-launch kernel
 * (fused_step.cu), 0 = one launch per layer (kernels_*.cu / tc_layers.cu). */
int vaeb_step_kernel(vaeb_handle* h, int64_t rows, int32_t* which);

/* Diagnostic, host arithmetic only (no device needed): the (row tile, column tile) pairs that CTA `cta` of a `grid`-CTA
 * launch of the persistent tensor-core layer kernel works on, in order, for a [rows x N] layer cut into 128 x bn tiles
 * (full tiles round-robin first, then the sliver column tiles; tc_layers.cu `TileSeq`).  *n_out = number of pairs written;
 * VAEB_EINVAL if `cap` is too small. */
int vaeb_diag_tile_schedule(int32_t rows, int32_t N, int32_t bn, int32_t grid, int32_t cta, int32_t cap,
                            int32_t* tm_out, int32_t* tn_out, int32_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* VAEB_B200_H_ */
