// Handle, flat-buffer layout and error plumbing shared by the translation units.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/vaeb_b200.h"
#include "tc_layers.h"
#include "fused_step.cuh"
#include "step_tc.cuh"

void vaeb_set_error(const std::string& msg);

#define VAEB_CUDA(expr)                                                                      \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      vaeb_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                     ":" + std::to_string(__LINE__) + ")");                                  \
      return VAEB_ECUDA;                                                                     \
    }                                                                                        \
  } while (0)

#define VAEB_TRY(expr)            \
  do {                            \
    int _r = (expr);              \
    if (_r != VAEB_OK) return _r; \
  } while (0)

#define VAEB_REQUIRE(cond, msg)                  \
  do {                                           \
    if (!(cond)) {                               \
      vaeb_set_error(std::string("invalid argument: ") + (msg)); \
      return VAEB_EINVAL;                        \
    }                                            \
  } while (0)

// Tensor indices in the reference's list order (VAEB.py:111-115).
struct Layout {
  int n = 0;                 // 10 (Bernoulli) or 12 (Gaussian), + 2 per extra encoder hidden layer
  int rows[20], cols[20];
  int64_t off[20];           // element offset inside the flat buffer (tightly packed)
  int64_t total = 0;         // P
  int64_t padded = 0;        // P rounded up to a multiple of 4 (float4 kernels)
  int iW3, iW4, iW5, iW1, iW2, iW6, ib3, ib4, ib5, ib1, ib2, ib6;
  int depth = 1;             // encoder hidden layers; layer k = 2..depth: iW3x[k - 2] (H x H), ib3x[k - 2]
  int iW3x[3] = {-1, -1, -1}, ib3x[3] = {-1, -1, -1};
};

// NCCL entry points resolved with dlopen (no link-time dependency; the host passes the path
// of the libnccl.so.2 that torch bundles).
struct NcclId { char internal[128]; };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId /* ncclUniqueId by value: 128 bytes */, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};

struct Workspace {
  int64_t cap_enc = 0, cap_dec = 0;   // rows the buffers hold (encoder rows, decoder rows)
  bool with_grads = false;
  float *h_e = nullptr, *mu = nullptr, *ls = nullptr, *eps = nullptr, *z = nullptr, *h_d = nullptr;
  float *da2 = nullptr, *dlv = nullptr, *da1 = nullptr, *dz = nullptr, *dmu = nullptr, *dls = nullptr, *da3 = nullptr;
  float *partial = nullptr, *row_aux = nullptr, *per_row = nullptr, *dec_aux = nullptr, *logw = nullptr;
  float* wg_scratch = nullptr;        // row-chunk partials of the thin weight gradients (large batches)
  // deeper encoders: activations of hidden layers 1 .. depth-1 (h_e holds the LAST one, which the heads read) and a second
  // buffer for the gradient walking back through them
  float* h_x[3] = {nullptr, nullptr, nullptr}; float* da3b = nullptr;
};

// Tensor-core path state: bf16 (hi/lo) mirrors and their TMA descriptors.
struct TcState {
  bool active = false;
  int ns = 1;                              // 1: bf16, 2: bf16 hi+lo (three MMAs per k-step)
  TcBuffers data;                          // mirrors with the resident dataset as x
  void *xsh = nullptr, *xsl = nullptr;     // mirror of a staged (host-supplied) batch
  int64_t cap_stage = 0, cap_R = 0, cap_rows = 0;
  TcMaps maps;
  int64_t key_rows = -1, key_R = -1, key_data = -1; int key_bn = 0; const void* key_x = nullptr;
  int n_sm = 0;
  // the fused tail of an update (tc_tail.cu)
  bool weights_ready = false;              // the weight mirrors hold the CURRENT parameters (written by the tail)
  unsigned int* tail_bar = nullptr; unsigned int tail_bar_count = 0;
  // data parallel over peer memory: this rank's comm buffer [padded + 4 floats | 2 * world flags], everybody's mappings
  float* p2p_buf = nullptr; bool p2p_ready = false; unsigned int p2p_epoch = 0;
  float* p2p_gsum[8] = {}; unsigned int* p2p_flags[8] = {}; float* p2p_params[8] = {}; float* p2p_ada[8] = {};
  void* p2p_opened[24] = {}; int p2p_n_opened = 0;
};

// State of the fused single-launch step (fused_step.cu).
struct FusedState {
  bool ready = false;
  int n_sm = 0;
  unsigned long long* bar = nullptr;       // grid-barrier counter (monotonic)
  unsigned long long bar_count = 0;        // arrivals so far = the next launch's base
  float* params_alt = nullptr;             // the other half of the parameter double buffer
  float* partial = nullptr; float* aux_part = nullptr;
  float* tprior_part = nullptr;            // per-CTA thetaPrior partial sums (sampled full VB)
  long long* d_timing = nullptr; int timing_cap = 0;
  int rows = -1;
  fs::JobCfg job[fs::J_COUNT];
};

// State of the tensor-core importance-sampling estimator (is_tc.cu).
struct IsTcState {
  void* w2t = nullptr;                               // W2^T [D, KP] bf16
  void* w1t = nullptr;                               // [W1^T | b1] [512, 64] bf16
  float* bias26 = nullptr;                           // Gaussian decoder: b2 / b6 interleaved like the output columns
  alignas(64) unsigned char map_w1[128];             // CUtensorMap over w1t, boxes of 64 rows (one pass)
  alignas(64) unsigned char map_full[128];           // CUtensorMap over w2t, boxes of `tail_cols` rows (one output chunk)
  int n_sm = 0, n_chunks = 0, tail_cols = 0;         // tail_cols = chunk width NC (multiple of 16)
  void* partial = nullptr; int64_t partial_cap = 0;  // per-tile (max, sum exp)
  // pipelined host input of vaeb_is_logpx: the next chunk of points is copied on `copy` while this one is sampled
  cudaStream_t copy = nullptr;
  cudaEvent_t copied[2] = {}, consumed[2] = {};
  float* xbuf[2] = {nullptr, nullptr}; int64_t xbuf_cap = 0;
};

struct vaeb_handle {
  vaeb_config cfg;
  TcState tc;
  int D, H, Z, M, L;
  bool cont;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  Layout lay;
  // flat buffers: [padded + 4]; slot [padded] of d_grads carries the bound for the all-reduce
  float *d_params = nullptr, *d_ada = nullptr, *d_grads = nullptr;
  float *d_vmu = nullptr, *d_vsig = nullptr, *d_ada_mu = nullptr, *d_ada_sig = nullptr;
  float *d_gmu = nullptr, *d_gsig = nullptr, *d_theta = nullptr, *d_zeta = nullptr;
  float* d_tprior = nullptr;          // [TP_BLOCKS] partial sums of thetaPrior
  unsigned int* d_counter = nullptr;  // last-block-done counter of latent_bwd
  float* d_w45t = nullptr;            // [2Z, H] transposed latent-head weights of the current theta
  float* d_x = nullptr; int64_t n_data = 0;
  Workspace ws;
  int optimizer = 0; float rho = 0.95f; float* d_ada2 = nullptr;   // AdaDelta: d_ada = g_ac, d_ada2 = dx_ac
  // Adam: d_ada = m and d_adam_v = v, in ONE allocation (v right after m, so that the accumulator's IPC handle maps both);
  // adam_t = updates applied since Adam was selected; alpha_t / s2_t of the update being enqueued
  float adam_b1 = 0.9f, adam_b2 = 0.999f, adam_eps = 1e-8f; float* d_adam_v = nullptr; int64_t adam_t = 0;
  float adam_alpha_t = 0.f, adam_s2_t = 0.f;
  // KL weight (vaeb_set_kl_weight): the n-th update applied since the call, n = kl_t + 1, ascends
  // loglik + beta_n aux with beta_n = kl_beta * min(1, n / kl_warmup); d_kl holds beta_n of each update of one
  // single-launch call (grown as d_order)
  float kl_beta = 1.f; int64_t kl_warmup = 0, kl_t = 0;
  float* d_kl = nullptr; int kl_cap = 0;
  float* d_stage = nullptr; int64_t stage_cap = 0;       // device staging for host inputs
  // streaming host-input updates (vaeb_update_host_async): copy stream + ring of staging buffers
  static constexpr int ASYNC_BUFS = 4;
  cudaStream_t copy_stream = nullptr;
  float* a_stage[ASYNC_BUFS] = {nullptr, nullptr, nullptr, nullptr}; int64_t a_stage_cap = 0;
  uint8_t* a_stage_u8[ASYNC_BUFS] = {nullptr, nullptr, nullptr, nullptr}; int64_t a_stage_u8_cap = 0;   // byte-valued inputs
  cudaEvent_t a_copied[ASYNC_BUFS] = {}, a_consumed[ASYNC_BUFS] = {};
  bool a_used[ASYNC_BUFS] = {false, false, false, false};
  static constexpr int ASYNC_GROUP = 4;                   // updates per launch of the fused kernel
  int a_pending = 0, a_group = 0; int64_t a_rows = 0;     // minibatches copied but not yet launched; current group buffer
  int* d_iota = nullptr;                                  // {0, 1, .., ASYNC_GROUP-1}: slot order inside a group buffer
  int a_outstanding = 0;
  float* h_async = nullptr; int h_async_cap = 0;          // pinned host landing zone of the bounds
  float* d_stage2 = nullptr; int64_t stage2_cap = 0;     // eps staging
  float* d_out = nullptr; int64_t out_cap = 0;           // device staging for outputs
  float* d_scalars = nullptr; float* h_scalars = nullptr; int scalars_cap = 0;
  int* d_order = nullptr; int order_cap = 0;             // minibatch indices of a single-launch update (device)
  uint32_t step = 0;
  int64_t launches = 0;
  bool grads_have_prior = false;
  FusedState fused;
  IsTcState istc;
  StepTcState steptc;                 // tensor-core single-launch step (step_tc.cu)
  bool env_no_step_tc = false;        // VAEB_B200_STEP_TC=0: the FFMA kernel of fused_step.cu serves M <= 128 too
  bool env_no_fused = false;          // VAEB_B200_FUSED=0: the FFMA single-launch kernel is off
  int hidden_act = 1;                 // VAEB_ACT_*: activation of both hidden layers (tanh in the reference's VAEB.py:246,254)
  // data parallel
  NcclApi nccl; void* comm = nullptr; int rank = 0, world = 1;
};

// The parameters changed behind the cached bf16 weight mirrors: those of the tensor-core step kernel (step_tc.cu) and
// those of the large-batch path (written by tc_prepare_weights or the tail kernel).
// the parameters may have changed: the operand mirrors and the sampled full-VB theta of the step kernel are stale
inline void invalidate_weight_mirrors(vaeb_handle* h) {
  h->steptc.mirrors_valid = false;
  h->steptc.theta_step = -1;
  h->tc.weights_ready = false;
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
