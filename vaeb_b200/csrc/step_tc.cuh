// Shared declarations of the tensor-core single-launch AEVB step (step_tc.cu <-> api.cu).
//
// The M = 100 update of the reference (VAEB.py:408-415 -- forward, bound, backward, prior, Adagrad; configs C2 and
// the Bernoulli runs of scripts/pg_7_graphs.sh) as ONE persistent kernel of thread-block clusters: every contraction
// runs on tcgen05 (fp16 hi+lo operands, three MMAs per k step, fp32 accumulation in TMEM: the fp32 parity tier), the
// split of a contraction over the four CTAs of a cluster is reduced through distributed shared memory, and EVERY
// operand lives in global memory (L2) as an fp16 hi/lo mirror in the UMMA shared-memory image (pre-swizzled, K-major):
// weights are rewritten by the Adagrad epilogues of the weight-gradient GEMMs, activations by the epilogue that
// produces them -- so staging an operand is one cp.async.bulk.  Six grid barriers per update (the FFMA kernel of
// fused_step.cu needs eight), no parameter double buffer.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace st2 {

constexpr int NT = 512;                 // threads per CTA (16 warps)
constexpr int CL = 4;                   // CTAs per cluster = ways a contraction is split
constexpr int MP = 128;                 // rows of a minibatch tile (UMMA M); minibatches of up to 128 rows
constexpr int N_PHASES = 6;             // grid barriers per update

// tile rows (UMMA N) of the mirrored weight operands
constexpr int TR_ENC1 = 16, TR_DEC2 = 32, TR_DGRAD = 16;

struct Params {
  int D, H, Z, M;
  int HP;                               // H rounded up to 64 (leading dimension of the hidden activations)
  int KD, KH;                           // 64-wide k chunks over D and over H
  int NH;                               // 2Z rounded up to 16: UMMA N of the latent heads
  int NZ;                               // Z + 1 rounded up to 16: UMMA N of dz and of the W1 weight gradient
  int la;
  // Gaussian decoder (VAEB.py:257-258): the output layer is [W2 | W6] seen as ONE layer of "virtual" columns -- a tile
  // of 32 pixels is 64 virtual columns, [32 columns of W2 | the same 32 pixels of W6] -- so the decoder GEMM, its
  // backward (K = the virtual columns) and the weight gradients keep the Bernoulli code with TR3 = 64 / KV = n_tiles3
  int cont;
  int TR3;                              // rows of a dec2 B tile (UMMA N of the output layer): 32, or 64 (Gaussian)
  int KV;                               // 64-wide k chunks over the virtual output columns (Bernoulli: KD)
  float w, lr, ada_eps, prior, p2;
  const float* kl_beta;                 // device [n_steps]: weight of the latent term of each update (nullptr: 1)
  float* P;                             // flat fp32 parameters (reference tensor order), updated in place
  float* ada;
  int64_t oW3, oW4, oW5, oW1, oW2, ob3, ob4, ob5, ob1, ob2, oW6, ob6;
  // weight mirrors: [n tile][k chunk][hi, lo][rows x 128 B], K-major SWIZZLE_128B
  uint8_t *m_enc1, *m_heads, *m_dec2, *m_dgrad, *m_dz;
  uint8_t* m_dec1;                      // [W1^T | b1]: tiles of 64 hidden units x one k chunk (k = latent index, k = Z: the bias)
  // activation mirrors.  *_km: [k chunk][hi, lo][128 batch rows x 128 B] (A operand of the next layer);
  // *_t: [feature tile][batch chunk (2)][hi, lo][tile rows x 128 B] (operands of the weight gradients)
  uint8_t *he_km, *he_t, *hd_t, *da2_km, *da2_t, *da1_km, *da1_t, *dd_t, *z_t;
  uint8_t* z_km;                        // [z | 1]: one k chunk (column Z reads as 1: the bias of the decoder hidden layer)
  uint8_t* dd_km;                       // [dmu | dls]: one k chunk (A operand of the dh_e GEMM inside the W3-gradient items)
  uint8_t* m_w45k;                      // [W4 | W5] with the hidden unit as the row: tiles of 32 hidden units x one k chunk
                                        // (k = column of [dmu|dls]); TWO copies selected by the parity of the step: the
                                        // W4/W5 update of a step writes the copy the NEXT step's dh_e GEMMs read
  int w45k_bytes;                       // bytes of one copy
  // the minibatch as operands: x_km [k chunk][hi, lo][128 x 128 B] of the NEXT step (A of enc1) and x_t
  // [pixel tile (+ the ones row at pixel D)][batch chunk (2)][hi, lo][128 x 128 B] of THIS step (A of the W3 gradient),
  // both written during P2 by the clusters that have no latent-head item
  uint8_t *x_km, *x_t;
  const float* x_base; const int* batch_order; const float* x_direct;
  const float* eps_inj;
  uint64_t seed; uint32_t step0; int64_t row_offset;
  int w45_par0;                         // the copy of the k-major [W4|W5] mirror that holds theta at the first step
  float *he, *hd, *mu, *ls, *eps, *z;   // fp32 copies the epilogues read: [MP, HP], [MP, HP], [MP, Z] x 4
  float *partial, *aux;                 // [MP, tiles of dec2] log-likelihood row partials; [MP] KL / LA row terms
  int n_tiles3;                         // n tiles of dec2 (partial's leading dimension)
  float* scalars; float Mg; float bmult;
  int n_steps;
  // Gaussian decoder only: its deltas scale with exp(-log variance) and can leave the range of the fp16 operand
  // pairs.  A step whose da2 / da1 exceed DLIMIT writes its index here (-1 otherwise) and the launch stops BEFORE
  // that step's first parameter update; the host finishes the remaining steps with the fp32 FFMA kernel.
  int* status;
  // Full VB as the reference runs it (getFVBL, VAEB.py:349-367: the weights are never sampled): an update is the
  // forward phases P1-P3 on the frozen MAP parameters, thetaPrior, and the prior-only Adagrad step on (mu, sigma).
  // fvb = 2: the sampled-weights estimator (VAEB.py:127-129 live inside getFVBL).  P is then the buffer of the sampled
  // theta = mu + |sigma| zeta: the Adagrad epilogue of every weight-gradient tile updates (mu, sigma) with their own
  // accumulators, DRAWS the next step's zeta there (Philox, keyed by the step and the flat parameter index), and
  // writes theta' = mu' + |sigma'| zeta' both as fp32 (biases, rebuilds) and into the fp16 operand mirrors -- the
  // weights are sampled where the next step's GEMM operands are produced; no pass over the parameters.
  int fvb;
  float *vmu, *vsig, *ada_mu, *ada_sig; int64_t total;
  float* zeta;                          // the draws of the current step (written by the previous step's epilogues)
  float* tprior_part;                   // [2][gridDim.x] per-CTA partial sums of thetaPrior (step parity)
  unsigned long long* bar; unsigned long long bar_base;
  long long* timing;                    // nullptr or [n_steps * (N_PHASES + 1)] globaltimer stamps of CTA 0
};

}  // namespace st2

struct vaeb_handle;
struct StepTcState {
  bool ready = false, unavailable = false;
  int n_cta = 0;
  int rows_init = -1;                   // minibatch rows the activation mirrors were cleared for
  unsigned long long* bar = nullptr; unsigned long long bar_count = 0;
  uint8_t *m_enc1 = nullptr, *m_heads = nullptr, *m_dec2 = nullptr, *m_dgrad = nullptr, *m_dz = nullptr, *m_dec1 = nullptr,
          *m_w45k = nullptr;
  uint8_t* act = nullptr; size_t act_bytes = 0;      // one allocation for every activation mirror
  size_t o_he_km = 0, o_he_t = 0, o_hd_t = 0, o_da2_km = 0, o_da2_t = 0, o_da1_km = 0, o_da1_t = 0, o_dd_t = 0, o_z_t = 0, o_z_km = 0,
         o_dd_km = 0, o_x_km = 0, o_x_t = 0;
  bool mirrors_valid = false;
  float *he = nullptr, *hd = nullptr, *mu = nullptr, *ls = nullptr, *eps = nullptr, *z = nullptr,
        *partial = nullptr, *aux = nullptr;
  long long* d_timing = nullptr; int timing_cap = 0;
  int* d_status = nullptr;
  float* tprior_part = nullptr;
  long long theta_step = -1;            // sampled full VB: the step the theta / zeta buffers were drawn for (-1: stale)
  // which of the two copies of the k-major [W4|W5] mirror holds the current parameters: a step reads one and its
  // epilogue writes the next step's into the other.  Kept here rather than taken from the step counter's parity,
  // which validate / reconstruct advance without touching the mirrors.
  int w45_par = 0;
};

// n_steps updates in one launch (same contract as fused_step_launch)
int step_tc_launch(vaeb_handle* h, const int* d_order, const float* d_kl, const float* d_xrows, int rows, int n_steps,
                   const float* d_eps, int slot0, long long* d_timing);
void step_tc_free(StepTcState& s);
