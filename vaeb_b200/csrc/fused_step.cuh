// Shared declarations of the fused (single-launch) AEVB step: fused_step.cu <-> api.cu.
//
// One cooperative kernel runs n whole updates (VAEB.py:408-415: forward, bound, backward, prior,
// Adagrad) back to back: one CTA per SM, eight grid barriers per update, every dense layer a tile
// job on fp32 FFMA pipes, Adagrad fused into the weight-gradient epilogues.  It serves the
// small-minibatch regime (M = 100) where a step is launch/latency bound, not roofline bound.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace fs {

constexpr int NW = 16;            // warps per CTA
constexpr int NT = NW * 32;       // threads per CTA
constexpr int KC = 16;            // contraction chunk staged per warp
constexpr int NSTAGE = 2;          // cp.async stages per warp (3 measured: 74.3 vs 74.5 us per update, not the limiter)
constexpr int WBUF = 960 * NSTAGE; // floats of shared memory per warp (operand stages, then the tile)
constexpr int N_PHASES = 8;       // grid barriers per update (+1 with sampled full-VB weights)
constexpr size_t SMEM_BYTES = (size_t)NW * WBUF * sizeof(float) + 64;

// tile jobs of one update, in phase order
enum Job {
  J_ENC1 = 0,   // h_e = tanh(x.W3+b3)                       VAEB.py:246
  J_ENC2,       // mu|ls = h_e.[W4|W5]+b, eps, z, KL/LA row  VAEB.py:248-249,41-47,343
  J_DEC1,       // h_d = tanh(z.W1+b1)                       VAEB.py:254
  J_DEC2,       // a(|lv) = h_d.W2(|W6)+b, log-lik, da(,dlv) VAEB.py:257-263,302-313
  J_DGRAD,      // da1 = (da.W2^T (+dlv.W6^T))*(1-h_d^2)     T.grad, VAEB.py:397
  J_WG2,        // W2,b2 += Adagrad([h_d|1]^T.da)            VAEB.py:397,426-444
  J_WG6,        // W6,b6 (Gaussian decoder)
  J_DZ,         // dz = da1.W1^T -> dmu, dls
  J_WG1,        // W1,b1 += Adagrad([z|1]^T.da1)
  J_DHE,        // da3 = (dmu.W4^T + dls.W5^T)*(1-h_e^2)
  J_WG45,       // W4,b4,W5,b5 += Adagrad([h_e|1]^T.[dmu|dls])
  J_WG3,        // W3,b3 += Adagrad([x|1]^T.da3)
  J_COUNT
};

// per-thread micro tile (rows, cols) of each job: CTA tile = 8*TMT rows x 4*TNT cols
__host__ __device__ constexpr int job_tmt(int j) {
  return (j == J_WG2 || j == J_WG6 || j == J_WG45 || j == J_WG3) ? 4 : 2;
}
__host__ __device__ constexpr int job_tnt(int j) {
  return (j == J_ENC2 || j == J_DZ || j == J_WG45) ? 2 : (j == J_DEC2 ? 10 : 6);
}

struct JobCfg {
  int tiles_m, tiles_n;   // tile grid
  int ks;                 // warps sharing one tile (split of the contraction index)
  int tpi;                // tiles per CTA item (ks * tpi <= NW)
  int n_items;            // CTA items
};

struct StepParams {
  int D, H, Z, M;                 // M = rows of the minibatch (L == 1)
  int cont, la;
  float w;                        // weight of the data term in the criterion (1, or 1/M: VAEBfullbayes)
  const float* kl_beta;           // device [n_steps]: weight of the latent term of each update (nullptr: 1)
  float lr, ada_eps, prior, p2;
  float* params[2];               // ping-pong flat parameter buffers (reference tensor order)
  float* ada;
  int64_t oW3, oW4, oW5, oW1, oW2, oW6, ob3, ob4, ob5, ob1, ob2, ob6;
  const float* x_base;            // resident data (batch_order != nullptr)
  const int* batch_order;         // device [n_steps]
  const float* x_direct;          // minibatch rows of a single step
  const float* eps_inj;           // injected eps [M,Z] or nullptr (Philox)
  uint64_t seed; uint32_t step0; int64_t row_offset;
  float *h_e, *mu, *ls, *eps, *z, *h_d, *da2, *dlv, *da1, *dmu, *dls, *da3;
  float* partial;                 // [M, tiles_n(J_DEC2)] log-likelihood row partials
  float* aux_part;                // [M, tiles_n(J_ENC2)] KL / LA row partials
  float* scalars; float Mg;       // scalars[s] = (bmult * bound of step s + thetaPrior) / Mg
  float bmult;
  // full variational Bayes with sampled weights (VAEB.py:127-129 live, getFVBL :349-367): phase 0 draws
  // theta = mu + |sigma| zeta for the whole flat buffer, every layer reads theta, the weight-gradient epilogues
  // update (mu, sigma) and their accumulators
  int fvb;
  float *vmu, *vsig, *ada_sig;    // `ada` holds the accumulators of mu
  float *theta, *zeta;            // this step's weights and their noise (flat, parameter layout)
  float* tprior_part;             // [gridDim.x] partial sums of thetaPrior (VAEB.py:359-363)
  int64_t total;                  // parameters in the flat buffer
  int n_steps, parity0;
  unsigned long long* bar; unsigned long long bar_base;
  long long* timing;              // nullptr or [n_steps*(N_PHASES+1)] globaltimer stamps of CTA 0
  JobCfg job[J_COUNT];
};

}  // namespace fs

struct vaeb_handle;
// true if the fused kernel can run this configuration (api.cu, next to step_path, which chooses the update kernel)
bool fused_step_supported(const vaeb_handle* h, int rows);
// n_steps updates in one launch.  Rows of step s: minibatch d_order[s] (of `rows` rows) of the resident data -- or of
// d_xrows when both are given (the staging ring of the streaming host-input updates) -- else d_xrows itself every step.
// d_kl: nullptr, or device [n_steps] with the KL weight beta_n of each step (vaeb_set_kl_weight).
int fused_step_launch(vaeb_handle* h, const int* d_order, const float* d_kl, const float* d_xrows, int rows, int n_steps,
                      const float* d_eps, int slot0, long long* d_timing);
