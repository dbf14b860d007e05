// C-ABI of include/vaeb_b200.h: handle management and the orchestration of one AEVB step.
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "launchers.h"
#include "philox.cuh"

bool is_tc_supported(const vaeb_handle* h);   // is_tc.cu
int is_tc_run(vaeb_handle* h, const float* d_x, const float* d_mu, const float* d_ls, int n, int L, const float* d_eps,
              int64_t row_offset, float* d_logp, float* d_logw);

static thread_local std::string g_last_error;
void vaeb_set_error(const std::string& msg) { g_last_error = msg; }

#define VAEB_LAUNCH(expr)                                                     \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess) {                                                  \
      vaeb_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));     \
      return VAEB_ECUDA;                                                      \
    }                                                                         \
  } while (0)

// Per-phase profiling (vaeb_profile_update): every phase launch of one step is repeated `iters`
// times between two CUDA events on the handle's stream.
struct PhaseProf {
  int iters = 1;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  std::vector<std::string> names;
  std::vector<float> ms;
  std::vector<double> flops, bytes;
};
static thread_local PhaseProf* g_prof = nullptr;

#define PH(NAME, FLOPS, BYTES, EXPR)                                                   \
  do {                                                                                 \
    if (g_prof) {                                                                      \
      VAEB_CUDA(cudaEventRecord(g_prof->e0, h->stream));                               \
      for (int _i = 0; _i < g_prof->iters; ++_i) VAEB_LAUNCH(EXPR);                    \
      VAEB_CUDA(cudaEventRecord(g_prof->e1, h->stream));                               \
      VAEB_CUDA(cudaEventSynchronize(g_prof->e1));                                     \
      float _ms = 0.f;                                                                 \
      VAEB_CUDA(cudaEventElapsedTime(&_ms, g_prof->e0, g_prof->e1));                   \
      g_prof->names.push_back(NAME);                                                   \
      g_prof->ms.push_back(_ms / (float)g_prof->iters);                                \
      g_prof->flops.push_back((double)(FLOPS));                                        \
      g_prof->bytes.push_back((double)(BYTES));                                        \
    } else {                                                                           \
      VAEB_LAUNCH(EXPR);                                                               \
    }                                                                                  \
  } while (0)

namespace {

void build_layout(Layout& l, int D, int H, int Z, bool cont, int depth = 1) {
  int i = 0;
  auto add = [&](int& idx, int r, int c) { idx = i; l.rows[i] = r; l.cols[i] = c; ++i; };
  l.iW6 = l.ib6 = -1;
  add(l.iW3, D, H); add(l.iW4, H, Z); add(l.iW5, H, Z); add(l.iW1, Z, H); add(l.iW2, H, D);
  if (cont) add(l.iW6, H, D);
  add(l.ib3, 1, H); add(l.ib4, 1, Z); add(l.ib5, 1, Z); add(l.ib1, 1, H); add(l.ib2, 1, D);
  if (cont) add(l.ib6, 1, D);
  // deeper encoders (replic.tex:46-57): the extra layers come AFTER the reference's list, weights first
  l.depth = depth < 1 ? 1 : depth;
  for (int k = 2; k <= l.depth; ++k) add(l.iW3x[k - 2], H, H);
  for (int k = 2; k <= l.depth; ++k) add(l.ib3x[k - 2], 1, H);
  l.n = i;
  int64_t off = 0;
  for (int t = 0; t < l.n; ++t) { l.off[t] = off; off += (int64_t)l.rows[t] * l.cols[t]; }
  l.total = off;
  l.padded = (off + 3) / 4 * 4;
}

bool is_fvb(const vaeb_handle* h) {
  return h->cfg.estimator == VAEB_EST_FVB || h->cfg.estimator == VAEB_EST_FVB_SAMPLED;
}

int alloc_flat(float** p, int64_t n, float fill = 0.f) {
  VAEB_CUDA(cudaMalloc((void**)p, (size_t)n * sizeof(float)));
  if (fill == 0.f) {
    VAEB_CUDA(cudaMemset(*p, 0, (size_t)n * sizeof(float)));
  } else {
    std::vector<float> tmp((size_t)n, fill);
    VAEB_CUDA(cudaMemcpy(*p, tmp.data(), (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
  }
  return VAEB_OK;
}

int grow(float** p, int64_t* cap, int64_t need) {
  if (need <= *cap) return VAEB_OK;
  if (*p) VAEB_CUDA(cudaFree(*p));
  *p = nullptr;
  VAEB_CUDA(cudaMalloc((void**)p, (size_t)need * sizeof(float)));
  *cap = need;
  return VAEB_OK;
}

void free_ws(Workspace& w) {
  float** all[] = {&w.h_e, &w.mu, &w.ls, &w.eps, &w.z, &w.h_d, &w.da2, &w.dlv, &w.da1, &w.dz, &w.dmu, &w.dls,
                   &w.da3, &w.partial, &w.row_aux, &w.per_row, &w.dec_aux, &w.logw, &w.wg_scratch,
                   &w.h_x[0], &w.h_x[1], &w.h_x[2], &w.da3b};
  for (float** p : all) { if (*p) cudaFree(*p); *p = nullptr; }
  w.cap_enc = w.cap_dec = 0;
  w.with_grads = false;
}

int ensure_ws(vaeb_handle* h, int64_t enc, int64_t dec, bool grads) {
  Workspace& w = h->ws;
  if (enc <= w.cap_enc && dec <= w.cap_dec && (!grads || w.with_grads)) return VAEB_OK;
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  enc = std::max(enc, w.cap_enc);
  dec = std::max(dec, w.cap_dec);
  grads = grads || w.with_grads;
  free_ws(w);
  const int D = h->D, H = h->H, Z = h->Z;
  const int Dd = h->cont && h->tc.active ? 2 * D : D;      // tensor-core Gaussian head: 2 D interleaved columns
  const int64_t T = std::max<int64_t>((D + 31) / 32, 4 * ((Dd + 63) / 64));   // row-sum partials per row
  auto A = [&](float** p, int64_t n) -> int {
    VAEB_CUDA(cudaMalloc((void**)p, (size_t)std::max<int64_t>(n, 1) * sizeof(float)));
    return VAEB_OK;
  };
  VAEB_TRY(A(&w.h_e, enc * H)); VAEB_TRY(A(&w.mu, enc * Z)); VAEB_TRY(A(&w.ls, enc * Z));
  for (int k = 0; k + 1 < h->lay.depth; ++k) VAEB_TRY(A(&w.h_x[k], enc * H));
  VAEB_TRY(A(&w.row_aux, enc)); VAEB_TRY(A(&w.per_row, enc));
  VAEB_TRY(A(&w.eps, dec * Z)); VAEB_TRY(A(&w.z, dec * Z)); VAEB_TRY(A(&w.h_d, dec * H));
  VAEB_TRY(A(&w.partial, dec * T)); VAEB_TRY(A(&w.dec_aux, dec)); VAEB_TRY(A(&w.logw, dec));
  if (grads) {
    VAEB_TRY(A(&w.da2, dec * D));
    if (h->cont) VAEB_TRY(A(&w.dlv, dec * D));
    VAEB_TRY(A(&w.da1, dec * H)); VAEB_TRY(A(&w.dz, dec * Z));
    VAEB_TRY(A(&w.dmu, enc * Z)); VAEB_TRY(A(&w.dls, enc * Z)); VAEB_TRY(A(&w.da3, enc * H));
    if (h->lay.depth > 1) VAEB_TRY(A(&w.da3b, enc * H));
    VAEB_TRY(A(&w.wg_scratch, (int64_t)small_wgrad_scratch_elems((int)enc, H, Z)));
  }
  w.cap_enc = enc; w.cap_dec = dec; w.with_grads = grads;
  return VAEB_OK;
}

int grow_bytes(void** p, size_t bytes) {
  if (*p) VAEB_CUDA(cudaFree(*p));
  *p = nullptr;
  VAEB_CUDA(cudaMalloc(p, bytes));
  return VAEB_OK;
}

// Allocate / grow the bf16 mirrors for `R` decoder rows and `rows` encoder rows.
int tc_ensure(vaeb_handle* h, int64_t rows, int64_t R) {
  TcState& t = h->tc;
  TcBuffers& b = t.data;
  const int D = h->D, H = h->H;
  const bool lo = t.ns == 2;
  if (b.ldh == 0) {
    // rows of the mirrors start on 32-byte sectors: a thread of a tcgen05 epilogue writes 16 bf16 = one whole sector
    // (and on whole 64-element column groups: the MN-major operands are loaded with one 3-D TMA box per tile)
    const int Dd = h->cont ? 2 * D : D;        // Gaussian decoder: [W2|W6]' and its deltas, interleaved
    b.ldh = (H + 1 + 63) / 64 * 64; b.ldd = (Dd + 1 + 63) / 64 * 64; b.ldx = (D + 1 + 63) / 64 * 64;
    VAEB_TRY(grow_bytes(&b.w3h, (size_t)D * b.ldh * 2));
    VAEB_TRY(grow_bytes(&b.w2h, (size_t)H * b.ldd * 2));
    VAEB_CUDA(cudaMemsetAsync(b.w3h, 0, (size_t)D * b.ldh * 2, h->stream));
    VAEB_CUDA(cudaMemsetAsync(b.w2h, 0, (size_t)H * b.ldd * 2, h->stream));
    VAEB_TRY(grow_bytes((void**)&b.wg_scratch, 4 * tc_wgrad_scratch_elems(D, H) * sizeof(float)));   // a region per weight gradient
    if (lo) {
      VAEB_TRY(grow_bytes(&b.w3l, (size_t)D * b.ldh * 2));
      VAEB_TRY(grow_bytes(&b.w2l, (size_t)H * b.ldd * 2));
      VAEB_CUDA(cudaMemsetAsync(b.w3l, 0, (size_t)D * b.ldh * 2, h->stream));
      VAEB_CUDA(cudaMemsetAsync(b.w2l, 0, (size_t)H * b.ldd * 2, h->stream));
    }
  }
  if (R > t.cap_R) {
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    VAEB_TRY(grow_bytes(&b.hdh, (size_t)R * b.ldh * 2));
    VAEB_TRY(grow_bytes(&b.da2h, (size_t)R * b.ldd * 2));
    if (lo) {
      VAEB_TRY(grow_bytes(&b.hdl, (size_t)R * b.ldh * 2));
      VAEB_TRY(grow_bytes(&b.da2l, (size_t)R * b.ldd * 2));
    }
    // zero padding + the ones column at H (bias row of the W2 weight-gradient GEMM)
    VAEB_LAUNCH(tc_split_matrix(h->stream, &h->launches, nullptr, R, 0, 0, b.hdh, b.hdl, b.ldh, H));
    VAEB_CUDA(cudaMemsetAsync(b.da2h, 0, (size_t)R * b.ldd * 2, h->stream));
    if (lo) VAEB_CUDA(cudaMemsetAsync(b.da2l, 0, (size_t)R * b.ldd * 2, h->stream));
    if (latent_large_batch((int)rows, H, h->Z, (int)(R / std::max<int64_t>(rows, 1)))) {
      VAEB_TRY(grow_bytes(&b.d1h, (size_t)R * b.ldh * 2));
      VAEB_TRY(grow_bytes(&b.zh, (size_t)R * b.ldz * 2));
      VAEB_CUDA(cudaMemsetAsync(b.d1h, 0, (size_t)R * b.ldh * 2, h->stream));
      if (lo) {
        VAEB_TRY(grow_bytes(&b.d1l, (size_t)R * b.ldh * 2));
        VAEB_TRY(grow_bytes(&b.zl, (size_t)R * b.ldz * 2));
        VAEB_CUDA(cudaMemsetAsync(b.d1l, 0, (size_t)R * b.ldh * 2, h->stream));
      }
      // zero padding + the ones column at Z (bias row of the W1 weight-gradient GEMM)
      VAEB_LAUNCH(tc_split_matrix(h->stream, &h->launches, nullptr, R, 0, 0, b.zh, b.zl, b.ldz, h->Z));
    }
    t.cap_R = R;
    t.key_rows = -1;
  }
  if (rows > t.cap_rows) {
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    VAEB_TRY(grow_bytes(&b.da3h, (size_t)rows * b.ldh * 2));
    VAEB_CUDA(cudaMemsetAsync(b.da3h, 0, (size_t)rows * b.ldh * 2, h->stream));
    if (lo) {
      VAEB_TRY(grow_bytes(&b.da3l, (size_t)rows * b.ldh * 2));
      VAEB_CUDA(cudaMemsetAsync(b.da3l, 0, (size_t)rows * b.ldh * 2, h->stream));
    }
    if (latent_large_batch((int)rows, H, h->Z, 1)) {
      VAEB_TRY(grow_bytes(&b.heh, (size_t)rows * b.ldh * 2));
      if (!b.w45h) {
        VAEB_TRY(grow_bytes(&b.w45h, (size_t)2 * h->Z * b.ldh * 2));
        VAEB_TRY(grow_bytes(&b.w1h, (size_t)h->Z * b.ldh * 2));
        VAEB_CUDA(cudaMemsetAsync(b.w45h, 0, (size_t)2 * h->Z * b.ldh * 2, h->stream));
        VAEB_CUDA(cudaMemsetAsync(b.w1h, 0, (size_t)h->Z * b.ldh * 2, h->stream));
        VAEB_TRY(grow_bytes(&b.whh, (size_t)H * b.ldq * 2));
        VAEB_CUDA(cudaMemsetAsync(b.whh, 0, (size_t)H * b.ldq * 2, h->stream));
        if (lo) {
          VAEB_TRY(grow_bytes(&b.whl, (size_t)H * b.ldq * 2));
          VAEB_CUDA(cudaMemsetAsync(b.whl, 0, (size_t)H * b.ldq * 2, h->stream));
        }
        if (lo) {
          VAEB_TRY(grow_bytes(&b.w45l, (size_t)2 * h->Z * b.ldh * 2));
          VAEB_TRY(grow_bytes(&b.w1l, (size_t)h->Z * b.ldh * 2));
          VAEB_CUDA(cudaMemsetAsync(b.w45l, 0, (size_t)2 * h->Z * b.ldh * 2, h->stream));
          VAEB_CUDA(cudaMemsetAsync(b.w1l, 0, (size_t)h->Z * b.ldh * 2, h->stream));
        }
      }
      VAEB_TRY(grow_bytes(&b.ddh, (size_t)rows * b.ldq * 2));
      VAEB_CUDA(cudaMemsetAsync(b.ddh, 0, (size_t)rows * b.ldq * 2, h->stream));
      if (lo) {
        VAEB_TRY(grow_bytes(&b.hel, (size_t)rows * b.ldh * 2));
        VAEB_TRY(grow_bytes(&b.ddl, (size_t)rows * b.ldq * 2));
        VAEB_CUDA(cudaMemsetAsync(b.ddl, 0, (size_t)rows * b.ldq * 2, h->stream));
      }
      // zero padding + the ones column at H (bias row of the W4|W5 weight-gradient GEMM)
      VAEB_LAUNCH(tc_split_matrix(h->stream, &h->launches, nullptr, rows, 0, 0, b.heh, b.hel, b.ldh, H));
    }
    t.cap_rows = rows;
    t.key_rows = -1;
  }
  return VAEB_OK;
}

inline float* T_(vaeb_handle* h, float* base, int idx) { return base + h->lay.off[idx]; }
inline const float* T_(vaeb_handle* h, const float* base, int idx) { return base + h->lay.off[idx]; }

// Where the bound of a step goes: base (sum of per-row bounds) always; the scalar
// (mult*base + sum(tprior))/div if scalar_out != nullptr; with loglik_rows / aux_rows (evaluation only) the two terms
// of every per-row bound.
struct BoundOut {
  float* base_out; float mult; const float* tprior; int n_tprior; float div; float* scalar_out;
  float* loglik_rows = nullptr; float* aux_rows = nullptr;
};

// Hidden layers of the encoder (VAEB.py:246; deeper encoders: replic.tex:46-57) for x[rows, D] on the fp32 per-layer kernels:
// the activations of layers 1 .. depth-1 go to ws.h_x[], the last one -- what the heads read -- to ws.h_e.
int encoder_hidden(vaeb_handle* h, const float* theta, const float* x, int rows) {
  const Layout& l = h->lay;
  Workspace& s = h->ws;
  const int D = h->D, H = h->H;
  const float* in = x;
  int K = D;
  for (int k = 1; k <= l.depth; ++k) {
    float* out = k == l.depth ? s.h_e : s.h_x[k - 1];
    const float* W = k == 1 ? T_(h, theta, l.iW3) : T_(h, theta, l.iW3x[k - 2]);
    const float* b = k == 1 ? T_(h, theta, l.ib3) : T_(h, theta, l.ib3x[k - 2]);
    VAEB_LAUNCH(launch_dense_act(h->stream, &h->launches, in, rows, K, W, b, H, h->hidden_act, out));
    in = out; K = H;
  }
  return VAEB_OK;
}

// UMMA N of the weight-gradient layers, of the activation layers and of dec2 (D wide: more column tiles per row block than
// the H-wide layers), and the x mirror the maps read, for the tcgen05 layers of one step (tc_setup)
struct TcStep {
  int bn = 64, bna = 64, bnd = 64;
  int x_row_off = 0; const void *x_hi = nullptr, *x_lo = nullptr;
};

// What both tensor-core paths set up before their first layer: the bf16 mirrors for this shape, the mirror of an x staged
// from the host, the tile widths, programmatic dependent launch and the tensor maps.
int tc_setup(vaeb_handle* h, const float* x, int rows, int R, TcStep& ts) {
  TcState& t = h->tc;
  const int D = h->D, H = h->H;
  VAEB_TRY(tc_ensure(h, rows, R));
  ts.bn = R >= 1024 ? 128 : 64;
  ts.bna = tc_act_bn(rows, std::min(H, D));
  ts.bnd = ts.bna;
  // few row blocks (the data-parallel split): one tile per CTA, and a layer should fill most of the SMs in ONE wave --
  // 64-wide tiles for the H-wide layers when 128-wide ones give fewer than 96 CTAs (2048 rows: 64 -> 128 CTAs, enc1
  // 14.5 -> 12.2 us, dgrad 15.6 -> 13.1), dec2 keeps 128 (7 column tiles per row block: 112 CTAs)
  if (ts.bna == 128) {
    const int rb = (rows + 127) / 128;
    if (rb * ((H + 127) / 128) < 96) ts.bna = 64;
    if (rb * (((h->cont ? 2 * D : D) + 127) / 128) < 96) ts.bnd = 64;
  }
  // Programmatic dependent launch for the one-tile-per-CTA kernels: bf16x3 (one CTA per SM: an early dependent grid
  // never takes slots from the running one; 16384 rows: 523 -> 499 us per update) and, in plain bf16, whenever the
  // activation layers are NOT in the persistent form (8192 rows: 215 -> 196 us); next to the persistent kernels the
  // early two-per-SM grids cost more than they hide (16384 rows: 241 -> 247 us).  Persistent launches always use it.
  tc_set_pdl(ts.bna != 256 || t.ns == 2);
  TcBuffers b = t.data;
  int64_t rows_data;
  const bool resident = h->d_x && x >= h->d_x && x < h->d_x + (size_t)h->n_data * D;
  if (resident) {
    ts.x_row_off = (int)((x - h->d_x) / D);
    rows_data = h->n_data;
  } else {
    // x was staged from the host for this call: mirror it now
    if (rows > t.cap_stage) {
      VAEB_CUDA(cudaStreamSynchronize(h->stream));
      VAEB_TRY(grow_bytes(&t.xsh, (size_t)rows * b.ldx * 2));
      if (t.ns == 2) VAEB_TRY(grow_bytes(&t.xsl, (size_t)rows * b.ldx * 2));
      t.cap_stage = rows;
      t.key_rows = -1;
    }
    PH("mirror staged x", 0, 4.0 * rows * D,
       tc_split_matrix(h->stream, &h->launches, x, rows, D, D, t.xsh, t.xsl, b.ldx, D));
    b.xh = t.xsh; b.xl = t.xsl;
    rows_data = rows;
  }
  ts.x_hi = b.xh; ts.x_lo = t.ns == 2 ? b.xl : nullptr;
  const int key_bn = (ts.bna * 1024 + ts.bn) * 1024 + ts.bnd;
  if (t.key_rows != rows || t.key_R != R || t.key_data != rows_data || t.key_bn != key_bn || t.key_x != b.xh) {
    VAEB_TRY(tc_build_maps(&t.maps, b, (int)rows_data, R, rows, D, H, ts.bna, h->Z, ts.bn, ts.bnd, h->cont ? 2 * D : D));
    t.key_rows = rows; t.key_R = R; t.key_data = rows_data; t.key_bn = key_bn; t.key_x = b.xh;
  }
  return VAEB_OK;
}

// Forward (+ backward into `grads`) of the graph of VAEB.getGradient for x[rows,D] on device, one launch per layer: the
// fp32 kernels, or with tc.active the wide layers (enc1, dec2, dgrad h_d, the W2 and W3 gradients) on tcgen05.
int forward_backward(vaeb_handle* h, const float* theta, const float* x, int rows, int L, bool want_grads, float w,
                     float w_aux, EpsSource src, float* grads, const BoundOut& bo) {
  const Layout& l = h->lay;
  Workspace& s = h->ws;
  const int D = h->D, H = h->H, Z = h->Z;
  const int R = rows * L;
  const int la = h->cfg.estimator == VAEB_EST_LA ? 1 : 0;
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  int tiles = 0;
  const double dR = R, dr = rows, dD = D, dH = H, dZ = Z, c = h->cont ? 2.0 : 1.0;
  const bool tcp = h->tc.active;
  TcState& t = h->tc;
  const TcBuffers& tb = t.data;
  TcStep ts;
  if (tcp) {
    VAEB_TRY(tc_setup(h, x, rows, R, ts));
    PH("mirror W3,W2 -> bf16", 0, 12.0 * dD * dH,
       tc_mirror_weights(st, lc, T_(h, theta, l.iW3), tb.w3h, tb.w3l, D, H, tb.ldh, T_(h, theta, l.iW2), tb.w2h, tb.w2l,
                         tb.ldd, h->cont ? T_(h, theta, l.iW6) : nullptr));
  }
  // encoder hidden layer, VAEB.py:246
  if (tcp)
    PH("enc1 x.W3+tanh [tcgen05]", 2 * dr * dD * dH, 2.0 * t.ns * (dr * dD + dD * dH) + 4 * dr * dH,
       tc_enc1(st, lc, t.maps, t.ns, ts.bna, rows, D, H, ts.x_row_off, T_(h, theta, l.ib3), s.h_e, nullptr, nullptr,
               tb.ldh));
  else if (l.depth > 1)
    VAEB_TRY(encoder_hidden(h, theta, x, rows));      // deeper encoders: replic.tex:46-57
  else
    PH("enc1 x.W3+tanh", 2 * dr * dD * dH, 4 * (dr * dD + dD * dH + dr * dH),
       launch_dense_act(st, lc, x, rows, D, T_(h, theta, l.iW3), T_(h, theta, l.ib3), H, h->hidden_act, s.h_e));
  // latent heads + reparameterisation + row terms + decoder hidden layer, VAEB.py:248-254,41-47,343
  PH("transpose W4,W5", 0, 16 * dH * dZ,
     launch_transpose_heads(st, lc, T_(h, theta, l.iW4), T_(h, theta, l.iW5), H, Z, h->d_w45t));
  PH("latent fwd (enc2,reparam,KL,dec1)", 4 * dr * dH * dZ + 2 * dR * dZ * dH,
     4 * (dr * dH + 3 * dH * dZ + 2 * dr * dZ + 2 * dR * dZ + dR * dH),
     launch_latent_fwd(st, lc, s.h_e, rows, H, h->d_w45t, T_(h, theta, l.ib4), T_(h, theta, l.ib5), T_(h, theta, l.iW1),
                       T_(h, theta, l.ib1), Z, L, la, src, s.mu, s.ls, s.eps, s.z, s.row_aux, s.h_d,
                       tcp ? tb.hdh : nullptr, tcp ? tb.hdl : nullptr, tb.ldh, h->hidden_act));
  // decoder output layer + log-likelihood, VAEB.py:257-263,302-313
  const float scale = w / (float)L;
  const float* W6 = h->cont ? T_(h, theta, l.iW6) : nullptr;
  const float* b6 = h->cont ? T_(h, theta, l.ib6) : nullptr;
  if (tcp && h->cont)
    PH("dec2 h.[W2|W6]+Gaussian loglik [tcgen05]", 4 * dR * dH * dD,
       2.0 * t.ns * (dR * dH + 2 * dH * dD) + 4 * dr * dD + (want_grads ? 4.0 * t.ns * dR * dD : 0.0),
       tc_dec2_gaussian(st, lc, t.maps, t.ns, ts.bnd, R, H, D, T_(h, theta, l.ib2), b6, x, 1, rows, scale,
                        want_grads ? tb.da2h : nullptr, want_grads ? tb.da2l : nullptr, tb.ldd, s.partial, &tiles,
                        ts.x_hi, ts.x_lo, tb.ldx, ts.x_row_off));
  else if (tcp)
    PH("dec2 h.W2+loglik [tcgen05]", 2 * dR * dH * dD,
       2.0 * t.ns * (dR * dH + dH * dD) + 4 * dr * dD + (want_grads ? 2.0 * t.ns * dR * dD : 0.0),
       tc_dec2_bernoulli(st, lc, t.maps, t.ns, ts.bnd, R, H, D, T_(h, theta, l.ib2), x, 1, rows, scale,
                         want_grads ? tb.da2h : nullptr, want_grads ? tb.da2l : nullptr, tb.ldd, s.partial, &tiles,
                         ts.x_hi, ts.x_lo, tb.ldx, ts.x_row_off));
  else
    PH("dec2 h.W2+loglik", 2 * dR * dH * dD * c,
       4 * (dR * dH + c * dH * dD + dr * dD + (want_grads ? c * dR * dD : 0.0)),
       launch_dec2_loglik(st, lc, h->cont, s.h_d, R, H, T_(h, theta, l.iW2), T_(h, theta, l.ib2), W6, b6, D, x, 1,
                          rows, scale, want_grads ? s.da2 : nullptr, want_grads ? s.dlv : nullptr, s.partial,
                          &tiles));
  if (!want_grads) {
    PH("finalize bound", 0, 4.0 * R * tiles,
       launch_finalize(st, lc, s.partial, tiles, s.row_aux, rows, L, s.per_row, bo.base_out, bo.mult, bo.tprior,
                       bo.n_tprior, bo.div, bo.scalar_out, nullptr, nullptr, bo.loglik_rows, bo.aux_rows));
    return VAEB_OK;
  }
  // backward (T.grad, VAEB.py:397); formulas in SURVEY.md 8a
  if (tcp) {
    PH("wgrad W2,b2 [tcgen05]", 2 * dR * dH * dD, 2.0 * t.ns * (dR * dH + dR * dD) + 4 * dH * dD,
       tc_wgrad2(st, lc, t.maps, t.ns, ts.bn, R, H, h->cont ? 2 * D : D, T_(h, grads, l.iW2), T_(h, grads, l.ib2),
                 tb.wg_scratch, h->cont ? T_(h, grads, l.iW6) : nullptr, h->cont ? T_(h, grads, l.ib6) : nullptr));
    PH("dgrad h_d (.W2^T)*(1-h^2) [tcgen05]", 2 * dR * dH * dD * c, 2.0 * t.ns * c * (dR * dD + dH * dD) + 8 * dR * dH,
       tc_dgrad_hd(st, lc, t.maps, t.ns, ts.bna, R, h->cont ? 2 * D : D, H, s.h_d, s.da1, nullptr, nullptr, tb.ldh,
                   tb.hdh, tb.hdl));
  } else {
    PH("wgrad W2,b2", 2 * dR * dH * dD, 4 * (dR * dH + dR * dD + dH * dD),
       launch_wgrad(st, lc, s.h_d, R, H, s.da2, D, T_(h, grads, l.iW2), T_(h, grads, l.ib2)));
    if (h->cont)
      PH("wgrad W6,b6", 2 * dR * dH * dD, 4 * (dR * dH + dR * dD + dH * dD),
         launch_wgrad(st, lc, s.h_d, R, H, s.dlv, D, T_(h, grads, l.iW6), T_(h, grads, l.ib6)));
    PH("dgrad h_d (.W2^T)*(1-h^2)", 2 * dR * dH * dD * c, 4 * (c * dR * dD + c * dH * dD + 2 * dR * dH),
       launch_dgrad_tanh(st, lc, s.da2, T_(h, theta, l.iW2), h->cont ? s.dlv : nullptr, W6, R, D, H, s.h_d, s.da1, h->hidden_act));
  }
  PH("latent bwd (dz,dmu,dls,da3,bound)", 2 * dR * dZ * dH + 4 * dr * dH * dZ,
     4 * (dR * dH + 3 * dZ * dH + 2 * dr * dH + 3 * dR * dZ + dR * tiles),
     launch_latent_bwd(st, lc, s.da1, T_(h, theta, l.iW1), h->d_w45t, s.h_e, s.z, s.eps, s.mu, s.ls, rows, H, Z, L, la, w_aux,
                       s.dmu, s.dls, s.da3, tcp ? tb.da3h : nullptr, tcp ? tb.da3l : nullptr, tb.ldh, s.partial, tiles,
                       s.row_aux, s.per_row, h->d_counter, bo.base_out, bo.mult, bo.tprior, bo.n_tprior, bo.div,
                       bo.scalar_out, h->hidden_act));
  PH("wgrad W1,b1,W4,b4,W5,b5", 2 * dR * dZ * dH + 4 * dr * dH * dZ,
     4 * (dR * dZ + dR * dH + dr * dH + 2 * dr * dZ + 3 * dH * dZ),
     launch_small_wgrad(st, lc, s.z, s.da1, R, s.h_e, s.dmu, s.dls, rows, H, Z, T_(h, grads, l.iW1),
                        T_(h, grads, l.ib1), T_(h, grads, l.iW4), T_(h, grads, l.ib4), T_(h, grads, l.iW5),
                        T_(h, grads, l.ib5), s.wg_scratch));
  if (tcp)
    PH("wgrad W3,b3 [tcgen05]", 2 * dr * dD * dH, 2.0 * t.ns * (dr * dD + dr * dH) + 4 * dD * dH,
       tc_wgrad3(st, lc, t.maps, t.ns, ts.bn, rows, D, H, ts.x_row_off, T_(h, grads, l.iW3), T_(h, grads, l.ib3),
                 tb.wg_scratch));
  else {
    // deeper encoders: da3 is the gradient at the pre-activation of the LAST hidden layer; for k = depth .. 2 the layer's
    // weight gradient is h_{k-1}^T . da_k and da_{k-1} = (da_k . W3_k^T) * f'(h_{k-1})
    float* dcur = s.da3;
    float* dnext = s.da3b;
    for (int k = l.depth; k >= 2; --k) {
      const float* hprev = s.h_x[k - 2];
      VAEB_LAUNCH(launch_wgrad(st, lc, hprev, rows, H, dcur, H, T_(h, grads, l.iW3x[k - 2]), T_(h, grads, l.ib3x[k - 2])));
      VAEB_LAUNCH(launch_dgrad_tanh(st, lc, dcur, T_(h, theta, l.iW3x[k - 2]), nullptr, nullptr, rows, H, H, hprev, dnext,
                                    h->hidden_act));
      float* t2 = dcur; dcur = dnext; dnext = t2;
    }
    PH("wgrad W3,b3", 2 * dr * dD * dH, 4 * (dr * dD + dr * dH + dD * dH),
       launch_wgrad(st, lc, x, rows, D, dcur, H, T_(h, grads, l.iW3), T_(h, grads, l.ib3)));
  }
  return VAEB_OK;
}

// Training gradients of a large batch on the tensor-core path (latent_large_batch: L = 1): every layer runs on tcgen05,
// the thin latent ones too (their operands' bf16 mirrors come from the kernels that produce h_e, z, da1 and [dmu|dls]),
// and the four weight-gradient GEMMs are one launch after the last dgrad, their split-K slices left in scratch.  With
// `tail` the update ends in ONE launch that also applies prior + Adagrad or Adam; else the bound and the sum of the slices are
// launched here and the caller applies the update.
int large_batch_step(vaeb_handle* h, const float* theta, const float* x, int rows, float w, float w_aux, EpsSource src,
                     float* grads, const BoundOut& bo, bool tail) {
  const Layout& l = h->lay;
  Workspace& s = h->ws;
  const int D = h->D, H = h->H, Z = h->Z;
  const int R = rows;                     // L = 1
  const int la = h->cfg.estimator == VAEB_EST_LA ? 1 : 0;
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  int tiles = 0;
  const double dR = R, dr = rows, dD = D, dH = H, dZ = Z, c = h->cont ? 2.0 : 1.0;
  TcState& t = h->tc;
  const TcBuffers& tb = t.data;
  TcStep ts;
  VAEB_TRY(tc_setup(h, x, rows, R, ts));
  if (!t.weights_ready || theta != h->d_params)   // (else the tail of the previous update wrote the mirrors of theta)
    PH("weight mirrors / transposes -> bf16 (one launch)", 0, 12.0 * dD * dH + 60.0 * dZ * dH,
       tc_prepare_weights(st, lc, T_(h, theta, l.iW3), T_(h, theta, l.iW2), T_(h, theta, l.iW4), T_(h, theta, l.iW5),
                          T_(h, theta, l.iW1), tb, h->d_w45t, D, H, Z, h->cont ? T_(h, theta, l.iW6) : nullptr));
  // encoder hidden layer, VAEB.py:246: every consumer of h_e reads its mirror
  PH("enc1 x.W3+tanh [tcgen05]", 2 * dr * dD * dH, 2.0 * t.ns * (dr * dD + dD * dH) + 4 * dr * dH,
     tc_enc1(st, lc, t.maps, t.ns, ts.bna, rows, D, H, ts.x_row_off, T_(h, theta, l.ib3), nullptr, tb.heh, tb.hel, tb.ldh));
  // latent heads + reparameterisation + row terms, VAEB.py:248-249,41-47,343.  The KL / L^A row partials: when the tail
  // kernel ends the update it sums them itself (they are parked in the dz workspace, idle on this path: s.partial is
  // overwritten by dec2), else a small launch folds them into row_aux now
  const bool aux_to_tail = tail && 4 * ((2 * Z + 63) / 64) <= Z;
  int n_aux = 0;
  PH("enc2 h_e.[W4|W5] + reparam + KL [tcgen05]", 4 * dr * dH * dZ, 2.0 * t.ns * (dr * dH + 2 * dH * dZ) + 20 * dr * dZ,
     tc_enc2_heads(st, lc, t.maps, t.ns, rows, H, Z, la, T_(h, theta, l.ib4), T_(h, theta, l.ib5), src, s.mu, s.ls,
                   s.eps, s.z, tb.zh, tb.zl, tb.ldz, aux_to_tail ? s.dz : s.partial, &n_aux));
  if (!aux_to_tail) VAEB_LAUNCH(launch_row_partials_sum(st, lc, s.partial, n_aux, rows, s.row_aux));
  // decoder hidden layer, VAEB.py:254
  PH("dec1 tanh(z.W1+b1) [tcgen05]", 2 * dR * dZ * dH, 2.0 * t.ns * (dR * 32 + dZ * dH) + 4 * dR * dH + 2.0 * t.ns * dR * dH,
     tc_dec1(st, lc, t.maps, t.ns, ts.bna, R, Z, H, T_(h, theta, l.ib1), nullptr, tb.hdh, tb.hdl, tb.ldh));
  // decoder output layer + log-likelihood, VAEB.py:257-263,302-313; x from the mirror enc1 reads
  if (h->cont)
    PH("dec2 h.[W2|W6]+Gaussian loglik [tcgen05]", 4 * dR * dH * dD,
       2.0 * t.ns * (dR * dH + 2 * dH * dD) + 4 * dr * dD + 4.0 * t.ns * dR * dD,
       tc_dec2_gaussian(st, lc, t.maps, t.ns, ts.bnd, R, H, D, T_(h, theta, l.ib2), T_(h, theta, l.ib6), nullptr, 1, rows,
                        w, tb.da2h, tb.da2l, tb.ldd, s.partial, &tiles, ts.x_hi, ts.x_lo, tb.ldx, ts.x_row_off));
  else
    PH("dec2 h.W2+loglik [tcgen05]", 2 * dR * dH * dD,
       2.0 * t.ns * (dR * dH + dH * dD) + 4 * dr * dD + 2.0 * t.ns * dR * dD,
       tc_dec2_bernoulli(st, lc, t.maps, t.ns, ts.bnd, R, H, D, T_(h, theta, l.ib2), nullptr, 1, rows, w, tb.da2h,
                         tb.da2l, tb.ldd, s.partial, &tiles, ts.x_hi, ts.x_lo, tb.ldx, ts.x_row_off));
  // backward (T.grad, VAEB.py:397); formulas in SURVEY.md 8a
  PH("dgrad h_d (.W2^T)*(1-h^2) [tcgen05]", 2 * dR * dH * dD * c, 2.0 * t.ns * c * (dR * dD + dH * dD) + 8 * dR * dH,
     tc_dgrad_hd(st, lc, t.maps, t.ns, ts.bna, R, h->cont ? 2 * D : D, H, nullptr, nullptr, tb.d1h, tb.d1l, tb.ldh,
                 tb.hdh, tb.hdl));
  PH("dz da1.W1^T + dmu,dls [tcgen05]", 2 * dR * dZ * dH, 2.0 * t.ns * (dR * dH + dZ * dH) + 28 * dR * dZ,
     tc_dz_dprep(st, lc, t.maps, t.ns, R, H, Z, la, w_aux, s.z, s.eps, s.mu, s.ls, s.dmu, s.dls, tb.ddh, tb.ddl, tb.ldq));
  if (!tail)
    PH("bound (per row + total)", 0, 4 * (dR * tiles + 2 * dr),
       launch_finalize(st, lc, s.partial, tiles, s.row_aux, rows, 1, s.per_row, bo.base_out, bo.mult, bo.tprior,
                       bo.n_tprior, bo.div, bo.scalar_out, h->d_counter, s.dec_aux));   // dec_aux: idle outside the IS path
  PH("dgrad h_e ([dmu|dls].W45^T)*(1-h^2) [tcgen05]", 4 * dr * dH * dZ, 2.0 * t.ns * (dr * 64 + 2 * dZ * dH) + 8 * dr * dH,
     tc_dgrad_he(st, lc, t.maps, t.ns, ts.bna, rows, Z, H, nullptr, nullptr, tb.da3h, tb.da3l, tb.ldh, tb.heh, tb.hel));
  if (t.n_sm == 0) VAEB_CUDA(cudaDeviceGetAttribute(&t.n_sm, cudaDevAttrMultiProcessorCount, h->cfg.device));
  TcReduceJobs jobs;
  PH("wgrad W2,W1,W4|W5,W3 (+ biases) [tcgen05, one launch]", 4 * dR * dH * dD + 2 * dR * dZ * dH + 4 * dr * dH * dZ,
     2.0 * t.ns * (2 * dR * dH + 2 * dR * dD) + 8 * dH * dD,
     tc_wgrad_all(st, lc, t.maps, t.ns, ts.bn, R, rows, D, H, Z, ts.x_row_off, T_(h, grads, l.iW2), T_(h, grads, l.ib2),
                  T_(h, grads, l.iW1), T_(h, grads, l.ib1), T_(h, grads, l.iW4), T_(h, grads, l.ib4), T_(h, grads, l.iW5),
                  T_(h, grads, l.ib5), T_(h, grads, l.iW3), T_(h, grads, l.ib3), tb.wg_scratch,
                  tc_wgrad_scratch_elems(D, H), &jobs, t.n_sm, h->cont ? T_(h, grads, l.iW6) : nullptr,
                  h->cont ? T_(h, grads, l.ib6) : nullptr));
  if (!tail) {
    if (jobs.n > 0) PH("sum of the split-K weight-gradient slices (one launch)", 0, 0, tc_wgrad_reduce_all(st, lc, jobs));
    return VAEB_OK;
  }
  // the tail as one launch (tc_tail.cu): slices -> gradient, bound, (data parallel over peer memory: the gradient sum,)
  // prior + Adagrad or Adam and the bf16 weight mirrors of the new parameters
  const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES, dp = h->world > 1;
  if (!t.tail_bar) {
    VAEB_CUDA(cudaMalloc((void**)&t.tail_bar, sizeof(unsigned int)));
    VAEB_CUDA(cudaMemsetAsync(t.tail_bar, 0, sizeof(unsigned int), st));
    t.tail_bar_count = 0;
  }
  TcTailArgs ta{};
  ta.jobs = jobs;
  ta.params = h->d_params; ta.ada = h->d_ada; ta.grads = h->d_grads; ta.padded = l.padded;
  ta.lr = h->cfg.learning_rate; ta.eps = h->cfg.adagrad_eps; ta.prior = fb ? 0.f : h->cfg.prior_scale;
  ta.p2 = fb ? h->cfg.learning_rate * 1e-6f : 0.f;
  ta.partial = s.partial; ta.n_tiles = tiles; ta.rows = rows;
  ta.aux_part = aux_to_tail ? s.dz : nullptr; ta.n_aux = aux_to_tail ? n_aux : 0; ta.row_aux = aux_to_tail ? nullptr : s.row_aux;
  ta.per_row = s.per_row; ta.block_part = s.dec_aux; ta.base_out = bo.base_out;
  ta.mult = bo.mult; ta.div = bo.div; ta.scalar_out = bo.scalar_out;
  ta.w3h = tb.w3h; ta.w3l = tb.w3l; ta.w2h = tb.w2h; ta.w2l = tb.w2l; ta.w45h = tb.w45h; ta.w45l = tb.w45l;
  ta.whh = tb.whh; ta.whl = tb.whl; ta.w1h = tb.w1h; ta.w1l = tb.w1l; ta.w45t = h->d_w45t;
  ta.D = D; ta.H = H; ta.Z = Z; ta.ldh = tb.ldh; ta.ldd = tb.ldd; ta.ldq = tb.ldq;
  ta.oW3 = l.off[l.iW3]; ta.oW4 = l.off[l.iW4]; ta.oW5 = l.off[l.iW5]; ta.oW1 = l.off[l.iW1]; ta.oW2 = l.off[l.iW2];
  ta.oW6 = h->cont ? l.off[l.iW6] : -1;
  ta.bar = t.tail_bar;
  ta.world = h->world; ta.rank = h->rank;
  const bool adam = h->optimizer == VAEB_OPT_ADAM;
  if (adam) {
    ta.alpha_t = h->adam_alpha_t; ta.s2_t = h->adam_s2_t; ta.b1 = h->adam_b1; ta.b2 = h->adam_b2; ta.adam_eps = h->adam_eps;
    ta.v = h->d_adam_v;
  }
  for (int r = 0; r < h->world && dp; ++r) {
    ta.gsum[r] = t.p2p_gsum[r]; ta.flags[r] = t.p2p_flags[r];
    ta.peer_params[r] = t.p2p_params[r]; ta.peer_ada[r] = t.p2p_ada[r];
    if (adam) ta.peer_v[r] = t.p2p_ada[r] + (l.padded + 4);      // every rank keeps v right after m (vaeb_set_adam)
  }
  const int grid = tc_tail_grid(t.n_sm, adam);
  auto launch_tail = [&]() -> cudaError_t {
    ta.bar_base = t.tail_bar_count;
    ta.epoch = ++t.p2p_epoch;
    t.tail_bar_count += (unsigned int)grid * (dp ? 2u : 1u);
    return tc_tail_launch(st, lc, ta, grid, adam);
  };
  if (adam)
    PH("tail: slices -> gradient, bound, (all-reduce over peer memory,) prior + Adam, weight mirrors (one launch)", 0,
       36.0 * (double)l.total, launch_tail());
  else
    PH("tail: slices -> gradient, bound, (all-reduce over peer memory,) prior + Adagrad, weight mirrors (one launch)", 0,
       28.0 * (double)l.total, launch_tail());
  return VAEB_OK;
}

int ensure_scalars(vaeb_handle* h, int n) {
  if (n <= h->scalars_cap) return VAEB_OK;
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  if (h->d_scalars) VAEB_CUDA(cudaFree(h->d_scalars));
  if (h->h_scalars) VAEB_CUDA(cudaFreeHost(h->h_scalars));
  VAEB_CUDA(cudaMalloc((void**)&h->d_scalars, (size_t)n * sizeof(float)));
  VAEB_CUDA(cudaMallocHost((void**)&h->h_scalars, (size_t)n * sizeof(float)));
  h->scalars_cap = n;
  return VAEB_OK;
}

// beta_n of vaeb_set_kl_weight for the n-th update applied since the call (n >= 1): in double, rounded to float once
float kl_weight_at(const vaeb_handle* h, int64_t n) {
  if (h->kl_warmup == 0 || n >= h->kl_warmup) return h->kl_beta;
  return (float)((double)h->kl_beta * ((double)n / (double)h->kl_warmup));
}

int stage_in(vaeb_handle* h, float** dbuf, int64_t* cap, const float* host, int64_t n) {
  VAEB_TRY(grow(dbuf, cap, n));
  VAEB_CUDA(cudaMemcpyAsync(*dbuf, host, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  return VAEB_OK;
}

int all_reduce_grads(vaeb_handle* h) {
  if (h->world <= 1) return VAEB_OK;
  const int r = h->nccl.AllReduce(h->d_grads, h->d_grads, (size_t)(h->lay.padded + 4), /*ncclFloat32*/ 7,
                                  /*ncclSum*/ 0, h->comm, h->stream);
  if (r != 0) {
    vaeb_set_error(std::string("ncclAllReduce: ") + (h->nccl.GetErrorString ? h->nccl.GetErrorString(r) : "?"));
    return VAEB_ENCCL;
  }
  return VAEB_OK;
}

// One update on device-resident rows; the scalar lands in d_scalars[slot].
int enqueue_update(vaeb_handle* h, const float* d_xrows, int rows, const float* d_eps, const float* d_zeta,
                   int slot, bool apply) {
  const Layout& l = h->lay;
  const int L = h->L;
  VAEB_TRY(ensure_ws(h, rows, (int64_t)rows * L, true));
  EpsSource src{d_eps, h->cfg.seed, VAEB_STREAM_TRAIN, h->step, (int64_t)h->rank * rows};
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  float* base = h->d_grads + l.padded;
  const int64_t n4 = l.padded / 4;
  const float Mg = (float)rows * (float)h->world;
  const bool large = h->tc.active && latent_large_batch(rows, h->H, h->Z, L);
  bool tail = false;
  const bool adam = h->optimizer == VAEB_OPT_ADAM;
  if (apply && adam) {            // Adam step t of this update: bias corrections in double, rounded to float once
    const double t = (double)(h->adam_t + 1);          // (h->adam_t advances below, once the update is enqueued)
    h->adam_alpha_t = (float)((double)h->cfg.learning_rate / (1.0 - std::pow((double)h->adam_b1, t)));
    h->adam_s2_t = (float)std::sqrt(1.0 - std::pow((double)h->adam_b2, t));
  }
  if (!is_fvb(h)) {
    const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES;
    const float w = fb ? 1.0f / Mg : 1.0f;
    // the latent term's weight: beta_n of the update this one would be if applied (h->kl_t advances below)
    const float w_aux = w * kl_weight_at(h, h->kl_t + 1);
    const bool dp = h->world > 1;
    const float prior = fb ? 0.f : h->cfg.prior_scale;
    // Large-batch tensor-core path: everything after the last GEMM is ONE launch (tc_tail.cu) -- and in data-parallel
    // runs whose ranks mapped each other's buffers (vaeb_comm_p2p_attach) that launch is also the gradient all-reduce.
    // With the single weight-gradient launch in front of it, it measures equal to the five separate launches at 16384 rows
    // and 1-3 % faster below on one GPU; VAEB_TC_TAIL=0 switches it off (then: slice sum, row sums, bound, Adagrad, mirrors).
    static const int env_tail = getenv("VAEB_TC_TAIL") ? atoi(getenv("VAEB_TC_TAIL")) : -1;      // measurement switch
    tail = large && apply && (h->optimizer == VAEB_OPT_ADAGRAD || adam) && env_tail != 0 && (!dp || h->tc.p2p_ready);
    // data parallel without the tail: the optimizer launch writes the scalar, after the all-reduce
    BoundOut bo{base, 1.0f, nullptr, 0, Mg, dp && !tail ? nullptr : h->d_scalars + slot};
    if (large) VAEB_TRY(large_batch_step(h, h->d_params, d_xrows, rows, w, w_aux, src, h->d_grads, bo, tail));
    else VAEB_TRY(forward_backward(h, h->d_params, d_xrows, rows, L, true, w, w_aux, src, h->d_grads, bo));
    if (!tail) {                          // (the tail applied prior + Adagrad / Adam)
      VAEB_TRY(all_reduce_grads(h));
      if (apply && adam)
        PH("adam+prior (flat)", 0, 28.0 * (double)l.total,
           launch_adam(st, lc, h->d_params, h->d_ada, h->d_adam_v, h->d_grads, n4, h->adam_alpha_t, h->adam_s2_t,
                       h->adam_b1, h->adam_b2, h->adam_eps, prior, base, 1.0f, Mg, dp ? h->d_scalars + slot : nullptr));
      else if (apply && h->optimizer == VAEB_OPT_ADADELTA)
        PH("adadelta+prior (flat)", 0, 28.0 * (double)l.total,
           launch_adadelta(st, lc, h->d_params, h->d_ada, h->d_ada2, h->d_grads, n4, h->rho, h->cfg.adagrad_eps, prior,
                           base, 1.0f, Mg, dp ? h->d_scalars + slot : nullptr));
      else if (apply)
        PH("adagrad+prior (flat)", 0, 20.0 * (double)l.total,
           launch_adagrad(st, lc, h->d_params, h->d_ada, h->d_grads, n4, h->cfg.learning_rate, h->cfg.adagrad_eps,
                          prior, fb ? h->cfg.learning_rate * 1e-6f : 0.f, base, 1.0f, Mg,
                          dp ? h->d_scalars + slot : nullptr));
      else
        VAEB_LAUNCH(launch_add_prior(st, lc, h->d_grads, h->d_params, n4, prior, base, 1.0f, Mg,
                                     dp ? h->d_scalars + slot : nullptr));
    }
    h->grads_have_prior = !apply;
  } else {
    VAEB_REQUIRE(h->world == 1, "full-VB estimators are single-GPU (replicas only)");
    const bool sampled = h->cfg.estimator == VAEB_EST_FVB_SAMPLED;
    const float* theta = h->d_params;  // VAEB.py:119,352: frozen MAP parameters, weights never sampled
    if (sampled) {
      VAEB_LAUNCH(launch_sample_theta(st, lc, h->d_vmu, h->d_vsig, d_zeta, h->cfg.seed, h->step, l.total, h->d_theta,
                                      h->d_zeta));
      theta = h->d_theta;
    }
    VAEB_LAUNCH(launch_theta_prior(st, lc, h->d_vmu, h->d_vsig, l.total, h->d_tprior));
    // SGVB = x.shape[0]*(sum logp + sum KL) + thetaPrior (VAEB.py:364); update returns SGVB/M
    BoundOut bo{base, (float)rows, h->d_tprior, VAEB_TP_BLOCKS, apply ? (float)rows : 1.0f, h->d_scalars + slot};
    if (large && sampled) VAEB_TRY(large_batch_step(h, theta, d_xrows, rows, (float)rows, (float)rows, src, h->d_grads, bo, false));
    else VAEB_TRY(forward_backward(h, theta, d_xrows, rows, L, sampled, (float)rows, (float)rows, src, h->d_grads, bo));
    VAEB_LAUNCH(launch_fvb_adagrad(st, lc, h->d_vmu, h->d_vsig, h->d_ada_mu, h->d_ada_sig, h->d_grads, h->d_zeta,
                                   sampled ? 1 : 0, l.total, h->cfg.learning_rate, h->cfg.adagrad_eps,
                                   h->cfg.prior_scale, h->d_gmu, h->d_gsig, apply ? 1 : 0));
  }
  if (apply) invalidate_weight_mirrors(h);
  if (tail) h->tc.weights_ready = true;         // the tail wrote the large-batch path's mirrors of the new parameters
  if (apply && adam) ++h->adam_t;
  if (apply) ++h->kl_t;
  ++h->step;
  return VAEB_OK;
}

int read_scalars(vaeb_handle* h, int n, float* out) {
  VAEB_CUDA(cudaMemcpyAsync(h->h_scalars, h->d_scalars, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  std::memcpy(out, h->h_scalars, (size_t)n * sizeof(float));
  return VAEB_OK;
}

float* flat_by_which(vaeb_handle* h, int which) {
  switch (which) {
    case 0: return h->d_params;
    case 1: return h->d_ada;
    case 2: return h->d_grads;
    case 3: return h->d_vmu;
    case 4: return h->d_vsig;
    case 5: return h->d_ada_mu;
    case 6: return h->d_ada_sig;
    case 7: return h->d_gmu;
    case 8: return h->d_gsig;
    case 9: return h->optimizer == VAEB_OPT_ADAM ? h->d_adam_v : h->d_ada2;
    case 10: return h->d_theta;     // sampled full VB: theta and zeta of the next step (training state)
    case 11: return h->d_zeta;
    default: return nullptr;
  }
}

int load_nccl(NcclApi& api, const char* path) {
  if (api.lib) return VAEB_OK;
  api.lib = dlopen(path && path[0] ? path : "libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
  if (!api.lib) { vaeb_set_error(std::string("dlopen nccl: ") + dlerror()); return VAEB_ENCCL; }
  api.GetUniqueId = (int (*)(void*))dlsym(api.lib, "ncclGetUniqueId");
  api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(api.lib, "ncclCommInitRank");
  api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(api.lib, "ncclAllReduce");
  api.CommDestroy = (int (*)(void*))dlsym(api.lib, "ncclCommDestroy");
  api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) {
    vaeb_set_error("nccl library lacks a required symbol");
    return VAEB_ENCCL;
  }
  return VAEB_OK;
}

}  // namespace

// How an update of `rows` rows runs: ONE launch of the tensor-core step kernel (step_tc.cu) or of the fp32 FFMA one
// (fused_step.cu), or the per-layer kernels of enqueue_update.  The values are those of vaeb_step_kernel.
enum StepPath { PER_LAYER = 0, FUSED = 1, STEP_TC = 2 };

// What both single-launch kernels implement: the four estimators, L = 1, one GPU, one encoder hidden layer, tanh hidden
// layers and Adagrad applied in their weight-gradient epilogues.
static bool single_launch_model(const vaeb_handle* h) {
  const int e = h->cfg.estimator;
  return (e == VAEB_EST_LB || e == VAEB_EST_LA || e == VAEB_EST_FVB || e == VAEB_EST_FVB_SAMPLED) && h->L == 1 &&
         h->world == 1 && h->lay.depth == 1 && h->hidden_act == VAEB_ACT_TANH && h->optimizer == VAEB_OPT_ADAGRAD;
}

bool fused_step_supported(const vaeb_handle* h, int rows) {
  return !h->env_no_fused && single_launch_model(h) && h->cfg.precision == VAEB_PREC_FP32 && rows >= 1 && rows <= 4096;
}

static bool step_tc_supported(const vaeb_handle* h, int rows) {
  return !h->steptc.unavailable && !h->env_no_step_tc && single_launch_model(h) && h->cfg.precision != VAEB_PREC_BF16 &&
         rows >= 1 && rows <= st2::MP && (h->D % 8) == 0 && (h->H % 4) == 0 && h->D >= 64 && h->H >= 64 && h->D <= 1024 &&
         h->H <= 512 && h->Z >= 1 && h->Z <= 20 &&
         (!h->cont || fused_step_supported(h, rows));   // Gaussian decoder: the fp32 kernel takes over a step whose deltas
}                                                       // leave the fp16 range

static StepPath step_path(const vaeb_handle* h, int rows) {
  if (step_tc_supported(h, rows)) return STEP_TC;
  return fused_step_supported(h, rows) ? FUSED : PER_LAYER;
}

// n updates of `rows` rows in ONE launch of the kernel of `path` (STEP_TC or FUSED); their bounds land in
// d_scalars[slot0 ..].  The minibatch indices of the updates come from the host (host_order) or are on the device
// already (d_order); see fused_step_launch for how they and d_xrows address the rows.
static int run_single_launch(vaeb_handle* h, StepPath path, const int32_t* host_order, const int* d_order,
                             const float* d_xrows, int rows, int n, const float* d_eps, int slot0, long long* d_timing) {
  // the fp32 kernel's workspace, for step_tc_launch too: it hands a Gaussian step whose deltas overflow to that kernel
  VAEB_TRY(ensure_ws(h, rows, rows, true));
  VAEB_TRY(ensure_scalars(h, slot0 + n));
  if (host_order) {
    if (n > h->order_cap) {
      VAEB_CUDA(cudaStreamSynchronize(h->stream));
      if (h->d_order) VAEB_CUDA(cudaFree(h->d_order));
      h->d_order = nullptr;
      VAEB_CUDA(cudaMalloc((void**)&h->d_order, (size_t)n * sizeof(int)));
      h->order_cap = n;
    }
    VAEB_CUDA(cudaMemcpyAsync(h->d_order, host_order, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    d_order = h->d_order;
  }
  // the KL weight of every update of the launch (none while it is 1 throughout: the kernels then read no weights)
  const float* d_kl = nullptr;
  if (h->kl_beta != 1.f || h->kl_warmup != 0) {
    if (n > h->kl_cap) {
      VAEB_CUDA(cudaStreamSynchronize(h->stream));
      if (h->d_kl) VAEB_CUDA(cudaFree(h->d_kl));
      h->d_kl = nullptr;
      VAEB_CUDA(cudaMalloc((void**)&h->d_kl, (size_t)n * sizeof(float)));
      h->kl_cap = n;
    }
    std::vector<float> kl((size_t)n);
    for (int i = 0; i < n; ++i) kl[(size_t)i] = kl_weight_at(h, h->kl_t + 1 + i);
    // (pageable source: the call returns once the values are staged, so `kl` may go out of scope)
    VAEB_CUDA(cudaMemcpyAsync(h->d_kl, kl.data(), (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    d_kl = h->d_kl;
  }
  const int rc = path == STEP_TC ? step_tc_launch(h, d_order, d_kl, d_xrows, rows, n, d_eps, slot0, d_timing)
                                 : fused_step_launch(h, d_order, d_kl, d_xrows, rows, n, d_eps, slot0, d_timing);
  if (rc == VAEB_OK) h->kl_t += n;
  return rc;
}

extern "C" {

// Backup of params + accumulators (Adam: m, v and the Adam step; the KL step) around the profiling entry points: restored and freed
// on EVERY exit path
struct StateBackup {
  vaeb_handle* h; size_t nb, nba; float* bp = nullptr; float* ba = nullptr; uint32_t step0; int64_t launches0, adam_t0, kl_t0;
  StateBackup(vaeb_handle* hh, size_t n)
      : h(hh), nb(n), nba(hh->d_adam_v ? 2 * n : n), step0(hh->step), launches0(hh->launches), adam_t0(hh->adam_t),
        kl_t0(hh->kl_t) {}
  cudaError_t take() {
    cudaError_t e = cudaMalloc((void**)&bp, nb);
    if (e == cudaSuccess) e = cudaMalloc((void**)&ba, nba);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bp, h->d_params, nb, cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ba, h->d_ada, nba, cudaMemcpyDeviceToDevice, h->stream);   // m and v
    return e;
  }
  ~StateBackup() {
    invalidate_weight_mirrors(h);
    h->step = step0;
    h->launches = launches0;
    h->adam_t = adam_t0;
    h->kl_t = kl_t0;
    if (bp && ba) {
      cudaMemcpyAsync(h->d_params, bp, nb, cudaMemcpyDeviceToDevice, h->stream);
      cudaMemcpyAsync(h->d_ada, ba, nba, cudaMemcpyDeviceToDevice, h->stream);
      cudaStreamSynchronize(h->stream);
    }
    if (bp) cudaFree(bp);
    if (ba) cudaFree(ba);
  }
};

static int async_flush(vaeb_handle* h);
static void p2p_release(vaeb_handle* h);   // unmaps the peers' buffers (data parallel over peer memory)   // launches streaming updates that were copied but not yet started

const char* vaeb_last_error(void) { return g_last_error.c_str(); }
int vaeb_version(void) { return 106; }   // 106: vaeb_step_counter; 105: vaeb_profile_optimizer without variant; 104: KL weight; 103: Adam; 102: vaeb_encode, vaeb_sample, vaeb_validate_terms (101: encoder_hidden_layers)
int vaeb_config_size(void) { return (int)sizeof(vaeb_config); }

int vaeb_create(const vaeb_config* cfg, vaeb_handle** out) {
  VAEB_REQUIRE(cfg && out, "null argument");
  VAEB_REQUIRE(cfg->input_dim > 0 && cfg->hidden_units > 0 && cfg->latent_size > 0, "dimensions must be positive");
  VAEB_REQUIRE(cfg->batch_size > 0 && cfg->L > 0, "batch_size and L must be positive");
  VAEB_REQUIRE(cfg->estimator >= 0 && cfg->estimator <= 3, "unknown estimator");
  VAEB_REQUIRE(cfg->variant == 0 || cfg->variant == 1, "unknown variant");
  VAEB_REQUIRE(cfg->precision >= VAEB_PREC_FP32 && cfg->precision <= VAEB_PREC_BF16X3, "unknown precision");
  const bool fvb = cfg->estimator >= VAEB_EST_FVB;
  VAEB_REQUIRE(cfg->encoder_hidden_layers >= 0 && cfg->encoder_hidden_layers <= 4, "encoder_hidden_layers must be 0..4");
  VAEB_REQUIRE(cfg->encoder_hidden_layers <= 1 || (cfg->precision == VAEB_PREC_FP32 && !fvb),
               "deeper encoders: fp32 per-layer kernels, L^A / L^B estimators");
  // getFVBL overwrites `mu` inside the sample loop (VAEB.py:361): undefined for L > 1
  VAEB_REQUIRE(!(fvb && cfg->L != 1), "full-VB bound is only defined for L == 1 (VAEB.py:361)");
  VAEB_REQUIRE(!(fvb && cfg->variant != VAEB_VARIANT_VAEB), "full-VB exists only in VAEB.py");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    vaeb_set_error(std::string("no CUDA device: ") + cudaGetErrorString(e) + " (there is no CPU fallback)");
    return VAEB_ECUDA;
  }
  VAEB_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device ordinal out of range");
  VAEB_CUDA(cudaSetDevice(cfg->device));
  vaeb_handle* h = new vaeb_handle();
  h->cfg = *cfg;
  h->D = cfg->input_dim; h->H = cfg->hidden_units; h->Z = cfg->latent_size; h->M = cfg->batch_size; h->L = cfg->L;
  h->cont = cfg->continuous != 0;
  build_layout(h->lay, h->D, h->H, h->Z, h->cont, cfg->encoder_hidden_layers);
  { const char* e = getenv("VAEB_B200_FUSED"); h->env_no_fused = e && e[0] == '0'; }
  { const char* e = getenv("VAEB_B200_STEP_TC"); h->env_no_step_tc = e && e[0] == '0'; }
  h->tc.active = cfg->precision != VAEB_PREC_FP32;
  h->tc.ns = cfg->precision == VAEB_PREC_BF16X3 ? 2 : 1;
  VAEB_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  const int64_t n = h->lay.padded + 4;
  VAEB_TRY(alloc_flat(&h->d_params, n));
  VAEB_TRY(alloc_flat(&h->d_ada, n));
  VAEB_TRY(alloc_flat(&h->d_grads, n));
  if (fvb) {
    VAEB_TRY(alloc_flat(&h->d_vmu, n));
    VAEB_TRY(alloc_flat(&h->d_vsig, n, cfg->sigma_vb_init));
    VAEB_TRY(alloc_flat(&h->d_ada_mu, n));
    VAEB_TRY(alloc_flat(&h->d_ada_sig, n));
    VAEB_TRY(alloc_flat(&h->d_gmu, n));
    VAEB_TRY(alloc_flat(&h->d_gsig, n));
    VAEB_TRY(alloc_flat(&h->d_theta, n));
    VAEB_TRY(alloc_flat(&h->d_zeta, n));
    VAEB_TRY(alloc_flat(&h->d_tprior, VAEB_TP_BLOCKS));
  }
  VAEB_CUDA(cudaMalloc((void**)&h->d_counter, sizeof(unsigned int)));
  VAEB_CUDA(cudaMalloc((void**)&h->d_w45t, (size_t)2 * h->Z * h->H * sizeof(float)));
  VAEB_CUDA(cudaMemset(h->d_counter, 0, sizeof(unsigned int)));
  VAEB_TRY(ensure_scalars(h, 1024));
  *out = h;
  return VAEB_OK;
}

int vaeb_destroy(vaeb_handle* h) {
  if (!h) return VAEB_OK;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  p2p_release(h);
  if (h->tc.tail_bar) cudaFree(h->tc.tail_bar);
  if (h->comm && h->nccl.CommDestroy) h->nccl.CommDestroy(h->comm);
  free_ws(h->ws);
  float* bufs[] = {h->d_params, h->d_ada, h->d_grads, h->d_vmu, h->d_vsig, h->d_ada_mu, h->d_ada_sig, h->d_gmu,
                   h->d_gsig, h->d_theta, h->d_zeta, h->d_tprior, h->d_x, h->d_stage, h->d_stage2, h->d_out,
                   h->d_scalars, h->d_ada2};
  for (float* p : bufs) if (p) cudaFree(p);
  if (h->d_order) cudaFree(h->d_order);
  if (h->d_kl) cudaFree(h->d_kl);
  if (h->d_counter) cudaFree(h->d_counter);
  if (h->d_w45t) cudaFree(h->d_w45t);
  step_tc_free(h->steptc);
  {
    FusedState& f = h->fused;
    void* fb[] = {f.bar, f.params_alt, f.partial, f.aux_part, f.tprior_part, f.d_timing};
    for (void* q : fb) if (q) cudaFree(q);
  }
  {
    TcBuffers& b = h->tc.data;
    void* tb[] = {b.xh, b.xl, b.w3h, b.w3l, b.w2h, b.w2l, b.hdh, b.hdl, b.da2h, b.da2l, b.da3h, b.da3l, h->tc.xsh, h->tc.xsl, b.wg_scratch,
                  b.heh, b.hel, b.d1h, b.d1l, b.zh, b.zl, b.ddh, b.ddl, b.w45h, b.w45l, b.w1h, b.w1l, b.whh, b.whl};
    for (void* q : tb) if (q) cudaFree(q);
  }
  {
    IsTcState& q = h->istc;
    if (q.bias26) cudaFree(q.bias26);
    if (q.copy) {
      cudaStreamSynchronize(q.copy);
      for (int i = 0; i < 2; ++i) { cudaEventDestroy(q.copied[i]); cudaEventDestroy(q.consumed[i]); if (q.xbuf[i]) cudaFree(q.xbuf[i]); }
      cudaStreamDestroy(q.copy);
    }
    if (q.w2t) cudaFree(q.w2t);
    if (q.w1t) cudaFree(q.w1t);
    if (q.partial) cudaFree(q.partial);
  }
  if (h->h_scalars) cudaFreeHost(h->h_scalars);
  if (h->copy_stream) {
    cudaStreamSynchronize(h->copy_stream);
    for (int i = 0; i < vaeb_handle::ASYNC_BUFS; ++i) {
      if (h->a_stage[i]) cudaFree(h->a_stage[i]);
      if (h->a_stage_u8[i]) cudaFree(h->a_stage_u8[i]);
      cudaEventDestroy(h->a_copied[i]);
      cudaEventDestroy(h->a_consumed[i]);
    }
    if (h->h_async) cudaFreeHost(h->h_async);
    if (h->d_iota) cudaFree(h->d_iota);
    cudaStreamDestroy(h->copy_stream);
  }
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return VAEB_OK;
}

int vaeb_set_stream(vaeb_handle* h, void* cuda_stream) {
  VAEB_REQUIRE(h, "null handle");
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return VAEB_OK;
}

int vaeb_synchronize(vaeb_handle* h) {
  VAEB_REQUIRE(h, "null handle");
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  return VAEB_OK;
}

int vaeb_num_tensors(vaeb_handle* h, int32_t* n_tensors, int64_t* n_elements) {
  VAEB_REQUIRE(h, "null handle");
  if (n_tensors) *n_tensors = h->lay.n;
  if (n_elements) *n_elements = h->lay.total;
  return VAEB_OK;
}

int vaeb_tensor_shape(vaeb_handle* h, int32_t i, int32_t* rows, int32_t* cols) {
  VAEB_REQUIRE(h && i >= 0 && i < h->lay.n, "tensor index out of range");
  if (rows) *rows = h->lay.rows[i];
  if (cols) *cols = h->lay.cols[i];
  return VAEB_OK;
}

int vaeb_set_tensors(vaeb_handle* h, int32_t which, const float* const* tensors) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && tensors, "null argument");
  float* flat = flat_by_which(h, which);
  VAEB_REQUIRE(flat, "buffer not available for this estimator");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  invalidate_weight_mirrors(h);
  for (int t = 0; t < h->lay.n; ++t) {
    const size_t n = (size_t)h->lay.rows[t] * h->lay.cols[t];
    VAEB_CUDA(cudaMemcpyAsync(flat + h->lay.off[t], tensors[t], n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  }
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  // sampled full VB: a theta / zeta written here is the draw of the current step (the training state, see the header)
  if ((which == 10 || which == 11) && h->cfg.estimator == VAEB_EST_FVB_SAMPLED) h->steptc.theta_step = (long long)h->step;
  return VAEB_OK;
}

int vaeb_get_tensors(vaeb_handle* h, int32_t which, float* const* tensors) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && tensors, "null argument");
  float* flat = flat_by_which(h, which);
  VAEB_REQUIRE(flat, "buffer not available for this estimator");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  if ((which == 10 || which == 11) && h->cfg.estimator == VAEB_EST_FVB_SAMPLED && h->steptc.theta_step != (long long)h->step) {
    // sampled full VB: return the theta / zeta the next update uses -- the draw the step kernel would make for the
    // current step, made now and kept for it (an update through another path draws its own, the same bits)
    VAEB_LAUNCH(launch_sample_theta(h->stream, &h->launches, h->d_vmu, h->d_vsig, nullptr, h->cfg.seed, h->step,
                                    h->lay.total, h->d_theta, h->d_zeta));
    invalidate_weight_mirrors(h);
    h->steptc.theta_step = (long long)h->step;
  }
  for (int t = 0; t < h->lay.n; ++t) {
    const size_t n = (size_t)h->lay.rows[t] * h->lay.cols[t];
    VAEB_CUDA(cudaMemcpyAsync(tensors[t], flat + h->lay.off[t], n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  }
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  return VAEB_OK;
}

int vaeb_device_buffer(vaeb_handle* h, int32_t which, void** d_ptr, int64_t* n_elements) {
  VAEB_REQUIRE(h && d_ptr, "null argument");
  float* flat = flat_by_which(h, which);
  VAEB_REQUIRE(flat, "buffer not available for this estimator");
  *d_ptr = flat;
  if (n_elements) *n_elements = h->lay.padded;
  return VAEB_OK;
}

int vaeb_upload_data(vaeb_handle* h, const float* x, int64_t n_rows) {
  VAEB_REQUIRE(h && x && n_rows > 0, "null data or no rows");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  if (h->d_x) VAEB_CUDA(cudaFree(h->d_x));
  h->d_x = nullptr;
  const size_t bytes = (size_t)n_rows * h->D * sizeof(float);
  VAEB_CUDA(cudaMalloc((void**)&h->d_x, bytes));
  VAEB_CUDA(cudaMemcpy(h->d_x, x, bytes, cudaMemcpyHostToDevice));
  h->n_data = n_rows;
  if (h->tc.active) {
    TcState& t = h->tc;
    VAEB_TRY(tc_ensure(h, 1, 1));
    VAEB_TRY(grow_bytes(&t.data.xh, (size_t)n_rows * t.data.ldx * 2));
    if (t.ns == 2) VAEB_TRY(grow_bytes(&t.data.xl, (size_t)n_rows * t.data.ldx * 2));
    VAEB_LAUNCH(tc_split_matrix(h->stream, &h->launches, h->d_x, n_rows, h->D, h->D, t.data.xh, t.data.xl, t.data.ldx,
                                h->D));
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    t.key_rows = -1;
  }
  return VAEB_OK;
}

static int stage_eps_zeta(vaeb_handle* h, const float* eps, int64_t n_eps, const float** d_eps) {
  *d_eps = nullptr;
  if (eps) { VAEB_TRY(stage_in(h, &h->d_stage2, &h->stage2_cap, eps, n_eps)); *d_eps = h->d_stage2; }
  return VAEB_OK;
}

int vaeb_update(vaeb_handle* h, int64_t index, const float* eps, float* elbo_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && elbo_out, "null argument");
  if (!h->d_x) { vaeb_set_error("vaeb_update before vaeb_upload_data"); return VAEB_ESTATE; }
  VAEB_REQUIRE(index >= 0 && (index + 1) * (int64_t)h->M <= h->n_data, "batch index outside the resident data");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const float* d_eps;
  VAEB_TRY(stage_eps_zeta(h, eps, (int64_t)h->L * h->M * h->Z, &d_eps));
  const float* x = h->d_x + (size_t)index * h->M * h->D;
  const StepPath path = step_path(h, h->M);
  if (path != PER_LAYER)
    VAEB_TRY(run_single_launch(h, path, nullptr, nullptr, x, h->M, 1, d_eps, 0, nullptr));
  else
    VAEB_TRY(enqueue_update(h, x, h->M, d_eps, nullptr, 0, true));
  return read_scalars(h, 1, elbo_out);
}

int vaeb_update_host(vaeb_handle* h, const float* x, int64_t rows, const float* eps, float* elbo_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && x && elbo_out && rows > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x, rows * h->D));
  const float* d_eps;
  VAEB_TRY(stage_eps_zeta(h, eps, (int64_t)h->L * rows * h->Z, &d_eps));
  const StepPath path = step_path(h, (int)rows);
  if (path != PER_LAYER)
    VAEB_TRY(run_single_launch(h, path, nullptr, nullptr, h->d_stage, (int)rows, 1, d_eps, 0, nullptr));
  else
    VAEB_TRY(enqueue_update(h, h->d_stage, (int)rows, d_eps, nullptr, 0, true));
  return read_scalars(h, 1, elbo_out);
}

int vaeb_ae_train(vaeb_handle* h, int32_t kind, const int32_t* idx, int32_t n, float* out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && idx && out && n > 0, "null argument");
  VAEB_REQUIRE(kind == VAEB_AE_DEGENERATE || kind == VAEB_AE_VANILLA, "unknown AE kind");
  VAEB_REQUIRE(!(kind == VAEB_AE_VANILLA && h->cont), "the vanilla AE has sigmoid outputs only (vanilla-ae/ae.py:62-67)");
  VAEB_REQUIRE(h->L == 1 && !is_fvb(h) && h->world == 1, "AE baselines: L = 1, single GPU");
  VAEB_REQUIRE(h->lay.depth <= 1, "AE baselines have one hidden layer per side (degenerate-vae/ae.py:41-117)");
  if (!h->d_x) { vaeb_set_error("vaeb_ae_train before vaeb_upload_data"); return VAEB_ESTATE; }
  invalidate_weight_mirrors(h);
  for (int i = 0; i < n; ++i) VAEB_REQUIRE(idx[i] >= 0 && idx[i] < h->n_data, "row index outside the resident data");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z, rows = n;
  VAEB_TRY(ensure_ws(h, rows, rows, true));
  VAEB_TRY(grow(&h->d_stage, &h->stage_cap, (int64_t)rows * D));
  VAEB_TRY(grow(&h->d_stage2, &h->stage2_cap, (int64_t)rows));            // the row indices (as bits)
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  Workspace& s = h->ws;
  float* th = h->d_params;
  float* gr = h->d_grads;
  VAEB_CUDA(cudaMemcpyAsync(h->d_stage2, idx, (size_t)rows * sizeof(int), cudaMemcpyHostToDevice, st));
  VAEB_LAUNCH(launch_gather_rows(st, lc, h->d_x, (const int*)h->d_stage2, rows, D, h->d_stage));
  const float* x = h->d_stage;
  // forward (ae.py:48-58)
  VAEB_LAUNCH(launch_dense_act(st, lc, x, rows, D, T_(h, th, l.iW3), T_(h, th, l.ib3), H, 1, s.h_e));
  VAEB_LAUNCH(launch_dense_act(st, lc, s.h_e, rows, H, T_(h, th, l.iW4), T_(h, th, l.ib4), Z,
                               kind == VAEB_AE_VANILLA ? 1 : 0, s.z));
  VAEB_LAUNCH(launch_dense_act(st, lc, s.z, rows, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, 1, s.h_d));
  int tiles = 0;
  if (h->cont)     // otype 'cont': OutToProbs mean, OutToReal log-variance, indep_normal (ae.py:64-72) = the Gaussian head
    VAEB_LAUNCH(launch_dec2_loglik(st, lc, true, s.h_d, rows, H, T_(h, th, l.iW2), T_(h, th, l.ib2), T_(h, th, l.iW6),
                                   T_(h, th, l.ib6), D, x, 1, rows, 1.0f, s.da2, s.dlv, s.partial, &tiles));
  else
    VAEB_LAUNCH(launch_dec2_ae(st, lc, kind == VAEB_AE_VANILLA ? 1 : 0, s.h_d, rows, H, T_(h, th, l.iW2),
                               T_(h, th, l.ib2), D, x, s.da2, s.partial, &tiles));
  // backward of logjoint (T.grad inside AdaGrad.construct, infalg.py:156)
  VAEB_CUDA(cudaMemsetAsync(gr, 0, (size_t)(l.padded + 4) * sizeof(float), st));     // W5, b5 are not part of theta
  VAEB_LAUNCH(launch_wgrad(st, lc, s.h_d, rows, H, s.da2, D, T_(h, gr, l.iW2), T_(h, gr, l.ib2)));
  if (h->cont) VAEB_LAUNCH(launch_wgrad(st, lc, s.h_d, rows, H, s.dlv, D, T_(h, gr, l.iW6), T_(h, gr, l.ib6)));
  VAEB_LAUNCH(launch_dgrad_tanh(st, lc, s.da2, T_(h, th, l.iW2), h->cont ? s.dlv : nullptr,
                                h->cont ? T_(h, th, l.iW6) : nullptr, rows, D, H, s.h_d, s.da1));
  VAEB_LAUNCH(launch_wgrad(st, lc, s.z, rows, Z, s.da1, H, T_(h, gr, l.iW1), T_(h, gr, l.ib1)));
  if (kind == VAEB_AE_VANILLA) {   // through Z = tanh(.)
    VAEB_LAUNCH(launch_dgrad_tanh(st, lc, s.da1, T_(h, th, l.iW1), nullptr, nullptr, rows, H, Z, s.z, s.dmu));
  } else {                         // + d/dZ of ConstructNormalPrior([Z], 1.0) = -Z   (ae.py:77)
    VAEB_LAUNCH(launch_dgrad(st, lc, s.da1, T_(h, th, l.iW1), rows, H, Z, s.dmu));
    VAEB_LAUNCH(launch_axpy(st, lc, s.dmu, s.z, -1.0f, (int64_t)rows * Z));
  }
  VAEB_LAUNCH(launch_wgrad(st, lc, s.h_e, rows, H, s.dmu, Z, T_(h, gr, l.iW4), T_(h, gr, l.ib4)));
  VAEB_LAUNCH(launch_dgrad_tanh(st, lc, s.dmu, T_(h, th, l.iW4), nullptr, nullptr, rows, Z, H, s.h_e, s.da3));
  VAEB_LAUNCH(launch_wgrad(st, lc, x, rows, D, s.da3, H, T_(h, gr, l.iW3), T_(h, gr, l.ib3)));
  // reported value: loglik / n (ae.py:81) or se / n (vanilla-ae/ae.py:79); row_aux = 0: no latent term in it
  VAEB_CUDA(cudaMemsetAsync(s.row_aux, 0, (size_t)rows * sizeof(float), st));
  float* base = gr + l.padded;
  VAEB_LAUNCH(launch_finalize(st, lc, s.partial, tiles, s.row_aux, rows, 1, s.per_row, base,
                              kind == VAEB_AE_VANILLA ? -1.0f : 1.0f, nullptr, 0, (float)rows, h->d_scalars));
  // AdaGrad ascent with the weight prior -p/s2 folded in (mlp.py:87-91; infalg.py:157-162)
  VAEB_LAUNCH(launch_adagrad(st, lc, th, h->d_ada, gr, l.padded / 4, h->cfg.learning_rate, h->cfg.adagrad_eps,
                             h->cfg.prior_scale, 0.f, base, 1.0f, 1.0f, nullptr));
  h->grads_have_prior = false;
  return read_scalars(h, 1, out);
}

int vaeb_ae_forward(vaeb_handle* h, int32_t kind, int32_t what, const float* in, int64_t rows, float* out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && in && out && rows > 0, "null argument");
  VAEB_REQUIRE(kind == VAEB_AE_DEGENERATE || kind == VAEB_AE_VANILLA, "unknown AE kind");
  VAEB_REQUIRE(what >= 0 && what <= 2, "what: 0 reconstruct, 1 encode, 2 decode");
  VAEB_REQUIRE(h->lay.depth <= 1, "AE baselines have one hidden layer per side (degenerate-vae/ae.py:41-117)");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z, r = (int)rows;
  VAEB_TRY(ensure_ws(h, rows, rows, false));
  const int in_w = what == 2 ? Z : D, out_w = what == 1 ? Z : D;
  VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, in, rows * in_w));
  VAEB_TRY(grow(&h->d_out, &h->out_cap, rows * out_w));
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  Workspace& s = h->ws;
  const float* th = h->d_params;
  const float* z = h->d_stage;
  if (what != 2) {
    VAEB_LAUNCH(launch_dense_act(st, lc, h->d_stage, r, D, T_(h, th, l.iW3), T_(h, th, l.ib3), H, 1, s.h_e));
    VAEB_LAUNCH(launch_dense_act(st, lc, s.h_e, r, H, T_(h, th, l.iW4), T_(h, th, l.ib4), Z,
                                 kind == VAEB_AE_VANILLA ? 1 : 0, what == 1 ? h->d_out : s.z));
    z = s.z;
  }
  if (what != 1) {
    VAEB_LAUNCH(launch_dense_act(st, lc, z, r, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, 1, s.h_d));
    VAEB_LAUNCH(launch_dense_act(st, lc, s.h_d, r, H, T_(h, th, l.iW2), T_(h, th, l.ib2), D, 2, h->d_out));   // OutToProbs
  }
  VAEB_CUDA(cudaMemcpyAsync(out, h->d_out, (size_t)rows * out_w * sizeof(float), cudaMemcpyDeviceToHost, st));
  VAEB_CUDA(cudaStreamSynchronize(st));
  return VAEB_OK;
}

int vaeb_set_hidden_activation(vaeb_handle* h, int32_t act) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h, "null handle");
  VAEB_REQUIRE(act == VAEB_ACT_TANH || act == VAEB_ACT_SIGMOID || act == VAEB_ACT_RELU, "unknown activation");
  VAEB_REQUIRE(act == VAEB_ACT_TANH || (h->cfg.precision == VAEB_PREC_FP32 && !is_fvb(h) && h->world == 1),
               "sigmoid / ReLU hidden layers: fp32 per-layer kernels, L^A / L^B estimators, one GPU");
  h->hidden_act = act;
  invalidate_weight_mirrors(h);
  return VAEB_OK;
}

int vaeb_set_optimizer(vaeb_handle* h, int32_t optimizer, float rho) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h, "null handle");
  VAEB_REQUIRE(optimizer == VAEB_OPT_ADAGRAD || optimizer == VAEB_OPT_ADADELTA, "unknown optimizer");
  VAEB_REQUIRE(optimizer == VAEB_OPT_ADAGRAD || !is_fvb(h), "AdaDelta is not wired to the full-VB estimators");
  VAEB_REQUIRE(optimizer == VAEB_OPT_ADAGRAD || (rho > 0.f && rho < 1.f), "rho must lie in (0, 1)");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const size_t nb = (size_t)(h->lay.padded + 4) * sizeof(float);
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  if (optimizer == VAEB_OPT_ADADELTA && !h->d_ada2) VAEB_CUDA(cudaMalloc((void**)&h->d_ada2, nb));
  if (h->d_ada2) VAEB_CUDA(cudaMemsetAsync(h->d_ada2, 0, nb, h->stream));
  VAEB_CUDA(cudaMemsetAsync(h->d_ada, 0, nb, h->stream));
  h->optimizer = optimizer;
  h->rho = rho;
  return VAEB_OK;
}

int vaeb_set_adam(vaeb_handle* h, float beta1, float beta2, float eps) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h, "null handle");
  VAEB_REQUIRE(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f, "beta1 and beta2 must lie in [0, 1)");
  VAEB_REQUIRE(eps > 0.f && std::isfinite(eps), "eps must be positive and finite");
  VAEB_REQUIRE(!is_fvb(h), "Adam is not wired to the full-VB estimators");
  if (h->tc.p2p_buf) {
    vaeb_set_error("vaeb_set_adam after vaeb_comm_p2p_export: the peers mapped an accumulator buffer without room for v");
    return VAEB_ESTATE;
  }
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const int64_t n = h->lay.padded + 4;
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  if (!h->d_adam_v) {               // m and v in one allocation: the accumulator's IPC handle maps both
    float* mv = nullptr;
    VAEB_CUDA(cudaMalloc((void**)&mv, (size_t)2 * n * sizeof(float)));
    VAEB_CUDA(cudaFree(h->d_ada));
    h->d_ada = mv;
    h->d_adam_v = mv + n;
  }
  VAEB_CUDA(cudaMemsetAsync(h->d_ada, 0, (size_t)2 * n * sizeof(float), h->stream));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  h->optimizer = VAEB_OPT_ADAM;
  h->adam_b1 = beta1; h->adam_b2 = beta2; h->adam_eps = eps;
  h->adam_t = 0;
  return VAEB_OK;
}

int vaeb_adam_step(vaeb_handle* h, int64_t* t) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));       // the copied-but-unlaunched updates count
  VAEB_REQUIRE(h && t, "null argument");
  *t = h->adam_t;
  return VAEB_OK;
}

int vaeb_set_adam_step(vaeb_handle* h, int64_t t) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && t >= 0, "the Adam step must be non-negative");
  h->adam_t = t;
  return VAEB_OK;
}

int vaeb_set_kl_weight(vaeb_handle* h, float beta, int64_t warmup_updates) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));      // updates enqueued before the call keep the old weights
  VAEB_REQUIRE(h, "null handle");
  VAEB_REQUIRE(std::isfinite(beta) && beta >= 0.f, "the KL weight must be finite and non-negative");
  VAEB_REQUIRE(warmup_updates >= 0, "the KL warm-up must be non-negative");
  VAEB_REQUIRE(!is_fvb(h), "the KL weight is not wired to the full-VB estimators");
  h->kl_beta = beta;
  h->kl_warmup = warmup_updates;
  h->kl_t = 0;
  return VAEB_OK;
}

int vaeb_kl_step(vaeb_handle* h, int64_t* t) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));       // the copied-but-unlaunched updates count
  VAEB_REQUIRE(h && t, "null argument");
  *t = h->kl_t;
  return VAEB_OK;
}

int vaeb_set_kl_step(vaeb_handle* h, int64_t t) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && t >= 0, "the KL step must be non-negative");
  h->kl_t = t;
  return VAEB_OK;
}

// Launches the minibatches copied into the current group buffer: ONE launch of a single-launch step kernel for up to
// ASYNC_GROUP updates (per-layer kernels otherwise), then the readback of their bounds.
static int async_flush(vaeb_handle* h) {
  if (h->a_pending == 0) return VAEB_OK;
  const int g = h->a_group, n = h->a_pending;
  const int rows = (int)h->a_rows;
  const int slot0 = h->a_outstanding - n;
  VAEB_CUDA(cudaEventRecord(h->a_copied[g], h->copy_stream));
  VAEB_CUDA(cudaStreamWaitEvent(h->stream, h->a_copied[g], 0));
  const StepPath path = step_path(h, rows);
  if (path != PER_LAYER) {
    VAEB_TRY(run_single_launch(h, path, nullptr, h->d_iota, h->a_stage[g], rows, n, nullptr, slot0, nullptr));
  } else {
    for (int i = 0; i < n; ++i)
      VAEB_TRY(enqueue_update(h, h->a_stage[g] + (size_t)i * rows * h->D, rows, nullptr, nullptr, slot0 + i, true));
  }
  VAEB_CUDA(cudaEventRecord(h->a_consumed[g], h->stream));
  VAEB_CUDA(cudaMemcpyAsync(h->h_async + slot0, h->d_scalars + slot0, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost,
                            h->stream));
  h->a_used[g] = true;
  h->a_pending = 0;
  h->a_group = (g + 1) % vaeb_handle::ASYNC_BUFS;
  return VAEB_OK;
}

// x: PINNED host minibatch, fp32 (x_u8 == nullptr) or bytes (x = (float)x_u8 * scale, expanded on the device)
static int host_async_submit(vaeb_handle* h, const float* x, const uint8_t* x_u8, float scale, int64_t rows) {
  VAEB_REQUIRE(h && (x || x_u8) && rows > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  {
    // pageable memory would turn the copy into a staged, synchronous one and serialise the pipeline silently
    cudaPointerAttributes pa{};
    const cudaError_t pe = cudaPointerGetAttributes(&pa, x ? (const void*)x : (const void*)x_u8);
    if (pe != cudaSuccess) (void)cudaGetLastError();
    VAEB_REQUIRE(pe == cudaSuccess && (pa.type == cudaMemoryTypeHost || pa.type == cudaMemoryTypeManaged),
                 "vaeb_update_host_async needs PINNED host memory (cudaHostAlloc / cudaHostRegister / "
                 "torch pin_memory); use vaeb_update_host for pageable buffers");
  }
  constexpr int NB = vaeb_handle::ASYNC_BUFS, GROUP = vaeb_handle::ASYNC_GROUP;
  constexpr int MAX_OUT = 8192;
  const int64_t n = rows * h->D;
  if (!h->copy_stream) {
    VAEB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < NB; ++i) {
      VAEB_CUDA(cudaEventCreateWithFlags(&h->a_copied[i], cudaEventDisableTiming));
      VAEB_CUDA(cudaEventCreateWithFlags(&h->a_consumed[i], cudaEventDisableTiming));
    }
    VAEB_CUDA(cudaMallocHost((void**)&h->h_async, (size_t)MAX_OUT * sizeof(float)));
    h->h_async_cap = MAX_OUT;
    const int iota[GROUP] = {0, 1, 2, 3};
    VAEB_CUDA(cudaMalloc((void**)&h->d_iota, sizeof(iota)));
    VAEB_CUDA(cudaMemcpy(h->d_iota, iota, sizeof(iota), cudaMemcpyHostToDevice));
  }
  VAEB_REQUIRE(h->a_outstanding < h->h_async_cap, "too many uncollected updates: call vaeb_collect");
  if (h->a_pending > 0 && rows != h->a_rows) VAEB_TRY(async_flush(h));     // a group holds minibatches of one size
  if (n > h->a_stage_cap) {
    VAEB_TRY(async_flush(h));
    VAEB_CUDA(cudaStreamSynchronize(h->copy_stream));
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < NB; ++i) {
      if (h->a_stage[i]) VAEB_CUDA(cudaFree(h->a_stage[i]));
      h->a_stage[i] = nullptr;
      VAEB_CUDA(cudaMalloc((void**)&h->a_stage[i], (size_t)GROUP * n * sizeof(float)));
      h->a_used[i] = false;
    }
    h->a_stage_cap = n;
  }
  if (x_u8 && n > h->a_stage_u8_cap) {
    VAEB_TRY(async_flush(h));
    VAEB_CUDA(cudaStreamSynchronize(h->copy_stream));
    for (int i = 0; i < NB; ++i) {
      if (h->a_stage_u8[i]) VAEB_CUDA(cudaFree(h->a_stage_u8[i]));
      h->a_stage_u8[i] = nullptr;
      VAEB_CUDA(cudaMalloc((void**)&h->a_stage_u8[i], (size_t)GROUP * n));
    }
    h->a_stage_u8_cap = n;
  }
  VAEB_TRY(ensure_scalars(h, h->h_async_cap));
  const int g = h->a_group;
  // copy stream: before the first copy into a group buffer, wait for the kernel that last read it
  if (h->a_pending == 0 && h->a_used[g]) VAEB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->a_consumed[g], 0));
  float* dst = h->a_stage[g] + (size_t)h->a_pending * n;
  if (x_u8) {
    // a quarter of the PCIe bytes; the expansion to fp32 follows the copy on the copy stream (12.8 MB in, 51 MB out for
    // 16384 MNIST rows: ~15 us of HBM time next to the previous update's kernels)
    uint8_t* d8 = h->a_stage_u8[g] + (size_t)h->a_pending * n;
    VAEB_CUDA(cudaMemcpyAsync(d8, x_u8, (size_t)n, cudaMemcpyHostToDevice, h->copy_stream));
    VAEB_CUDA(launch_expand_u8(h->copy_stream, d8, dst, n, scale));
    ++h->launches;
  } else {
    VAEB_CUDA(cudaMemcpyAsync(dst, x, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream));
  }
  h->a_rows = rows;
  ++h->a_pending;
  ++h->a_outstanding;
  if (h->a_pending == GROUP) VAEB_TRY(async_flush(h));
  return VAEB_OK;
}

int vaeb_update_host_async(vaeb_handle* h, const float* x, int64_t rows) {
  VAEB_REQUIRE(h && x && rows > 0, "null argument");
  return host_async_submit(h, x, nullptr, 1.f, rows);
}

int vaeb_update_host_async_u8(vaeb_handle* h, const uint8_t* x, int64_t rows, float scale) {
  VAEB_REQUIRE(h && x && rows > 0, "null argument");
  VAEB_REQUIRE(scale > 0.f && std::isfinite(scale), "scale must be positive and finite");
  return host_async_submit(h, nullptr, x, scale, rows);
}

int vaeb_collect(vaeb_handle* h, int32_t* n_inout, float* elbo_out) {
  VAEB_REQUIRE(h && n_inout && elbo_out, "null argument");
  VAEB_REQUIRE(*n_inout >= h->a_outstanding, "elbo_out is smaller than the number of outstanding updates");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_TRY(async_flush(h));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  std::memcpy(elbo_out, h->h_async, (size_t)h->a_outstanding * sizeof(float));
  *n_inout = h->a_outstanding;
  h->a_outstanding = 0;
  return VAEB_OK;
}

int vaeb_update_many(vaeb_handle* h, const int32_t* batch_order, int32_t n, float* elbo_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && batch_order && elbo_out && n > 0, "null argument");
  if (!h->d_x) { vaeb_set_error("vaeb_update_many before vaeb_upload_data"); return VAEB_ESTATE; }
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_TRY(ensure_scalars(h, n));
  for (int i = 0; i < n; ++i) {
    const int64_t index = batch_order[i];
    VAEB_REQUIRE(index >= 0 && (index + 1) * (int64_t)h->M <= h->n_data, "batch index outside the resident data");
  }
  const StepPath path = step_path(h, h->M);
  if (path != PER_LAYER) {
    VAEB_TRY(run_single_launch(h, path, batch_order, nullptr, nullptr, h->M, n, nullptr, 0, nullptr));
    return read_scalars(h, n, elbo_out);
  }
  for (int i = 0; i < n; ++i) {
    const int64_t index = batch_order[i];
    VAEB_TRY(enqueue_update(h, h->d_x + (size_t)index * h->M * h->D, h->M, nullptr, nullptr, i, true));
  }
  return read_scalars(h, n, elbo_out);
}

int vaeb_gradients(vaeb_handle* h, const float* x, int64_t rows, int64_t index, const float* eps, const float* zeta,
                   float* sgvb_out, float* per_row_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && rows > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const float* d_x;
  if (x) {
    VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x, rows * h->D));
    d_x = h->d_stage;
  } else {
    if (!h->d_x) { vaeb_set_error("vaeb_gradients(x=NULL) before vaeb_upload_data"); return VAEB_ESTATE; }
    VAEB_REQUIRE(index >= 0 && index * (int64_t)h->M + rows <= h->n_data, "rows outside the resident data");
    d_x = h->d_x + (size_t)index * h->M * h->D;
  }
  const float* d_eps;
  VAEB_TRY(stage_eps_zeta(h, eps, (int64_t)h->L * rows * h->Z, &d_eps));
  const float* d_zeta = nullptr;
  if (zeta) {
    // the flat zeta (tightly packed, reference tensor order) is staged in d_out
    VAEB_TRY(grow(&h->d_out, &h->out_cap, h->lay.padded));
    VAEB_CUDA(cudaMemcpyAsync(h->d_out, zeta, (size_t)h->lay.total * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    d_zeta = h->d_out;
  }
  VAEB_TRY(enqueue_update(h, d_x, (int)rows, d_eps, d_zeta, 0, false));
  // slot 0 holds base/Mg (non-FVB: written by finalize when !apply) or the SGVB (FVB)
  float v = 0.f;
  VAEB_TRY(read_scalars(h, 1, &v));
  if (sgvb_out) {
    if (is_fvb(h)) *sgvb_out = v;
    else if (h->cfg.variant == VAEB_VARIANT_FULLBAYES) *sgvb_out = v;          // the mean objective
    else *sgvb_out = v * (float)rows * (float)h->world;                       // back to the sum
  }
  if (per_row_out) {
    VAEB_CUDA(cudaMemcpy(per_row_out, h->ws.per_row, (size_t)rows * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return VAEB_OK;
}

int vaeb_apply_update(vaeb_handle* h) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h, "null handle");
  VAEB_REQUIRE(!is_fvb(h), "vaeb_apply_update: use vaeb_update for the full-VB estimators");
  VAEB_REQUIRE(h->optimizer != VAEB_OPT_ADAM, "vaeb_apply_update applies the Adagrad rule: Adam handles use vaeb_update*");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES;
  const float prior = (fb || h->grads_have_prior) ? 0.f : h->cfg.prior_scale;
  invalidate_weight_mirrors(h);
  VAEB_LAUNCH(launch_adagrad(h->stream, &h->launches, h->d_params, h->d_ada, h->d_grads, h->lay.padded / 4,
                             h->cfg.learning_rate, h->cfg.adagrad_eps, prior,
                             fb ? h->cfg.learning_rate * 1e-6f : 0.f, h->d_grads + h->lay.padded, 1.f, 1.f, nullptr));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  return VAEB_OK;
}

// vaeb_validate / vaeb_validate_terms: the bound of x[n,D] with the current parameters; loglik_out / aux_out (both or
// neither, host float[n]) receive the two terms of every per-row bound.
static int validate_rows(vaeb_handle* h, const float* x, int64_t n, const float* eps, float* sgvb_out, float* per_row_out,
                         float* loglik_out, float* aux_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && x && sgvb_out && n > 0, "null argument");
  VAEB_REQUIRE(n * (int64_t)h->L < (int64_t)1 << 31, "too many rows for one validate call");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const int L = h->L;
  VAEB_TRY(ensure_ws(h, n, n * L, false));
  VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x, n * h->D));
  const float* d_eps;
  VAEB_TRY(stage_eps_zeta(h, eps, (int64_t)L * n * h->Z, &d_eps));
  // validate shares the eps stream with update in the reference (VAEB.py:158); here it
  // draws from its own Philox stream keyed by the same step counter
  EpsSource src{d_eps, h->cfg.seed, VAEB_STREAM_EVAL, h->step, 0};
  const float* theta = h->d_params;
  float mult = 1.f, div = 1.f;
  const float* tp = nullptr;
  if (is_fvb(h)) {
    if (h->cfg.estimator == VAEB_EST_FVB_SAMPLED) {
      VAEB_LAUNCH(launch_sample_theta(h->stream, &h->launches, h->d_vmu, h->d_vsig, nullptr, h->cfg.seed, h->step,
                                      h->lay.total, h->d_theta, h->d_zeta));
      theta = h->d_theta;
    }
    VAEB_LAUNCH(launch_theta_prior(h->stream, &h->launches, h->d_vmu, h->d_vsig, h->lay.total, h->d_tprior));
    mult = (float)n;                     // x.shape[0], VAEB.py:364
    tp = h->d_tprior;
  } else if (h->cfg.variant == VAEB_VARIANT_FULLBAYES) {
    div = (float)n;                      // T.mean, VAEBfullbayes.py:142
  }
  BoundOut bo{h->d_grads + h->lay.padded, mult, tp, VAEB_TP_BLOCKS, div, h->d_scalars};
  if (loglik_out) {
    VAEB_TRY(grow(&h->d_out, &h->out_cap, 2 * n));
    bo.loglik_rows = h->d_out;
    bo.aux_rows = h->d_out + n;
  }
  VAEB_TRY(forward_backward(h, theta, h->d_stage, (int)n, L, false, 1.f, 1.f, src, nullptr, bo));
  ++h->step;
  VAEB_TRY(read_scalars(h, 1, sgvb_out));
  if (per_row_out)
    VAEB_CUDA(cudaMemcpy(per_row_out, h->ws.per_row, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  if (loglik_out) {
    VAEB_CUDA(cudaMemcpy(loglik_out, bo.loglik_rows, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    VAEB_CUDA(cudaMemcpy(aux_out, bo.aux_rows, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return VAEB_OK;
}

int vaeb_validate(vaeb_handle* h, const float* x, int64_t n, const float* eps, float* sgvb_out, float* per_row_out) {
  return validate_rows(h, x, n, eps, sgvb_out, per_row_out, nullptr, nullptr);
}

int vaeb_validate_terms(vaeb_handle* h, const float* x, int64_t n, const float* eps, float* loglik_out, float* aux_out) {
  VAEB_REQUIRE(loglik_out && aux_out, "null argument");
  float sgvb = 0.f;
  return validate_rows(h, x, n, eps, &sgvb, nullptr, loglik_out, aux_out);
}

int vaeb_is_logpx(vaeb_handle* h, const float* x, int64_t n, int32_t L, const float* eps, int64_t row_offset,
                  float* logpx_out, float* logw_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && x && logpx_out && n > 0 && L > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  const bool tcp = is_tc_supported(h);
  // points per chunk: the fp32 path materialises every decoder row, the tensor-core path only per-point data
  const int64_t chunk_rows = (int64_t)1 << (tcp && logw_out ? 22 : 17);
  const int pc = tcp && !logw_out ? (int)std::min<int64_t>(n, 8192)
                                  : (int)std::max<int64_t>(1, std::min<int64_t>(n, chunk_rows / L));
  VAEB_REQUIRE((int64_t)pc * L < (int64_t)1 << 31, "L too large");
  VAEB_TRY(ensure_ws(h, pc, tcp && !logw_out ? pc : (int64_t)pc * L, false));
  VAEB_TRY(grow(&h->d_out, &h->out_cap, pc));
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  const float* th = h->d_params;
  if (tcp && !logw_out && !eps) {
    // Tensor-core estimator with Philox noise: host x in, host log p out, pipelined.  The points go through two
    // staging buffers: chunk i+1 is copied on a second stream while chunk i is encoded and sampled, so only the first
    // copy is exposed (31 MB of x for 10k points is ~3 ms of a 49 ms call; per GPU of an 8-way shard 14 % of the call).
    IsTcState& q = h->istc;
    if (!q.copy) {
      VAEB_CUDA(cudaStreamCreateWithFlags(&q.copy, cudaStreamNonBlocking));
      for (int i = 0; i < 2; ++i) {
        VAEB_CUDA(cudaEventCreateWithFlags(&q.copied[i], cudaEventDisableTiming));
        VAEB_CUDA(cudaEventCreateWithFlags(&q.consumed[i], cudaEventDisableTiming));
      }
    }
    // about four chunks per call, 512..8192 points each (a chunk of 512 points x 5000 samples is 20480 tiles: 138 per SM)
    int64_t pcp = ((n + 3) / 4 + 255) / 256 * 256;
    pcp = std::max<int64_t>(512, std::min<int64_t>(pcp, 8192));
    pcp = std::min<int64_t>(pcp, n);
    VAEB_REQUIRE(pcp * L < (int64_t)1 << 31, "L too large");
    VAEB_TRY(ensure_ws(h, pcp, pcp, false));
    VAEB_TRY(grow(&h->d_out, &h->out_cap, pcp));
    if (pcp * D > q.xbuf_cap) {
      VAEB_CUDA(cudaStreamSynchronize(st));
      VAEB_CUDA(cudaStreamSynchronize(q.copy));
      for (int i = 0; i < 2; ++i) {
        if (q.xbuf[i]) VAEB_CUDA(cudaFree(q.xbuf[i]));
        q.xbuf[i] = nullptr;
        VAEB_CUDA(cudaMalloc((void**)&q.xbuf[i], (size_t)pcp * D * sizeof(float)));
      }
      q.xbuf_cap = pcp * D;
    }
    const int64_t n_chunks = (n + pcp - 1) / pcp;
    auto copy_in = [&](int64_t k) -> int {
      const int64_t i0 = k * pcp, c = std::min<int64_t>(pcp, n - i0);
      if (k >= 2) VAEB_CUDA(cudaStreamWaitEvent(q.copy, q.consumed[k & 1], 0));     // the buffer's previous chunk was read
      VAEB_CUDA(cudaMemcpyAsync(q.xbuf[k & 1], x + i0 * D, (size_t)c * D * sizeof(float), cudaMemcpyHostToDevice, q.copy));
      VAEB_CUDA(cudaEventRecord(q.copied[k & 1], q.copy));
      return VAEB_OK;
    };
    // work queued on the handle's stream before this call may still read nothing of ours; order the copy stream after
    // nothing: the staging buffers belong to this path alone (their last readers were synchronised at the end of the
    // previous call)
    VAEB_TRY(copy_in(0));
    for (int64_t k = 0; k < n_chunks; ++k) {
      const int64_t i0 = k * pcp;
      const int c = (int)std::min<int64_t>(pcp, n - i0);
      const float* dx = q.xbuf[k & 1];
      VAEB_CUDA(cudaStreamWaitEvent(st, q.copied[k & 1], 0));
      EpsSource src{nullptr, h->cfg.seed, VAEB_STREAM_IS, 0u, row_offset + i0};
      Workspace& s = h->ws;
      VAEB_TRY(encoder_hidden(h, th, dx, c));
      VAEB_LAUNCH(launch_enc2(st, lc, s.h_e, c, H, T_(h, th, l.iW4), T_(h, th, l.ib4), T_(h, th, l.iW5),
                              T_(h, th, l.ib5), Z, 0, 0, src, s.mu, s.ls, s.eps, s.z, s.row_aux));
      VAEB_TRY(is_tc_run(h, dx, s.mu, s.ls, c, L, nullptr, row_offset + i0, h->d_out, nullptr));
      VAEB_CUDA(cudaEventRecord(q.consumed[k & 1], st));
      if (k + 1 < n_chunks) VAEB_TRY(copy_in(k + 1));       // the host stages the next chunk while this one runs
      VAEB_CUDA(cudaMemcpyAsync(logpx_out + i0, h->d_out, (size_t)c * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    VAEB_CUDA(cudaStreamSynchronize(st));
    return VAEB_OK;
  }
  std::vector<float> tmp;
  for (int64_t i0 = 0; i0 < n; i0 += pc) {
    const int c = (int)std::min<int64_t>(pc, n - i0);
    const int R = c * L;
    VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x + i0 * D, (int64_t)c * D));
    const float* d_eps = nullptr;
    if (eps) { VAEB_TRY(stage_in(h, &h->d_stage2, &h->stage2_cap, eps + i0 * L * Z, (int64_t)R * Z)); d_eps = h->d_stage2; }
    EpsSource src{d_eps, h->cfg.seed, VAEB_STREAM_IS, 0u, row_offset + i0};
    Workspace& s = h->ws;
    VAEB_TRY(encoder_hidden(h, th, h->d_stage, c));
    VAEB_LAUNCH(launch_enc2(st, lc, s.h_e, c, H, T_(h, th, l.iW4), T_(h, th, l.ib4), T_(h, th, l.iW5),
                            T_(h, th, l.ib5), Z, 0, 0, src, s.mu, s.ls, s.eps, s.z, s.row_aux));
    if (tcp) {
      // decoder + log-likelihood + logsumexp in ONE tcgen05 kernel (is_tc.cu); bf16 operands
      VAEB_TRY(is_tc_run(h, h->d_stage, s.mu, s.ls, c, L, d_eps, row_offset + i0, h->d_out, logw_out ? s.logw : nullptr));
      VAEB_CUDA(cudaMemcpyAsync(logpx_out + i0, h->d_out, (size_t)c * sizeof(float), cudaMemcpyDeviceToHost, st));
      if (logw_out)
        VAEB_CUDA(cudaMemcpyAsync(logw_out + i0 * L, s.logw, (size_t)R * sizeof(float), cudaMemcpyDeviceToHost, st));
      VAEB_CUDA(cudaStreamSynchronize(st));
      continue;
    }
    VAEB_LAUNCH(launch_is_sample(st, lc, s.mu, s.ls, c, L, Z, src, s.z, s.dec_aux));
    VAEB_LAUNCH(launch_dense_act(st, lc, s.z, R, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, h->hidden_act, s.h_d));
    int tiles = 0;
    VAEB_LAUNCH(launch_dec2_loglik(st, lc, h->cont, s.h_d, R, H, T_(h, th, l.iW2), T_(h, th, l.ib2),
                                   h->cont ? T_(h, th, l.iW6) : nullptr, h->cont ? T_(h, th, l.ib6) : nullptr, D,
                                   h->d_stage, L, c, 1.f, nullptr, nullptr, s.partial, &tiles, true));
    VAEB_LAUNCH(launch_is_reduce(st, lc, s.partial, tiles, s.dec_aux, c, L, s.logw, h->d_out));
    VAEB_CUDA(cudaMemcpyAsync(logpx_out + i0, h->d_out, (size_t)c * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (logw_out)
      VAEB_CUDA(cudaMemcpyAsync(logw_out + i0 * L, s.logw, (size_t)R * sizeof(float), cudaMemcpyDeviceToHost, st));
    VAEB_CUDA(cudaStreamSynchronize(st));
  }
  return VAEB_OK;
}

int vaeb_reconstruct(vaeb_handle* h, const float* x, int64_t n, int32_t n_samples, const float* eps, float* y_out,
                     float* lv_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && x && y_out && n > 0, "null argument");
  VAEB_REQUIRE(!h->cont || lv_out, "the Gaussian decoder also returns its log-variance output");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  VAEB_TRY(ensure_ws(h, n, n, false));
  VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x, n * D));
  const int ns = std::max(n_samples, 0);
  const float* d_eps = nullptr;
  if (eps && ns > 0) { VAEB_TRY(stage_in(h, &h->d_stage2, &h->stage2_cap, eps, (int64_t)ns * n * Z)); d_eps = h->d_stage2; }
  VAEB_TRY(grow(&h->d_out, &h->out_cap, 2 * n * D));
  float* d_y = h->d_out;
  float* d_lv = h->d_out + n * D;
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  const float* th = h->d_params;
  Workspace& s = h->ws;
  EpsSource src{d_eps, h->cfg.seed, VAEB_STREAM_RECON, h->step, 0};
  VAEB_TRY(encoder_hidden(h, th, h->d_stage, (int)n));
  VAEB_LAUNCH(launch_enc2(st, lc, s.h_e, (int)n, H, T_(h, th, l.iW4), T_(h, th, l.ib4), T_(h, th, l.iW5),
                          T_(h, th, l.ib5), Z, 0, 0, src, s.mu, s.ls, s.eps, s.z, s.row_aux));
  const float* W6 = h->cont ? T_(h, th, l.iW6) : nullptr;
  const float* b6 = h->cont ? T_(h, th, l.ib6) : nullptr;
  const int passes = std::max(ns, 1);
  for (int sidx = 0; sidx < passes; ++sidx) {
    const float* zin = s.mu;                                  // n_samples <= 0: decode mu (VAEB.py:269-270)
    if (ns > 0) {
      VAEB_LAUNCH(launch_recon_sample(st, lc, s.mu, s.ls, (int)n, Z, src, sidx, (int)n, s.z));
      zin = s.z;
    }
    VAEB_LAUNCH(launch_dense_act(st, lc, zin, (int)n, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, h->hidden_act, s.h_d));
    VAEB_LAUNCH(launch_dec2_recon(st, lc, h->cont, s.h_d, (int)n, H, T_(h, th, l.iW2), T_(h, th, l.ib2), W6, b6, D,
                                  d_y, d_lv, 1.0f / (float)passes, sidx == 0));
  }
  ++h->step;
  VAEB_CUDA(cudaMemcpyAsync(y_out, d_y, (size_t)n * D * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (h->cont)
    VAEB_CUDA(cudaMemcpyAsync(lv_out, d_lv, (size_t)n * D * sizeof(float), cudaMemcpyDeviceToHost, st));
  VAEB_CUDA(cudaStreamSynchronize(st));
  return VAEB_OK;
}

int vaeb_decode(vaeb_handle* h, const float* z, int64_t n, float* y_out, float* lv_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && z && y_out && n > 0, "null argument");
  VAEB_REQUIRE(!h->cont || lv_out, "the Gaussian decoder needs lv_out");
  VAEB_REQUIRE(n < (int64_t)1 << 24, "too many latent points for one decode call");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  VAEB_TRY(ensure_ws(h, n, n, false));
  VAEB_TRY(stage_in(h, &h->d_stage2, &h->stage2_cap, z, n * Z));
  VAEB_TRY(grow(&h->d_out, &h->out_cap, 2 * n * D));
  float* d_y = h->d_out;
  float* d_lv = h->d_out + n * D;
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  const float* th = h->d_params;
  Workspace& s = h->ws;
  VAEB_LAUNCH(launch_dense_act(st, lc, h->d_stage2, (int)n, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, h->hidden_act, s.h_d));
  VAEB_LAUNCH(launch_dec2_recon(st, lc, h->cont, s.h_d, (int)n, H, T_(h, th, l.iW2), T_(h, th, l.ib2),
                                h->cont ? T_(h, th, l.iW6) : nullptr, h->cont ? T_(h, th, l.ib6) : nullptr, D, d_y, d_lv,
                                1.0f, true));
  VAEB_CUDA(cudaMemcpyAsync(y_out, d_y, (size_t)n * D * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (h->cont)
    VAEB_CUDA(cudaMemcpyAsync(lv_out, d_lv, (size_t)n * D * sizeof(float), cudaMemcpyDeviceToHost, st));
  VAEB_CUDA(cudaStreamSynchronize(st));
  return VAEB_OK;
}

int vaeb_encode(vaeb_handle* h, const float* x, int64_t n, float* mu_out, float* logvar_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && x && mu_out && logvar_out && n > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  // rows per chunk: the encoder's workspace is [rows, H] per hidden layer
  const int pc = (int)std::min<int64_t>(n, (int64_t)1 << 15);
  VAEB_TRY(ensure_ws(h, pc, 1, false));
  cudaStream_t st = h->stream;
  const float* th = h->d_params;
  Workspace& s = h->ws;
  const EpsSource no_eps{nullptr, 0, 0, 0, 0};
  for (int64_t i0 = 0; i0 < n; i0 += pc) {
    const int c = (int)std::min<int64_t>(pc, n - i0);
    VAEB_TRY(stage_in(h, &h->d_stage, &h->stage_cap, x + i0 * D, (int64_t)c * D));
    VAEB_TRY(encoder_hidden(h, th, h->d_stage, c));
    // L = 0 and no row terms: the heads alone
    VAEB_LAUNCH(launch_enc2(st, &h->launches, s.h_e, c, H, T_(h, th, l.iW4), T_(h, th, l.ib4), T_(h, th, l.iW5),
                            T_(h, th, l.ib5), Z, 0, 0, no_eps, s.mu, s.ls, nullptr, nullptr, nullptr));
    VAEB_CUDA(cudaMemcpyAsync(mu_out + i0 * Z, s.mu, (size_t)c * Z * sizeof(float), cudaMemcpyDeviceToHost, st));
    VAEB_CUDA(cudaMemcpyAsync(logvar_out + i0 * Z, s.ls, (size_t)c * Z * sizeof(float), cudaMemcpyDeviceToHost, st));
  }
  VAEB_CUDA(cudaStreamSynchronize(st));
  return VAEB_OK;
}

int vaeb_sample(vaeb_handle* h, int64_t n, uint32_t step, int64_t row_offset, float* z_out, float* mean_out,
                float* lv_out, float* x_out) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));
  VAEB_REQUIRE(h && n > 0 && row_offset >= 0, "null argument or negative row_offset");
  VAEB_REQUIRE(h->cont || !lv_out, "lv_out: the Bernoulli decoder has no log-variance output");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  VAEB_REQUIRE(row_offset + n <= ((int64_t)1 << 58) / std::max(D, Z), "rows beyond the 2^58 elements of a Philox stream");
  const int pc = (int)std::min<int64_t>(n, (int64_t)1 << 16);   // rows per chunk
  VAEB_TRY(ensure_ws(h, 1, pc, false));
  VAEB_TRY(grow(&h->d_out, &h->out_cap, 3 * (int64_t)pc * D));
  float* d_y = h->d_out;
  float* d_lv = h->d_out + (int64_t)pc * D;
  float* d_x = h->d_out + 2 * (int64_t)pc * D;
  cudaStream_t st = h->stream;
  int64_t* lc = &h->launches;
  const float* th = h->d_params;
  Workspace& s = h->ws;
  for (int64_t i0 = 0; i0 < n; i0 += pc) {
    const int c = (int)std::min<int64_t>(pc, n - i0);
    const int64_t r0 = row_offset + i0;                       // global row of the chunk's first sample
    VAEB_LAUNCH(launch_philox_fill(st, lc, h->cfg.seed, VAEB_STREAM_SAMPLE, step, 0u, r0 * Z, (int64_t)c * Z, s.z));
    VAEB_LAUNCH(launch_dense_act(st, lc, s.z, c, Z, T_(h, th, l.iW1), T_(h, th, l.ib1), H, h->hidden_act, s.h_d));
    VAEB_LAUNCH(launch_dec2_recon(st, lc, h->cont, s.h_d, c, H, T_(h, th, l.iW2), T_(h, th, l.ib2),
                                  h->cont ? T_(h, th, l.iW6) : nullptr, h->cont ? T_(h, th, l.ib6) : nullptr, D, d_y, d_lv,
                                  1.0f, true));
    if (x_out) VAEB_LAUNCH(launch_sample_x(st, lc, d_y, h->cont ? d_lv : nullptr, c, D, h->cfg.seed, step, r0, d_x));
    const size_t bz = (size_t)c * Z * sizeof(float), bd = (size_t)c * D * sizeof(float);
    if (z_out) VAEB_CUDA(cudaMemcpyAsync(z_out + i0 * Z, s.z, bz, cudaMemcpyDeviceToHost, st));
    if (mean_out) VAEB_CUDA(cudaMemcpyAsync(mean_out + i0 * D, d_y, bd, cudaMemcpyDeviceToHost, st));
    if (lv_out) VAEB_CUDA(cudaMemcpyAsync(lv_out + i0 * D, d_lv, bd, cudaMemcpyDeviceToHost, st));
    if (x_out) VAEB_CUDA(cudaMemcpyAsync(x_out + i0 * D, d_x, bd, cudaMemcpyDeviceToHost, st));
  }
  VAEB_CUDA(cudaStreamSynchronize(st));
  return VAEB_OK;
}

int vaeb_mlp_forward(vaeb_handle* h, const float* x, int64_t n, int32_t n_layers, const int32_t* dims,
                     const float* const* W, const float* const* b, int32_t act_last, float* out) {
  VAEB_REQUIRE(h && x && dims && W && b && out && n > 0 && n_layers > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  int maxd = 0;
  int64_t wtot = 0;
  for (int i = 0; i <= n_layers; ++i) maxd = std::max(maxd, dims[i]);
  for (int i = 0; i < n_layers; ++i) wtot += (int64_t)dims[i] * dims[i + 1] + dims[i + 1];
  float *d_a = nullptr, *d_b = nullptr, *d_w = nullptr;
  VAEB_CUDA(cudaMalloc((void**)&d_a, (size_t)n * maxd * sizeof(float)));
  VAEB_CUDA(cudaMalloc((void**)&d_b, (size_t)n * maxd * sizeof(float)));
  VAEB_CUDA(cudaMalloc((void**)&d_w, (size_t)wtot * sizeof(float)));
  int rc = VAEB_OK;
  do {
    if (cudaMemcpyAsync(d_a, x, (size_t)n * dims[0] * sizeof(float), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) { rc = VAEB_ECUDA; break; }
    int64_t o = 0;
    float* cur = d_a; float* nxt = d_b;
    for (int i = 0; i < n_layers && rc == VAEB_OK; ++i) {
      const int64_t nw = (int64_t)dims[i] * dims[i + 1];
      cudaMemcpyAsync(d_w + o, W[i], (size_t)nw * sizeof(float), cudaMemcpyHostToDevice, h->stream);
      cudaMemcpyAsync(d_w + o + nw, b[i], (size_t)dims[i + 1] * sizeof(float), cudaMemcpyHostToDevice, h->stream);
      const int act = (i + 1 < n_layers) ? 1 : act_last;
      if (launch_dense_act(h->stream, &h->launches, cur, (int)n, dims[i], d_w + o, d_w + o + nw, dims[i + 1], act, nxt) != cudaSuccess) { rc = VAEB_ECUDA; break; }
      o += nw + dims[i + 1];
      std::swap(cur, nxt);
    }
    if (rc != VAEB_OK) break;
    if (cudaMemcpyAsync(out, cur, (size_t)n * dims[n_layers] * sizeof(float), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) { rc = VAEB_ECUDA; break; }
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) rc = VAEB_ECUDA;
  } while (0);
  if (rc != VAEB_OK) vaeb_set_error(std::string("vaeb_mlp_forward: ") + cudaGetErrorString(cudaGetLastError()));
  cudaFree(d_a); cudaFree(d_b); cudaFree(d_w);
  return rc;
}

int vaeb_philox_normal(vaeb_handle* h, int32_t stream, uint32_t step, uint32_t sample, int64_t first_elem, int64_t n,
                       float* out) {
  VAEB_REQUIRE(h && out && n > 0, "null argument");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_TRY(grow(&h->d_out, &h->out_cap, n));
  VAEB_LAUNCH(launch_philox_fill(h->stream, &h->launches, h->cfg.seed, (uint32_t)stream, step, sample, first_elem, n,
                                 h->d_out));
  VAEB_CUDA(cudaMemcpyAsync(out, h->d_out, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  return VAEB_OK;
}

int vaeb_set_step_counter(vaeb_handle* h, uint32_t step) {
  VAEB_REQUIRE(h, "null handle");
  h->step = step;
  return VAEB_OK;
}

int vaeb_step_counter(vaeb_handle* h, uint32_t* step) {
  if (h && h->a_pending) VAEB_TRY(async_flush(h));     // streaming updates advance the counter when they are launched
  VAEB_REQUIRE(h && step, "null argument");
  *step = h->step;
  return VAEB_OK;
}

int vaeb_comm_unique_id(const char* nccl_library, uint8_t id_out[128]) {
  VAEB_REQUIRE(id_out, "null argument");
  static NcclApi api;
  VAEB_TRY(load_nccl(api, nccl_library));
  NcclId id;
  std::memset(&id, 0, sizeof(id));
  const int r = api.GetUniqueId(&id);
  if (r != 0) { vaeb_set_error(std::string("ncclGetUniqueId: ") + (api.GetErrorString ? api.GetErrorString(r) : "?")); return VAEB_ENCCL; }
  std::memcpy(id_out, &id, 128);
  return VAEB_OK;
}

int vaeb_comm_attach(vaeb_handle* h, const char* nccl_library, const uint8_t id[128], int32_t rank,
                     int32_t world_size) {
  VAEB_REQUIRE(h && id && world_size >= 1 && rank >= 0 && rank < world_size, "bad communicator arguments");
  VAEB_REQUIRE(!is_fvb(h), "full-VB estimators are single-GPU (replicas only)");
  VAEB_REQUIRE(h->lay.depth <= 1, "deeper encoders are single-GPU");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_TRY(load_nccl(h->nccl, nccl_library));
  NcclId nid;
  std::memcpy(&nid, id, 128);
  const int r = h->nccl.CommInitRank(&h->comm, world_size, nid, rank);
  if (r != 0) {
    vaeb_set_error(std::string("ncclCommInitRank: ") + (h->nccl.GetErrorString ? h->nccl.GetErrorString(r) : "?"));
    return VAEB_ENCCL;
  }
  h->rank = rank;
  h->world = world_size;
  return VAEB_OK;
}

static void p2p_release(vaeb_handle* h) {
  TcState& t = h->tc;
  for (int i = 0; i < t.p2p_n_opened; ++i) cudaIpcCloseMemHandle(t.p2p_opened[i]);
  t.p2p_n_opened = 0;
  if (t.p2p_buf) cudaFree(t.p2p_buf);
  t.p2p_buf = nullptr;
  t.p2p_ready = false;
}

int vaeb_comm_p2p_export(vaeb_handle* h, uint8_t handles_out[192]) {
  VAEB_REQUIRE(h && handles_out, "null argument");
  VAEB_REQUIRE(h->world > 1 && h->world <= TC_MAX_PEERS, "attach the communicator first (2..8 ranks)");
  VAEB_REQUIRE(!is_fvb(h), "full-VB estimators are single-GPU (replicas only)");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  VAEB_CUDA(cudaStreamSynchronize(h->stream));
  TcState& t = h->tc;
  p2p_release(h);
  const size_t bytes = (size_t)(h->lay.padded + 4) * sizeof(float) + 2 * TC_MAX_PEERS * sizeof(unsigned int);
  VAEB_CUDA(cudaMalloc((void**)&t.p2p_buf, bytes));
  VAEB_CUDA(cudaMemset(t.p2p_buf, 0, bytes));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t hh[3];
  VAEB_CUDA(cudaIpcGetMemHandle(&hh[0], t.p2p_buf));
  VAEB_CUDA(cudaIpcGetMemHandle(&hh[1], h->d_params));
  VAEB_CUDA(cudaIpcGetMemHandle(&hh[2], h->d_ada));
  std::memcpy(handles_out, hh, 192);
  return VAEB_OK;
}

int vaeb_comm_p2p_attach(vaeb_handle* h, const uint8_t* all_handles, int32_t world_size) {
  VAEB_REQUIRE(h && all_handles, "null argument");
  VAEB_REQUIRE(world_size == h->world && h->tc.p2p_buf, "vaeb_comm_p2p_export first, with the attached world size");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  TcState& t = h->tc;
  for (int r = 0; r < world_size; ++r) {
    float *buf = t.p2p_buf, *par = h->d_params, *ada = h->d_ada;
    if (r != h->rank) {
      cudaIpcMemHandle_t hh[3];
      std::memcpy(hh, all_handles + (size_t)r * 192, 192);
      void* p[3] = {nullptr, nullptr, nullptr};
      for (int q = 0; q < 3; ++q) {
        VAEB_CUDA(cudaIpcOpenMemHandle(&p[q], hh[q], cudaIpcMemLazyEnablePeerAccess));
        t.p2p_opened[t.p2p_n_opened++] = p[q];
      }
      buf = (float*)p[0]; par = (float*)p[1]; ada = (float*)p[2];
    }
    t.p2p_gsum[r] = buf;
    t.p2p_flags[r] = reinterpret_cast<unsigned int*>(buf + h->lay.padded + 4);
    t.p2p_params[r] = par;
    t.p2p_ada[r] = ada;
  }
  t.p2p_epoch = 0;
  t.p2p_ready = true;
  return VAEB_OK;
}

int vaeb_comm_detach(vaeb_handle* h) {
  VAEB_REQUIRE(h, "null handle");
  if (h->tc.p2p_buf || h->tc.p2p_n_opened) {
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    p2p_release(h);
  }
  if (h->comm) {
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    h->nccl.CommDestroy(h->comm);
    h->comm = nullptr;
  }
  h->rank = 0;
  h->world = 1;
  return VAEB_OK;
}

int vaeb_profile_update(vaeb_handle* h, int64_t index, int32_t iters, int32_t max_phases, int32_t* n_phases,
                        float* ms, double* flops, double* bytes, char* names) {
  VAEB_REQUIRE(h && n_phases && ms && flops && bytes && names && iters > 0 && max_phases > 0, "null argument");
  VAEB_REQUIRE(!is_fvb(h) && h->world == 1, "profiling covers the single-GPU LB/LA step");
  if (!h->d_x) { vaeb_set_error("vaeb_profile_update before vaeb_upload_data"); return VAEB_ESTATE; }
  VAEB_REQUIRE(index >= 0 && (index + 1) * (int64_t)h->M <= h->n_data, "batch index outside the resident data");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  // the repeated Adagrad launches must not disturb the model: back params/ADA up
  const size_t nb = (size_t)(h->lay.padded + 4) * sizeof(float);
  StateBackup backup(h, nb);              // restores params / ADA / step / launch count on every exit path
  VAEB_CUDA(backup.take());
  const StepPath path = step_path(h, h->M);
  // The single-launch kernels stamp %globaltimer at every phase boundary (CTA 0) into d_timing: ONE launch of `steps`
  // updates of minibatch `index`, its stamps read back into tm, ns per phase averaged over the last `iters` updates (the
  // first two are warm-up); kn / fl / by: the kernel's phase names, algorithmic flops and bytes.
  const int steps = iters + 2;
  auto stamped = [&](int np, long long*& d_timing, int& timing_cap, const char* const* kn, const double* fl,
                     const double* by) -> int {
    if (steps * (np + 1) > timing_cap) {
      if (d_timing) cudaFree(d_timing);
      d_timing = nullptr;
      VAEB_CUDA(cudaMalloc((void**)&d_timing, (size_t)steps * (np + 1) * sizeof(long long)));
      timing_cap = steps * (np + 1);
    }
    std::vector<long long> tm((size_t)steps * (np + 1));
    VAEB_CUDA(cudaMemsetAsync(d_timing, 0, tm.size() * sizeof(long long), h->stream));
    const std::vector<int32_t> order((size_t)steps, (int32_t)index);
    VAEB_TRY(run_single_launch(h, path, order.data(), nullptr, nullptr, h->M, steps, nullptr, 0, d_timing));
    VAEB_CUDA(cudaMemcpyAsync(tm.data(), d_timing, tm.size() * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    const int n = std::min(np, (int)max_phases);
    for (int i = 0; i < n; ++i) {
      double acc = 0;
      for (int s = 2; s < steps; ++s) acc += (double)(tm[(size_t)s * (np + 1) + i + 1] - tm[(size_t)s * (np + 1) + i]);
      ms[i] = (float)(acc / iters * 1e-6);
      flops[i] = fl[i]; bytes[i] = by[i];
      std::strncpy(names + 48 * i, kn[i], 47);
      names[48 * i + 47] = 0;
    }
    *n_phases = n;
    return VAEB_OK;
  };
  if (path == STEP_TC) {
    constexpr int NP = st2::N_PHASES;
    static const char* const kNames[NP] = {
        "P1 enc1 x.W3+tanh | W4,W5 update", "P2 heads+reparam+KL", "P3 dec1+dec2 h.W2+loglik+delta",
        "P4 dgrad (da.W2^T)*(1-h^2)", "P5 dz | W2 update | bound", "P6 W3 update | W1 update"};
    StepTcState& f = h->steptc;
    const double dM = h->M, dD = h->D, dH = h->H, dZ = h->Z;
    const double fl[NP] = {2 * dM * dD * dH + 4 * dM * dH * dZ, 4 * dM * dH * dZ, 2 * dM * dZ * dH + 2 * dM * dH * dD,
                           2 * dM * dH * dD, 2 * dM * dZ * dH + 2 * dM * dH * dD, 2 * dM * dD * dH + 4 * dM * dH * dZ + 2 * dM * dZ * dH};
    const double by[NP] = {4 * (dM * dD + dD * dH + dM * dH) + 40 * dH * dZ, 4 * (dM * dH + 2 * dH * dZ + 4 * dM * dZ),
                           4 * (dM * dZ + dZ * dH + dH * dD + 2 * dM * dD), 4 * (dM * dD + dH * dD + 2 * dM * dH),
                           4 * (dM * dH + dM * dD) + 24 * dH * dD, 4 * (dM * dD + dM * dH) + 20 * dD * dH + 20 * dZ * dH};
    return stamped(NP, f.d_timing, f.timing_cap, kNames, fl, by);
  }
  if (path == FUSED) {
    constexpr int NP = fs::N_PHASES;
    static const char* const kNames[NP] = {
        "P1 enc1 x.W3+tanh", "P2 heads+reparam+KL", "P3 dec1 z.W1+tanh", "P4 dec2 h.W2+loglik+delta",
        "P5 dgrad (da.W2^T)*(1-h^2)", "P6 W2,W1 wgrad+Adagrad | dz | bound", "P7 dh_e | W4,W5 wgrad+Adagrad",
        "P8 W3 wgrad+Adagrad"};
    FusedState& f = h->fused;
    const double dM = h->M, dD = h->D, dH = h->H, dZ = h->Z, c = h->cont ? 2.0 : 1.0;
    const double fl[NP] = {2 * dM * dD * dH, 4 * dM * dH * dZ, 2 * dM * dZ * dH, 2 * dM * dH * dD * c, 2 * dM * dH * dD * c,
                           2 * dM * dH * dD * c + 4 * dM * dZ * dH, 8 * dM * dH * dZ, 2 * dM * dD * dH};
    const double by[NP] = {4 * (dM * dD + dD * dH + dM * dH), 4 * (dM * dH + 2 * dH * dZ + 4 * dM * dZ),
                           4 * (dM * dZ + dZ * dH + dM * dH), 4 * (dM * dH + c * dH * dD + dM * dD + c * dM * dD),
                           4 * (c * dM * dD + c * dH * dD + 2 * dM * dH),
                           4 * (dM * dH + c * dM * dD + dM * dH + dM * dZ) + 16 * (c * dH * dD + dZ * dH),
                           4 * (2 * dM * dZ + 2 * dH * dZ + 2 * dM * dH) + 16 * 2 * dH * dZ,
                           4 * (dM * dD + dM * dH) + 16 * dD * dH};
    return stamped(NP, f.d_timing, f.timing_cap, kNames, fl, by);
  }
  PhaseProf prof;
  prof.iters = iters;
  VAEB_CUDA(cudaEventCreate(&prof.e0));
  VAEB_CUDA(cudaEventCreate(&prof.e1));
  g_prof = &prof;
  const int rc = enqueue_update(h, h->d_x + (size_t)index * h->M * h->D, h->M, nullptr, nullptr, 0, true);
  g_prof = nullptr;
  cudaEventDestroy(prof.e0); cudaEventDestroy(prof.e1);
  if (rc != VAEB_OK) return rc;
  const int n = std::min<int>((int)prof.ms.size(), max_phases);
  for (int i = 0; i < n; ++i) {
    ms[i] = prof.ms[i]; flops[i] = prof.flops[i]; bytes[i] = prof.bytes[i];
    std::strncpy(names + 48 * i, prof.names[i].c_str(), 47);
    names[48 * i + 47] = 0;
  }
  *n_phases = n;
  return VAEB_OK;
}

int vaeb_profile_optimizer(vaeb_handle* h, int32_t iters, float* ms_per_launch, double* bytes_per_launch) {
  VAEB_REQUIRE(h && ms_per_launch && bytes_per_launch && iters > 0, "null argument");
  VAEB_REQUIRE(!is_fvb(h), "vaeb_profile_optimizer covers the flat Adagrad pass of the LB/LA estimators");
  VAEB_CUDA(cudaSetDevice(h->cfg.device));
  const size_t nb = (size_t)(h->lay.padded + 4) * sizeof(float);
  StateBackup backup(h, nb);
  VAEB_CUDA(backup.take());
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  VAEB_CUDA(cudaEventCreate(&e0));
  if (cudaEventCreate(&e1) != cudaSuccess) { cudaEventDestroy(e0); VAEB_CUDA(cudaErrorUnknown); }
  const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES;
  cudaError_t ce = cudaSuccess;
  for (int i = -2; i < iters && ce == cudaSuccess; ++i) {          // two untimed launches first
    if (i == 0) ce = cudaEventRecord(e0, h->stream);
    if (ce == cudaSuccess)
      ce = launch_adagrad(h->stream, &h->launches, h->d_params, h->d_ada, h->d_grads, h->lay.padded / 4,
                          h->cfg.learning_rate, h->cfg.adagrad_eps, fb ? 0.f : h->cfg.prior_scale,
                          fb ? h->cfg.learning_rate * 1e-6f : 0.f, h->d_grads + h->lay.padded, 1.f, 1.f, nullptr);
  }
  if (ce == cudaSuccess) ce = cudaEventRecord(e1, h->stream);
  if (ce == cudaSuccess) ce = cudaEventSynchronize(e1);
  float ms = 0.f;
  if (ce == cudaSuccess) ce = cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  VAEB_CUDA(ce);
  *ms_per_launch = ms / (float)iters;
  *bytes_per_launch = 20.0 * (double)h->lay.total;                 // SURVEY 8d: read p, acc, g; write p, acc
  return VAEB_OK;
}

int vaeb_host_alloc(int64_t bytes, void** out) {
  VAEB_REQUIRE(out && bytes > 0, "null argument");
  VAEB_CUDA(cudaMallocHost(out, (size_t)bytes));
  return VAEB_OK;
}

int vaeb_host_free(void* p) {
  if (p) VAEB_CUDA(cudaFreeHost(p));
  return VAEB_OK;
}

int vaeb_launch_count(vaeb_handle* h, int64_t* n_launches) {
  VAEB_REQUIRE(h && n_launches, "null argument");
  *n_launches = h->launches;
  return VAEB_OK;
}

int vaeb_step_kernel(vaeb_handle* h, int64_t rows, int32_t* which) {
  VAEB_REQUIRE(h && which && rows > 0, "null argument");
  *which = step_path(h, (int)rows);
  return VAEB_OK;
}

}  // extern "C"
