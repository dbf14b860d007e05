// Importance-sampled log p(x) on the 5th-generation tensor cores (SURVEY.md 8a row a19, config c5).
//
// One persistent kernel, one CTA per SM.  A work tile is 128 samples of ONE test point:
//   z = mu + exp(.5 ls)*eps (Philox keyed by the global (point, sample, j)), written as a bf16 [z|1]
//       tile in the UMMA K-major SWIZZLE_128B layout                               -- producer warps
//   pre = [z|1].[W1^T|b1] : tcgen05.mma, 64 hidden units per pass into one of four small TMEM
//       accumulators (the bias rides along as contraction index Z)                 -- TMA + MMA warps
//   h = tanh(pre) -> bf16 -> k block of the A tile in shared memory: the decoder hidden layer never
//       exists in HBM                                                              -- producer warps
//   a = h.W2 : tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM), W2^T streamed through a TMA
//       ring of [NC n x 64 k] boxes, output swept in equal chunks of NC <= 160 columns (784 -> 5 x 160),
//       two TMEM accumulators so the epilogue of chunk c overlaps the MMAs of chunk c+1
//   log w = sum_d x_d a_d - softplus(a_d) + log p(z) - log q(z|x), per sample; then the tile's
//       (max, sum exp) pair -> partial[tile]                                       -- epilogue warps
// The hidden layer of tile i+1 is computed while the LAST output chunk of tile i runs: that chunk is the
// final reader of tile i's A blocks, each block is rewritten as soon as its MMAs retire (walk_items).
// A finishing kernel folds the per-tile pairs of a point into log p^(x) = logsumexp - log L.
// bf16 operands: the 1e-2 tier of the north star; the fp32 estimator (api.cu) stays the parity tier.
#include <cuda_bf16.h>
#include <cstdlib>

#include "common.cuh"
#include "philox.cuh"
#include "tc_common.cuh"

namespace istc {

constexpr int BM = 128, BK = 64, NC_MAX = 160, STAGES = 3;
constexpr int KB_MAX = 8;                       // hidden units padded to <= 512
constexpr int ZMAX = 20;                        // latent size; the bias rides along as contraction index Z
constexpr int ZG = 6;                           // groups of four contraction indices written per z row (24 >= Z + 1)
constexpr int DMAX = 1600;                      // output columns (Gaussian head: 2 x pixels, interleaved)
constexpr int PROD_WARPS = 8, EPI_WARPS = 16;     // epilogue: 4 TMEM lane quarters x (EPI_WARPS / 4) column slices
constexpr int THREADS = (4 + PROD_WARPS + EPI_WARPS) * 32;
constexpr int A_BLOCK = BM * 128;               // bytes of one 64-wide k block of the A tile
constexpr int B_STAGE = NC_MAX * 128;           // one ring stage: up to [128 rows x 64 k] bf16 (W2^T or W1^T box)
constexpr int TMEM_COLS = 512;
constexpr int W2T_PAD = 64;                     // W2^T row stride = KP + 64 elements: rows do not alias in L2
constexpr int ACC_STRIDE = 160;                 // two accumulators of the output sweep: columns [0,160), [160,320)
constexpr int MINI_COL0 = 320, MINI_BUFS = 3, MINI_N = 64;   // three 64-column accumulators of the hidden-layer GEMM
static_assert(MINI_COL0 + MINI_BUFS * MINI_N <= TMEM_COLS && 2 * ACC_STRIDE <= MINI_COL0 && NC_MAX <= ACC_STRIDE, "TMEM map");

struct Smem {                                   // offsets from a 1024-byte aligned base
  static constexpr int A = 0;                                // h tile, 8 k blocks, UMMA K-major SW128
  static constexpr int B = A + KB_MAX * A_BLOCK;             // TMA ring
  static constexpr int ZB = B + STAGES * B_STAGE;            // [z | 1] tile, [128 x 64] bf16, K-major SW128
  static constexpr int AUXP = ZB + BM * 128;                 // [128][ZG] partial prior/posterior terms
  static constexpr int AUX = AUXP + BM * ZG * 4;             // [3][128]
  static constexpr int XB = AUX + 3 * BM * 4;                // [DMAX] b2[col] then [DMAX] x[col] - 1/2; col >= D: (-30, -1/2)
  static constexpr int ROWSUM = XB + DMAX * 8;               // [EPI_WARPS / 4][128]
  static constexpr int RED = ROWSUM + (EPI_WARPS / 4) * BM * 4;   // [8]
  static constexpr int BARS = RED + 64;                      // mbarriers
  static constexpr int TOTAL = BARS + 512 + 1024;
};
static_assert(Smem::TOTAL <= 232448, "shared memory budget");

struct Params {
  int n_points, L, D, H, Z, KB;                 // KB = ceil(H / 64)
  int tiles_per_point, n_chunks, NC, zk;        // output chunks of NC columns (multiple of 16); zk = K=16 steps of [z|1]
  const float* x;                               // [n_points, D]
  const float* mu; const float* ls;             // [n_points, Z]
  const float* b2;                              // [D] output biases (Gaussian: b2 / b6 interleaved)
  int cont, Dx;                                 // Gaussian decoder; pixels per point (D = 2 Dx columns then)
  const float* eps_inj;                         // [n_points, L, Z] or nullptr
  uint64_t seed; int64_t row_offset;
  float2* partial;                              // [n_points * tiles_per_point] (max, sum exp)
  float* logw_out;                              // nullptr or [n_points * L]
};

__device__ __forceinline__ float tanh_approx(float v) {
  float r;
  asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
// ---- packed fp32 pairs (FADD2 / FMUL2 / FFMA2 of sm_100): the epilogue is issue- and MUFU-bound ----
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// Bernoulli log-likelihood of 8 accumulator columns of one row, two columns per instruction:
//   x a - softplus(a) = a (x - 1/2) - |a|/2 - ln(1 + e^-|a|),   a = acc + b2
// with m = -|a| log2(e), t = 2^m (one MUFU per element) and ln(1 + t) = t q(t) on the FMA pipe (q: degree-5
// fit on [0,1], |error| <= 1.5e-6).  bx: shared address of {b2[8]} ; xh: shared address of {x - 1/2 [8]}.
struct FoldConsts { uint64_t c0, c1, c2, c3, c4, c5, khalf; };
__device__ __forceinline__ FoldConsts fold_consts() {
  FoldConsts k;                                   // negated: the fold subtracts ln(1 + t)
  k.c0 = pk2(-0.9999016523361206f, -0.9999016523361206f);
  k.c1 = pk2(0.49787506461143494f, 0.49787506461143494f);
  k.c2 = pk2(-0.3176489472389221f, -0.3176489472389221f);
  k.c3 = pk2(0.19376075267791748f, 0.19376075267791748f);
  k.c4 = pk2(-0.08556976169347763f, -0.08556976169347763f);
  k.c5 = pk2(0.01833880878984928f, 0.01833880878984928f);
  k.khalf = pk2(0.34657359027997264f, 0.34657359027997264f);   // ln(2)/2: m * khalf = -|a|/2
  return k;
}
__device__ __forceinline__ void fold8(const float (&v)[8], uint32_t bx, uint32_t xh, const FoldConsts& k, uint64_t& acc) {
  uint64_t b[4], x[4];
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(b[0]), "=l"(b[1]) : "r"(bx));
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(b[2]), "=l"(b[3]) : "r"(bx + 16u));
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(x[0]), "=l"(x[1]) : "r"(xh));
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(x[2]), "=l"(x[3]) : "r"(xh + 16u));
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint64_t a2 = add2(pk2(v[2 * j], v[2 * j + 1]), b[j]);
    float a0, a1, t0, t1;
    upk2(a2, a0, a1);
    const float m0 = fabsf(a0) * -1.4426950408889634f, m1 = fabsf(a1) * -1.4426950408889634f;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(m0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(m1));
    const uint64_t t2 = pk2(t0, t1);
    uint64_t q = fma2(t2, k.c5, k.c4);
    q = fma2(q, t2, k.c3);
    q = fma2(q, t2, k.c2);
    q = fma2(q, t2, k.c1);
    q = fma2(q, t2, k.c0);
    acc = fma2(a2, x[j], acc);
    acc = fma2(pk2(m0, m1), k.khalf, acc);
    acc = fma2(t2, q, acc);
  }
}
// Gaussian decoder (VAEB.py:257-258, 304-307): the output columns are the interleaved head [W2|W6]' -- column 2d is the
// logit a_d of the mean, 2d + 1 the log-variance lv_d -- so 8 accumulator columns are 4 pixels:
//   -log(2 pi)/2 - lv/2 - (x - sigmoid(a))^2 e^{-lv} / 2.      bx: {b2, b6} interleaved; xh: x_d at both columns of a pair
// Padded pairs carry biases (-30, -log(2 pi)) and x = 0: mu = 0, e^{-lv} finite, the term vanishes.
__device__ __forceinline__ void fold8g(const float (&v)[8], uint32_t bx, uint32_t xh, float& acc) {
  float b[8], x[8];
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b[0]), "=f"(b[1]), "=f"(b[2]), "=f"(b[3]) : "r"(bx));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b[4]), "=f"(b[5]), "=f"(b[6]), "=f"(b[7]) : "r"(bx + 16u));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x[0]), "=f"(x[1]), "=f"(x[2]), "=f"(x[3]) : "r"(xh));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x[4]), "=f"(x[5]), "=f"(x[6]), "=f"(x[7]) : "r"(xh + 16u));
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float a = v[2 * j] + b[2 * j], lv = v[2 * j + 1] + b[2 * j + 1];
    float t, r, w;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-1.4426950408889634f * a));        // e^-a
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + t));                        // sigmoid(a)
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(w) : "f"(-1.4426950408889634f * lv));       // e^-lv
    const float d = x[2 * j] - r;
    acc += fmaf(-0.5f * d * d, w, fmaf(-0.5f, lv, -0.91893853320467274178f));
  }
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void named_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// ---- lean single-thread primitives on raw 32-bit shared addresses (the TMA and MMA issue loops are each ONE
// thread on the critical path of the whole CTA: every instruction in them costs ~8 cycles of latency) ----
__device__ __forceinline__ void bar_wait(uint32_t addr, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra WAIT_%=;\n\t}"
      ::"r"(addr), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void commit_to(uint32_t addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ uint64_t mk64(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO = 1024 B, version 1, SWIZZLE_128B

// The order in which one CTA consumes ring stages, shared by the TMA and the MMA thread.  A "pass" is the
// hidden-layer GEMM [z|1].W1^T for 64 hidden units of a tile (-> one k block of its A tile); a "w2" item is one
// k block of one output chunk.  The passes of tile i+1 are interleaved with the LAST output chunk of tile i:
// that chunk is the final reader of tile i's A blocks, so block kb can be rewritten as soon as its MMAs retire
// (a_free[kb]) and the conversion of tile i+1 hides behind the rest of the sweep.  Pass j >= MINI_BUFS re-uses
// the TMEM buffer of pass j-MINI_BUFS, whose conversion needs a_free[j-MINI_BUFS]: it is issued two k blocks later.
// FIRST / LAST are compile-time so the common (middle) chunk loop carries no per-item conditions.
template <bool FIRST, bool LAST, class R>
__device__ __forceinline__ void walk_chunk(const Params& p, uint32_t ti, int c, bool has_next, R& r) {
  r.chunk_begin();
  if (!LAST && r.template chunk_static<FIRST>(ti, c)) {
    // whole chunk issued by the unrolled fast path
  } else if (LAST && has_next) {
#pragma unroll 1
    for (int kb = 0; kb < p.KB; ++kb) {
      if (kb == 0) {
        for (int j = 0; j < MINI_BUFS && j < p.KB; ++j) r.pass(ti + 1, j);
      } else if (kb >= 2 && kb + MINI_BUFS - 2 < p.KB) {
        r.pass(ti + 1, kb + MINI_BUFS - 2);      // its TMEM buffer was read (a_free of pass - MINI_BUFS) two k blocks ago
      }
      r.template w2<FIRST, LAST>(ti, c, kb);
    }
  } else {
#pragma unroll 1
    for (int kb = 0; kb < p.KB; ++kb) r.template w2<FIRST, LAST>(ti, c, kb);
  }
  r.chunk_end();
}
template <class R>
__device__ __forceinline__ void walk_items(const Params& p, int n_tiles, R& r) {
  if ((int)blockIdx.x >= n_tiles) return;
  for (int j = 0; j < p.KB; ++j) r.pass(0u, j);
  const int last_c = p.n_chunks - 1;
  uint32_t ti = 0;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++ti) {
    const bool has_next = t + (int)gridDim.x < n_tiles;
    if (last_c == 0) { walk_chunk<true, true>(p, ti, 0, has_next, r); continue; }
    walk_chunk<true, false>(p, ti, 0, false, r);
#pragma unroll 1
    for (int c = 1; c < last_c; ++c) walk_chunk<false, false>(p, ti, c, false, r);
    walk_chunk<false, true>(p, ti, last_c, has_next, r);
  }
}

// barrier addresses (32-bit shared) used by the two issuing threads
struct BarAddrs {
  uint32_t b_full, b_empty, z_full, z_empty, mini_full, mini_empty, a_ready, a_free, acc_full, acc_empty;
};

struct TmaIssuer {
  const CUtensorMap* map_w2; const CUtensorMap* map_w1;
  BarAddrs bar;
  uint32_t ring;                 // shared address of the ring
  uint32_t w2_bytes; int NC;
  uint32_t stage = 0, parity = 0;
  // TWO issuing threads (lane 0 of warps 0 and 3) walk the same item sequence and issue alternate items: an item costs
  // its thread an mbarrier round trip (~0.3 us) whatever the bytes, and the fill rate scales with the number of
  // issuing threads (the TMA fill-rate probe, DESIGN.md 4.3: 30 / 59 / 118 GB/s per SM for 1 / 2 / 4 threads).
  uint32_t me = 0, turn = 0;
  __device__ __forceinline__ void load(const CUtensorMap* m, uint32_t bytes, int c0, int c1) {
    if (turn == me) {
      const uint32_t full = bar.b_full + 8u * stage;
      bar_wait(bar.b_empty + 8u * stage, parity ^ 1u);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"(bytes) : "memory");
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
          ::"r"(ring + stage * (uint32_t)B_STAGE), "l"(m), "r"(full), "r"(c0), "r"(c1)
          : "memory");
    }
    turn ^= 1u;
    if (++stage == STAGES) { stage = 0; parity ^= 1u; }
  }
  __device__ __forceinline__ void chunk_begin() {}
  __device__ __forceinline__ void chunk_end() {}
  template <bool FIRST>
  __device__ __forceinline__ bool chunk_static(uint32_t, int) { return false; }
  __device__ __forceinline__ void pass(uint32_t, int j) { load(map_w1, (uint32_t)MINI_N * 128u, 0, j * MINI_N); }
  template <bool FIRST, bool LAST>
  __device__ __forceinline__ void w2(uint32_t, int c, int kb) { load(map_w2, w2_bytes, kb * BK, c * NC); }
};

struct MmaIssuer {
  BarAddrs bar;
  uint32_t tmem_base, a_lo0, b_lo0, z_lo0, idesc, idesc_mini;
  int KB, zk;
  uint32_t stage = 0, parity = 0, acc_it = 0, mini_it = 0, d_acc = 0;
  __device__ __forceinline__ void advance() { if (++stage == STAGES) { stage = 0; parity ^= 1u; } }
  __device__ __forceinline__ void chunk_begin() {
    const uint32_t buf = acc_it & 1u;
    bar_wait(bar.acc_empty + 8u * buf, ((acc_it >> 1) & 1u) ^ 1u);
    tc::tc_fence_after();
    d_acc = tmem_base + buf * ACC_STRIDE;
  }
  __device__ __forceinline__ void chunk_end() {
    commit_to(bar.acc_full + 8u * (acc_it & 1u));
    ++acc_it;
  }
  __device__ __forceinline__ void pass(uint32_t tseq, int j) {
    if (j == 0) bar_wait(bar.z_full, tseq & 1u);
    const uint32_t mb = mini_it % MINI_BUFS;
    bar_wait(bar.b_full + 8u * stage, parity);
    bar_wait(bar.mini_empty + 8u * mb, ((mini_it / MINI_BUFS) & 1u) ^ 1u);
    tc::tc_fence_after();
    const uint32_t d = tmem_base + MINI_COL0 + mb * MINI_N;
    const uint32_t b_lo = b_lo0 + stage * (uint32_t)(B_STAGE >> 4);
    for (int k = 0; k < zk; ++k)
      tc::umma_bf16(d, mk64(z_lo0 + 2u * k, DESC_HI), mk64(b_lo + 2u * k, DESC_HI), idesc_mini, k ? 1u : 0u);
    commit_to(bar.b_empty + 8u * stage);
    commit_to(bar.mini_full + 8u * mb);
    if (j == KB - 1) commit_to(bar.z_empty);
    advance();
    ++mini_it;
  }
  // A whole chunk, fully unrolled, for the common case KB == 8: one instantiation per ring position the chunk can
  // start at, so that every descriptor / barrier address is base + constant.
  template <bool FIRST, int S0>
  __device__ __forceinline__ void chunk_unrolled(uint32_t tseq) {
#pragma unroll
    for (int kb = 0; kb < 8; ++kb) {
      constexpr int dummy = 0; (void)dummy;
      const uint32_t st = (uint32_t)((S0 + kb) % STAGES), wrap = (uint32_t)(((S0 + kb) / STAGES) & 1);
      if (FIRST) bar_wait(bar.a_ready + 8u * kb, tseq & 1u);
      bar_wait(bar.b_full + 8u * st, parity ^ wrap);
      tc::tc_fence_after();
      const uint32_t a_lo = a_lo0 + (uint32_t)kb * (uint32_t)(A_BLOCK >> 4);
      const uint32_t b_lo = b_lo0 + st * (uint32_t)(B_STAGE >> 4);
#pragma unroll
      for (int k = 0; k < BK / 16; ++k)
        tc::umma_bf16(d_acc, mk64(a_lo + 2u * k, DESC_HI), mk64(b_lo + 2u * k, DESC_HI), idesc, (kb | k) != 0 ? 1u : 0u);
      commit_to(bar.b_empty + 8u * st);
    }
    stage = (uint32_t)((S0 + 8) % STAGES);
    parity ^= (uint32_t)(((S0 + 8) / STAGES) & 1);
  }
  template <bool FIRST>
  __device__ __forceinline__ bool chunk_static(uint32_t tseq, int) {
    if (KB != 8) return false;
    static_assert(STAGES >= 2 && STAGES <= 4, "one unrolled chunk per starting stage");
    switch (stage) {
      case 0: chunk_unrolled<FIRST, 0>(tseq); break;
      case 1: chunk_unrolled<FIRST, 1>(tseq); break;
      case 2: chunk_unrolled<FIRST, 2 % STAGES>(tseq); break;
      default: chunk_unrolled<FIRST, 3 % STAGES>(tseq); break;
    }
    return true;
  }
  template <bool FIRST, bool LAST>
  __device__ __forceinline__ void w2(uint32_t tseq, int, int kb) {
    if (FIRST) bar_wait(bar.a_ready + 8u * kb, tseq & 1u);
    bar_wait(bar.b_full + 8u * stage, parity);
    tc::tc_fence_after();
    const uint32_t a_lo = a_lo0 + (uint32_t)kb * (uint32_t)(A_BLOCK >> 4);
    const uint32_t b_lo = b_lo0 + stage * (uint32_t)(B_STAGE >> 4);
#pragma unroll
    for (int k = 0; k < BK / 16; ++k)
      tc::umma_bf16(d_acc, mk64(a_lo + 2u * k, DESC_HI), mk64(b_lo + 2u * k, DESC_HI), idesc, (kb | k) != 0 ? 1u : 0u);
    commit_to(bar.b_empty + 8u * stage);
    if (LAST) commit_to(bar.a_free + 8u * kb);
    advance();
  }
};

// Roles (640 threads): warp 0 TMA, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-11 producers
// (z generation + TMEM -> tanh -> bf16 A tile conversion), warps 12-19 epilogue.
__global__ void __launch_bounds__(THREADS, 1)
is_tc_kernel(const __grid_constant__ CUtensorMap map_w2, const __grid_constant__ CUtensorMap map_w1, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + Smem::BARS);
  uint64_t* b_full = bars;                      // [STAGES]     TMA -> MMA
  uint64_t* b_empty = b_full + STAGES;          // [STAGES]     MMA -> TMA
  uint64_t* z_full = b_empty + STAGES;          //              producers -> MMA   ([z|1] tile written)
  uint64_t* z_empty = z_full + 1;               //              MMA -> producers   (all passes of the tile retired)
  uint64_t* mini_full = z_empty + 1;            // [MINI_BUFS]  MMA -> producers   (one pass of pre-activations in TMEM)
  uint64_t* mini_empty = mini_full + MINI_BUFS; // [MINI_BUFS]  producers -> MMA
  uint64_t* a_ready = mini_empty + MINI_BUFS;   // [KB_MAX]     producers -> MMA   (k block of the A tile written)
  uint64_t* a_free = a_ready + KB_MAX;          // [KB_MAX]     MMA -> producers   (last chunk done with the k block)
  uint64_t* acc_full = a_free + KB_MAX;         // [2]          MMA -> epilogue
  uint64_t* acc_empty = acc_full + 2;           // [2]          epilogue -> MMA
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);
  float* auxp = (float*)(smem + Smem::AUXP);
  float* aux_s = (float*)(smem + Smem::AUX);
  float* bb_s = (float*)(smem + Smem::XB);         // b2, padded with -30
  float* xh_s = bb_s + DMAX;                       // x - 1/2 of the tile's test point, padded with -1/2
  float* rowsum_s = (float*)(smem + Smem::ROWSUM);
  float* red_s = (float*)(smem + Smem::RED);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.n_points * p.tiles_per_point;

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&map_w2);
    tc::tma_prefetch_desc(&map_w1);
    for (int s = 0; s < STAGES; ++s) { tc::mbar_init(&b_full[s], 1); tc::mbar_init(&b_empty[s], 1); }
    tc::mbar_init(z_full, PROD_WARPS);
    tc::mbar_init(z_empty, 1);
    for (int b = 0; b < MINI_BUFS; ++b) { tc::mbar_init(&mini_full[b], 1); tc::mbar_init(&mini_empty[b], PROD_WARPS); }
    for (int j = 0; j < KB_MAX; ++j) { tc::mbar_init(&a_ready[j], PROD_WARPS); tc::mbar_init(&a_free[j], 1); }
    for (int b = 0; b < 2; ++b) { tc::mbar_init(&acc_full[b], 1); tc::mbar_init(&acc_empty[b], EPI_WARPS); }
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, TMEM_COLS);
  // columns past D: a = -30 (the W2^T rows are zero-filled), x - 1/2 = -1/2: a (x - 1/2) - |a|/2 = 15 - 15 and
  // ln(1 + e^-30) ~ 1e-13, so padding contributes nothing (no per-element bounds test)
  for (int i = threadIdx.x; i < DMAX; i += THREADS) {
    bb_s[i] = i < p.D ? p.b2[i] : ((p.cont && (i & 1)) ? -1.8378770664093453f : -30.f);
    xh_s[i] = p.cont ? 0.f : -0.5f;
  }
  for (int i = threadIdx.x; i < BM * 128 / 16; i += THREADS)          // [z|1] tile: k >= 24 stays zero
    reinterpret_cast<uint4*>(smem + Smem::ZB)[i] = make_uint4(0u, 0u, 0u, 0u);
  tc::fence_proxy_async();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  BarAddrs ba;
  ba.b_full = tc::smem_u32(b_full); ba.b_empty = tc::smem_u32(b_empty);
  ba.z_full = tc::smem_u32(z_full); ba.z_empty = tc::smem_u32(z_empty);
  ba.mini_full = tc::smem_u32(mini_full); ba.mini_empty = tc::smem_u32(mini_empty);
  ba.a_ready = tc::smem_u32(a_ready); ba.a_free = tc::smem_u32(a_free);
  ba.acc_full = tc::smem_u32(acc_full); ba.acc_empty = tc::smem_u32(acc_empty);

  if (warp == 0 || warp == 3) {
    // ===== TMA: W1^T boxes of the passes and W2^T boxes of the sweep, in walk_items order (alternate items) =====
    if (elect_one()) {
      TmaIssuer r;
      r.me = warp == 0 ? 0u : 1u;
      r.map_w2 = &map_w2; r.map_w1 = &map_w1; r.bar = ba;
      r.ring = tc::smem_u32(smem + Smem::B);
      r.w2_bytes = (uint32_t)p.NC * 128u; r.NC = p.NC;
      walk_items(p, n_tiles, r);
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer: ONE elected lane runs the whole loop =====
    if (elect_one()) {
      MmaIssuer r;
      r.bar = ba;
      r.tmem_base = tmem_base;
      // (the descriptor's address field takes 14 bits of the shared address >> 4)
      r.a_lo0 = ((tc::smem_u32(smem + Smem::A) & 0x3FFFFu) >> 4) | (1u << 16);       // LBO field = 1 (unused for SW128 K-major)
      r.b_lo0 = ((tc::smem_u32(smem + Smem::B) & 0x3FFFFu) >> 4) | (1u << 16);
      r.z_lo0 = ((tc::smem_u32(smem + Smem::ZB) & 0x3FFFFu) >> 4) | (1u << 16);
      r.idesc = tc::make_idesc_bf16(BM, p.NC, 0, 0);
      r.idesc_mini = tc::make_idesc_bf16(BM, MINI_N, 0, 0);
      r.KB = p.KB; r.zk = p.zk;
      walk_items(p, n_tiles, r);
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 4 + PROD_WARPS) {
    // ===== producers =====
    const int pw = warp - 4, pt = threadIdx.x - 128;           // pt in [0, 256)
    const int q = warp & 3, hsel = pw >> 2;                    // TMEM lane quarter, which 32-column half of a pass
    const int Z = p.Z;
    uint8_t* zb = smem + Smem::ZB;

    // z, [z|1] bf16 tile and the prior/posterior row terms of tile `t` (tile counter `ti`)
    auto make_z = [&](int t, uint32_t ti) {
      const int pi = t / p.tiles_per_point, l0 = (t - pi * p.tiles_per_point) * BM;
      tc::mbar_wait(z_empty, (ti & 1) ^ 1);
      const bool quad = (Z & 3) == 0 && !p.eps_inj;            // element groups line up with Philox groups
      for (int i = pt; i < BM * ZG; i += PROD_WARPS * 32) {
        const int r = i / ZG, g = i - r * ZG, j0 = 4 * g;
        const int l = l0 + r;
        float nrm[4] = {0.f, 0.f, 0.f, 0.f};
        if (quad && j0 < Z)
          philox_normal4(p.seed, VAEB_STREAM_IS, 0u, (uint32_t)l, (uint64_t)((p.row_offset + pi) * Z + j0) >> 2, nrm);
        float zq[4], a = 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = j0 + u;
          float zv = j == Z ? 1.0f : 0.f;                      // contraction index Z carries the bias b1
          if (j < Z) {
            float e;
            if (p.eps_inj) e = l < p.L ? p.eps_inj[((size_t)pi * p.L + l) * Z + j] : 0.f;
            else if (quad) e = nrm[u];
            else e = philox_normal1(p.seed, VAEB_STREAM_IS, 0u, (uint32_t)l, (uint64_t)((p.row_offset + pi) * Z + j));
            const float lsv = __ldg(p.ls + (size_t)pi * Z + j);
            zv = __ldg(p.mu + (size_t)pi * Z + j) + expf(0.5f * lsv) * e;
            a += -0.5f * zv * zv + 0.5f * lsv + 0.5f * e * e;  // log p(z) - log q(z|x), VAEB.py:322-325
          }
          zq[u] = zv;
        }
        auxp[r * ZG + g] = a;
        // 4 bf16 = 8 bytes at columns [4g, 4g+4) of row r (16-byte chunk g/2, swizzled)
        uint2 pk = make_uint2(pack_bf16(zq[0], zq[1]), pack_bf16(zq[2], zq[3]));
        *reinterpret_cast<uint2*>(zb + r * 128 + ((((uint32_t)g >> 1) ^ ((uint32_t)r & 7u)) << 4) + (g & 1) * 8) = pk;
      }
      tc::fence_proxy_async();
      named_bar(1, PROD_WARPS * 32);
      if (pt < BM) {
        float a = 0.f;
#pragma unroll
        for (int g = 0; g < ZG; ++g) a += auxp[pt * ZG + g];
        aux_s[(ti % 3) * BM + pt] = a;
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(z_full);
    };

    uint32_t tile_it = 0, mini_it = 0;
    if ((int)blockIdx.x < n_tiles) make_z(blockIdx.x, 0);
    const int r = q * 32 + lane;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tile_it) {
      // --- pre-activations -> tanh -> bf16 -> A tile: this warp owns rows [32q, 32q+32), columns [32 hsel, +32) of k block j
      for (int j = 0; j < p.KB; ++j, ++mini_it) {
        const uint32_t mb = mini_it % MINI_BUFS;
        tc::mbar_wait(&mini_full[mb], (mini_it / MINI_BUFS) & 1);
        tc::mbar_wait(&a_free[j], (tile_it & 1) ^ 1);          // the previous tile's last chunk has read this k block
        tc::tc_fence_after();
        const uint32_t taddr = tmem_base + MINI_COL0 + mb * MINI_N + hsel * 32 + ((uint32_t)(q * 32) << 16);
        uint8_t* arow = smem + Smem::A + j * A_BLOCK + r * 128;
        float v[32];
        tc::tmem_ld32(taddr, v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) {
          uint4 pk;
          pk.x = pack_bf16(tanh_approx(v[8 * c16 + 0]), tanh_approx(v[8 * c16 + 1]));
          pk.y = pack_bf16(tanh_approx(v[8 * c16 + 2]), tanh_approx(v[8 * c16 + 3]));
          pk.z = pack_bf16(tanh_approx(v[8 * c16 + 4]), tanh_approx(v[8 * c16 + 5]));
          pk.w = pack_bf16(tanh_approx(v[8 * c16 + 6]), tanh_approx(v[8 * c16 + 7]));
          const uint32_t chunk = (uint32_t)(hsel * 4 + c16);
          *reinterpret_cast<uint4*>(arow + ((chunk ^ ((uint32_t)r & 7u)) << 4)) = pk;
        }
        tc::fence_proxy_async();                               // generic-proxy writes -> visible to the MMA
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) { tc::mbar_arrive(&mini_empty[mb]); tc::mbar_arrive(&a_ready[j]); }
      }
      // --- z of the NEXT tile while this tile's output sweep runs
      const int tn = t + gridDim.x;
      if (tn < n_tiles) make_z(tn, tile_it + 1);
    }
  } else if (warp >= 4 + PROD_WARPS) {
    // ===== epilogue: TMEM -> x*a - softplus(a) row sums -> log w -> tile (max, sum exp) =====
    const int e = warp - 4 - PROD_WARPS, q = warp & 3, ch = e >> 2;   // TMEM lane quarter = warp % 4
    const int et = threadIdx.x - (4 + PROD_WARPS) * 32;                // [0, 256)
    const int row = q * 32 + lane;
    constexpr int SL = EPI_WARPS / 4;                                  // column slices of a chunk
    const int half = p.NC / SL, n8 = half >> 3, c_lo = ch * half;      // host: NC is a multiple of 8 * SL
    const uint32_t bb_addr = tc::smem_u32(bb_s), xh_addr = tc::smem_u32(xh_s);
    const FoldConsts fk = fold_consts();
    uint32_t acc_it = 0, tile_it = 0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++tile_it) {
      const int pi = t / p.tiles_per_point, l0 = (t - pi * p.tiles_per_point) * BM;
      if (p.cont) {
        for (int i = et; i < p.D; i += EPI_WARPS * 32) xh_s[i] = p.x[(size_t)pi * p.Dx + (i >> 1)];
      } else {
        for (int i = et; i < p.D; i += EPI_WARPS * 32) xh_s[i] = p.x[(size_t)pi * p.D + i] - 0.5f;
      }
      named_bar(2, EPI_WARPS * 32);
      uint64_t acc = 0ull;                                             // two fp32 partial sums (even / odd columns)
      float accg = 0.f;                                                // Gaussian decoder: one sum
      for (int c = 0; c < p.n_chunks; ++c, ++acc_it) {
        const uint32_t buf = acc_it & 1;
        tc::mbar_wait(&acc_full[buf], (acc_it >> 1) & 1);
        tc::tc_fence_after();
        const uint32_t taddr = tmem_base + buf * ACC_STRIDE + (uint32_t)c_lo + ((uint32_t)(q * 32) << 16);
        const uint32_t col4 = (uint32_t)(c * p.NC + c_lo) * 4u;
        const uint32_t ba = bb_addr + col4, xa = xh_addr + col4;
        // this warp's slice of the chunk; Gaussian decoder: 8 columns per TMEM load, the next load in flight while the
        // current 8 columns are folded
        float va[8], vb[8];
        tmem_ld8(taddr, va);
        if (p.cont) {
          for (int i = 0; i < n8; i += 2) {
            tc::tmem_ld_wait();
            if (i + 1 < n8) tmem_ld8(taddr + 8u * (i + 1), vb);
            fold8g(va, ba + 32u * i, xa + 32u * i, accg);
            if (i + 1 < n8) {
              tc::tmem_ld_wait();
              if (i + 2 < n8) tmem_ld8(taddr + 8u * (i + 2), va);
              fold8g(vb, ba + 32u * (i + 1), xa + 32u * (i + 1), accg);
            }
          }
        } else {
          // fewer, larger TMEM reads: a tcgen05.ld round trip is several times slower while MMAs accumulate into the other
          // buffer (DESIGN 4.3b), and a warp makes five of them per chunk with 8-column reads
          tc::tmem_ld_wait();
          fold8(va, ba, xa, fk, acc);
          for (int i = 1; i < n8; i += 2) {
            if (i + 1 < n8) {
              float w[16];
              tc::tmem_ld16(taddr + 8u * i, w);
              tc::tmem_ld_wait();
              fold8(*reinterpret_cast<const float(*)[8]>(w), ba + 32u * i, xa + 32u * i, fk, acc);
              fold8(*reinterpret_cast<const float(*)[8]>(w + 8), ba + 32u * (i + 1), xa + 32u * (i + 1), fk, acc);
            } else {
              tmem_ld8(taddr + 8u * i, vb);
              tc::tmem_ld_wait();
              fold8(vb, ba + 32u * i, xa + 32u * i, fk, acc);
            }
          }
        }
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&acc_empty[buf]);
      }
      float rs0, rs1;
      upk2(acc, rs0, rs1);
      const float rs = rs0 + rs1 + accg;
      rowsum_s[ch * BM + row] = rs;
      named_bar(2, EPI_WARPS * 32);
      if (ch == 0) {
        const int l = l0 + row;
        const bool valid = l < p.L;
        float lw = aux_s[(tile_it % 3) * BM + row];
#pragma unroll
        for (int sl = 0; sl < SL; ++sl) lw += rowsum_s[sl * BM + row];
        if (valid && p.logw_out) p.logw_out[(size_t)pi * p.L + l] = lw;
        float m = valid ? lw : -INFINITY;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float se = valid ? expf(lw - m) : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
        if (lane == 0) { red_s[2 * q] = m; red_s[2 * q + 1] = se; }
        named_bar(3, 4 * 32);
        if (et == 0) {
          float M = -INFINITY;
          for (int w = 0; w < 4; ++w) M = fmaxf(M, red_s[2 * w]);
          float S = 0.f;
          for (int w = 0; w < 4; ++w) if (red_s[2 * w] > -INFINITY) S += red_s[2 * w + 1] * expf(red_s[2 * w] - M);
          p.partial[t] = make_float2(M, S);
        }
        named_bar(3, 4 * 32);
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

// log p^(x_i) = log sum_t S_t exp(M_t - M) + M - log L   over the tiles of point i
__global__ void is_tc_finish_kernel(const float2* __restrict__ partial, int n_points, int tiles_per_point, int L,
                                    float* __restrict__ logp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_points) return;
  float M = -INFINITY;
  for (int t = 0; t < tiles_per_point; ++t) M = fmaxf(M, partial[(size_t)i * tiles_per_point + t].x);
  float S = 0.f;
  for (int t = 0; t < tiles_per_point; ++t) {
    const float2 v = partial[(size_t)i * tiles_per_point + t];
    if (v.x > -INFINITY) S += v.y * expf(v.x - M);
  }
  logp[i] = M + logf(S) - logf((float)L);
}

// W2 [H, D] fp32 -> W2^T [D, KP] bf16 (k contiguous, zero padded to KP = 64*KB)
// W6 != nullptr (Gaussian decoder): D output columns = the interleaved head, column 2d from W2[:, d], 2d + 1 from W6[:, d]
// (both [H, D / 2]); bias26 receives the interleaved biases
__global__ void is_tc_prep_kernel(const float* __restrict__ W2, int H, int D, int KP, int ld,
                                  __nv_bfloat16* __restrict__ w2t, const float* __restrict__ W6, const float* __restrict__ b2,
                                  const float* __restrict__ b6, float* __restrict__ bias26) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)D * KP) return;
  const int n = (int)(i / KP), k = (int)(i % KP);
  float v = 0.f;
  if (k < H) v = W6 ? ((n & 1) ? W6 : W2)[(size_t)k * (D / 2) + (n >> 1)] : W2[(size_t)k * D + n];
  w2t[(size_t)n * ld + k] = __float2bfloat16_rn(v);
  if (W6 && k == 0) bias26[n] = (n & 1) ? b6[n >> 1] : b2[n >> 1];
}

// [W1^T | b1] as the B operand of the hidden-layer GEMM: w1t[n][k] bf16, n < KP hidden units, 64 contraction
// slots: k < Z -> W1[k][n], k == Z -> b1[n], the rest (and rows n >= H) zero
__global__ void is_tc_prep_w1_kernel(const float* __restrict__ W1, const float* __restrict__ b1, int H, int Z, int KP,
                                     __nv_bfloat16* __restrict__ w1t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= KP * 64) return;
  const int n = i >> 6, k = i & 63;
  float v = 0.f;
  if (n < H) v = k < Z ? W1[(size_t)k * H + n] : (k == Z ? b1[n] : 0.f);
  w1t[i] = __float2bfloat16_rn(v);
}

}  // namespace istc

bool is_tc_supported(const vaeb_handle* h) {
  return h->cfg.precision == VAEB_PREC_BF16 && h->H <= 64 * istc::KB_MAX && h->Z <= istc::ZMAX &&
         (h->cont ? 2 * h->D : h->D) <= istc::DMAX && h->D >= 16;      // Gaussian decoder: 2 D interleaved output columns
}

// mu, ls: device [n, Z] (fp32 encoder already run); d_x device [n, D]; logp_out device [n]; logw_out device or nullptr
int is_tc_run(vaeb_handle* h, const float* d_x, const float* d_mu, const float* d_ls, int n, int L, const float* d_eps,
              int64_t row_offset, float* d_logp, float* d_logw) {
  using namespace istc;
  const Layout& l = h->lay;
  const int Dx = h->D, H = h->H, Z = h->Z;
  const int D = h->cont ? 2 * Dx : Dx;              // output columns of the decoder GEMM
  const int KB = (H + 63) / 64, KP = KB * 64;
  IsTcState& s = h->istc;
  cudaStream_t st = h->stream;
  if (!s.w2t) {
    VAEB_CUDA(cudaMalloc(&s.w2t, (size_t)D * (KP + W2T_PAD) * 2));
    VAEB_CUDA(cudaMalloc(&s.w1t, (size_t)(KB_MAX * 64) * 64 * 2));
    if (h->cont) VAEB_CUDA(cudaMalloc((void**)&s.bias26, (size_t)D * sizeof(float)));
    VAEB_CUDA(cudaMemset(s.w1t, 0, (size_t)(KB_MAX * 64) * 64 * 2));
    VAEB_TRY(vaeb_make_tmap_bf16((CUtensorMap*)s.map_w1, s.w1t, (uint64_t)(KB_MAX * 64), 64, 64, MINI_N));
    VAEB_CUDA(cudaFuncSetAttribute(is_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem::TOTAL));
    VAEB_CUDA(cudaDeviceGetAttribute(&s.n_sm, cudaDevAttrMultiProcessorCount, h->cfg.device));
    // output chunks: as few as fit NC_MAX accumulator columns, equal width (a multiple of 32): 784 -> 5 x 160
    const int n_chunks = (D + NC_MAX - 1) / NC_MAX;
    const int nc = (((D + n_chunks - 1) / n_chunks) + 31) & ~31;      // 8 columns per fold x EPI_WARPS / 4 slices
    s.n_chunks = n_chunks; s.tail_cols = nc;
    VAEB_TRY(vaeb_make_tmap_bf16((CUtensorMap*)s.map_full, s.w2t, (uint64_t)D, (uint64_t)KP, (uint64_t)(KP + W2T_PAD),
                                 (uint32_t)nc));
  }
  // the weights may have changed since the last call: refresh the bf16 transpose (0.8 MB)
  {
    const int64_t tot = (int64_t)D * KP;
    is_tc_prep_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
        h->d_params + l.off[l.iW2], H, D, KP, KP + W2T_PAD, (__nv_bfloat16*)s.w2t,
        h->cont ? h->d_params + l.off[l.iW6] : nullptr, h->d_params + l.off[l.ib2],
        h->cont ? h->d_params + l.off[l.ib6] : nullptr, s.bias26);
    ++h->launches;
    VAEB_CUDA(cudaGetLastError());
    is_tc_prep_w1_kernel<<<(KP * 64 + 255) / 256, 256, 0, st>>>(h->d_params + l.off[l.iW1], h->d_params + l.off[l.ib1], H,
                                                                Z, KP, (__nv_bfloat16*)s.w1t);
    ++h->launches;
    VAEB_CUDA(cudaGetLastError());
  }
  const int tpp = (L + BM - 1) / BM;
  const int64_t n_tiles = (int64_t)n * tpp;
  VAEB_REQUIRE(n_tiles < ((int64_t)1 << 31), "too many importance-sampling tiles in one call");
  if (n_tiles > s.partial_cap) {
    VAEB_CUDA(cudaStreamSynchronize(st));
    if (s.partial) VAEB_CUDA(cudaFree(s.partial));
    s.partial = nullptr;
    VAEB_CUDA(cudaMalloc(&s.partial, (size_t)n_tiles * sizeof(float2)));
    s.partial_cap = n_tiles;
  }
  Params p{};
  p.n_points = n; p.L = L; p.D = D; p.H = H; p.Z = Z; p.KB = KB;
  p.tiles_per_point = tpp; p.n_chunks = s.n_chunks; p.NC = s.tail_cols; p.zk = (Z + 1 + 15) / 16;
  p.x = d_x; p.mu = d_mu; p.ls = d_ls;
  p.b2 = h->cont ? s.bias26 : h->d_params + l.off[l.ib2];
  p.cont = h->cont ? 1 : 0; p.Dx = Dx;
  p.eps_inj = d_eps; p.seed = h->cfg.seed; p.row_offset = row_offset;
  p.partial = (float2*)s.partial; p.logw_out = d_logw;
  const int grid = (int)std::min<int64_t>(n_tiles, s.n_sm);
  is_tc_kernel<<<grid, THREADS, Smem::TOTAL, st>>>(*(const CUtensorMap*)s.map_full, *(const CUtensorMap*)s.map_w1, p);
  ++h->launches;
  VAEB_CUDA(cudaGetLastError());
  is_tc_finish_kernel<<<(n + 127) / 128, 128, 0, st>>>((const float2*)s.partial, n, tpp, L, d_logp);
  ++h->launches;
  VAEB_CUDA(cudaGetLastError());
  return VAEB_OK;
}

