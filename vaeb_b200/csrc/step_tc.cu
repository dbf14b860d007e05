// The tensor-core single-launch AEVB step (see step_tc.cuh): VAEB.py:408-415 at M <= 128 rows, Bernoulli decoder, L = 1.
//
// Work decomposition.  132 CTAs = 33 clusters of 4 (one CTA per SM).  A phase is a list of items:
//   * cluster items -- the skinny activation GEMMs out[128 x N] = act[128 x K] . W[K x N]: one N tile per cluster, the
//     contraction split four ways over the cluster's CTAs (k chunks of 64), partial accumulators read from TMEM and
//     reduce-scattered by rows through distributed shared memory (st.shared::cluster), each CTA finishing 32 rows with
//     the layer's fused epilogue (tanh / reparameterisation + KL / Bernoulli log-likelihood + delta / tanh' / dz);
//   * CTA items -- the weight-gradient GEMMs gW[128 features x N] = act^T . delta (K = the minibatch, zero padded to
//     128): one output tile per CTA, Adagrad with the prior (VAEB.py:389-390,426-444) in the epilogue, which also
//     rewrites the fp16 mirrors of the weights it just updated.
// Operands.  Every operand is a fp16 hi + lo pair of tiles in the UMMA K-major SWIZZLE_128B image.  Weights AND
// activations are kept in that image in global memory (L2): an epilogue thread stores the value it produced straight
// into the mirrors its consumers will load (row-major for the next layer, transposed for the weight gradients), so
// staging an operand is ONE cp.async.bulk issued by one thread and completed on an mbarrier.  Two operands are produced
// in software instead: the minibatch x (fp32 from the caller; staged while the CTA would otherwise wait at the
// preceding grid barrier) and the two thin layers around the latent code, recomputed with FFMA where they are consumed
// (h_d = tanh(z.W1 + b1) into the A tile of dec2, da3 = ([dmu|dls].W45^T)(1 - h_e^2) into the B tile of the W3 gradient).
// One thread issues hi*hi + hi*lo + lo*hi per k step (fp16 pairs, 22 mantissa bits: the fp32 parity tier) and commits to an mbarrier; all 16
// warps read TMEM.
// Phases of one update (a grid barrier after each):
//   P1 enc1 (+ the W4/W5 update of the previous step on the spare cluster)   P2 heads + reparam + KL
//   P3 dec1 (recomputed) + dec2 + log-lik + da2                              P4 dgrad -> da1
//   P5 dz -> dmu, dls | W2,b2 update | the bound                             P6 W3,b3 update (dh_e recomputed) | W1,b1 update
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "launchers.h"
#include "philox.cuh"
#include "step_tc.cuh"
#include "tc_common.cuh"

namespace st2 {

constexpr int TBA = MP * 128;                      // bytes of one 64-wide k chunk of a 128-row tile (hi or lo half)
constexpr int A_MAXCH = 4;
constexpr int SM_A = 0;                            // A_MAXCH chunks x (hi, lo) x 16 KB = 128 KB
constexpr int SM_B = A_MAXCH * 2 * TBA;            // B tiles: up to 32 KB (48 KB for the heads), scratch above
constexpr int SM_B_BYTES = 57344;
constexpr int SM_SCR = SM_B + 32768;               // 24 KB of producer scratch inside the B region
constexpr int SM_RECV = SM_B + SM_B_BYTES;         // [CL][32 rows][<= 64 cols] fp32 partials from the cluster
constexpr int SM_RECV_BYTES = CL * 32 * 64 * 4;
constexpr int SM_MISC = SM_RECV + SM_RECV_BYTES;   // mbarriers, TMEM slot, small reductions
constexpr int SMEM_BYTES = SM_MISC + 1024 + 1024;  // + slack for the 1024-byte alignment of the base
constexpr uint32_t TMEM_COLS = 256;                // columns 0..63: a layer's accumulator; 64..191: the decoder hidden layer

// Base of the (1024-byte aligned) dynamic shared memory, derived from the symbol itself: the compiler then knows every
// pointer built from it is a shared-memory pointer and emits LDS / STS instead of generic loads and stores.
extern __shared__ uint8_t st2_smem_raw[];
__device__ __forceinline__ uint8_t* smem_base() {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(st2_smem_raw);
  return st2_smem_raw + ((1024u - (a & 1023u)) & 1023u);
}

struct Ctx {
  uint8_t* sm;
  uint32_t tmem;
  uint64_t *mma_bar, *op_bar, *x_bar, *rs_bar;
  uint32_t mma_phase, op_phase, x_phase, rs_phase;
  int rank, cid, ncl, warp, lane;
  float tp;                            // sampled full VB: this thread's share of thetaPrior of the running step
  uint32_t step;                       // global index of the running step (Philox key of the weight noise)
};

// ---- PTX helpers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_idx() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_count() { uint32_t r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// 16 bytes into a peer CTA's shared memory; the peer's mbarrier counts them (no cluster barrier needed to hand them over)
__device__ __forceinline__ void st_async_v4(uint32_t addr, uint32_t mbar, float a, float b, float c, float d) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d), "r"(mbar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// one bulk copy global -> this CTA's shared memory, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(tc::smem_u32(dst)), "l"(src), "r"(bytes), "r"(tc::smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Operand format: every fp32 value v is carried as an fp16 pair hi = rn(v), lo = rn(v - hi): 22 mantissa bits
// (|error| <= max(2^-23 |v|, 2^-25): the residual of a small value is an fp16 subnormal with absolute spacing 2^-24),
// so hi*hi + hi*lo + lo*hi reproduces the fp32 product to ~2^-21 -- the fp32 parity tier.  Weights (|w| ~ 1e-2 at
// initialisation, VAEB.py:54) are mirrored times WSCALE = 2^8 so that their residuals stay normal numbers; the
// epilogue of a GEMM whose B operand is a weight mirror multiplies the sum by 2^-8 (exact).  Values are clamped to the
// fp16 range (a weight beyond +-255 or a delta beyond +-65504 is saturated instead of becoming inf - inf = NaN).
constexpr float WSCALE = 256.0f, WUNSCALE = 1.0f / 256.0f, H_MAX = 65504.0f;
__device__ __forceinline__ float clamp_h(float v) { return fminf(fmaxf(v, -H_MAX), H_MAX); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __half2 t = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&t);
}
// eight fp32 -> eight fp16 hi + eight fp16 lo
template <bool CLAMP = false>
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float a = CLAMP ? clamp_h(v[2 * q]) : v[2 * q], b = CLAMP ? clamp_h(v[2 * q + 1]) : v[2 * q + 1];
    h[q] = pack2(a, b);
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h[q]));
    l[q] = pack2(a - f.x, b - f.y);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}
template <bool CLAMP = false>
__device__ __forceinline__ void put_unit(uint8_t* d, int half_bytes, const float* v) {
  uint4 hi, lo;
  split8<CLAMP>(v, hi, lo);
  *reinterpret_cast<uint4*>(d) = hi;
  *reinterpret_cast<uint4*>(d + half_bytes) = lo;
}
// one element of a DELTA tensor (da2, da1, [dmu|dls], dh_e).  Their magnitude is unbounded (d/da of a Gaussian
// log-density scales with exp(-lv)) while fp16 ends at 65504, so the pair is (H, L) with v = 2^13 H + L: H = rn(v 2^-13)
// covers |v| < 5.4e8, L = rn(v - 2^13 H) is the residual (|L| <= 2^-11 |v|, or the whole value while it is below the
// spacing 2^-11 of H).  |error| <= max(2^-23 |v|, 2^-25) as for the other operands.  The two halves carry different
// scales, so the MMAs that read H accumulate into a second TMEM accumulator (DH_COL columns further) and the reader
// combines acc = 2^13 acc_H + acc_L.
constexpr float DSCALE = 8192.0f, DUNSCALE = 1.0f / 8192.0f;
// |da2|, |da1| above DLIMIT abort the step (Gaussian decoder): [dmu|dls] and dh_e, sums of at most 512 and 40 products
// of these with weights, then stay inside 65504 x DSCALE for any weights below ~1 in magnitude
constexpr float DLIMIT = 8192.0f;
constexpr uint32_t DH_COL = 192;                   // TMEM column offset of the accumulator of the H products
__device__ __forceinline__ void put_dl(uint8_t* d, int half_bytes, float v) {
  const __half h = __float2half_rn(clamp_h(v * DUNSCALE));
  *reinterpret_cast<__half*>(d) = h;
  *reinterpret_cast<__half*>(d + half_bytes) = __float2half_rn(clamp_h(fmaf(-DSCALE, __half2float(h), v)));
}
// one element (hi at d, lo half_bytes later)
__device__ __forceinline__ void put_hl(uint8_t* d, int half_bytes, float v) {
  v = clamp_h(v);
  const __half h = __float2half_rn(v);
  *reinterpret_cast<__half*>(d) = h;
  *reinterpret_cast<__half*>(d + half_bytes) = __float2half_rn(v - __half2float(h));
}
// branch-free tanh, relative error < 5e-6 (as the bf16x3 layer kernels, tc_layers.cu)
__device__ __forceinline__ float tanh_fast(float x) {
  const float ax = fabsf(x), x2 = x * x;
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * 2.8853900817779268f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  const float big = copysignf(fmaf(-2.0f, r, 1.0f), x);
  const float poly = fmaf(x * x2, fmaf(x2, fmaf(x2, fmaf(x2, 0.021869488536155203f, -0.053968253968253971f),
                                                0.13333333333333333f), -0.33333333333333331f), x);
  return ax < 0.1f ? poly : big;
}
// one exponential serves both: t = e^-|a|; softplus = max(a,0) + log(1+t); sigmoid = {1, t}/(1+t)  (MUFU ex2 / rcp /
// lg2 with ~1e-7 relative error each: the log-likelihood terms are O(1) and are summed over 784 pixels)
__device__ __forceinline__ void softplus_sigmoid(float a, float& sp, float& sg) {
  float t, r, lg;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-1.4426950408889634f * fabsf(a)));
  const float u = 1.0f + t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(u));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u));
  sp = fmaf(lg, 0.6931471805599453f, fmaxf(a, 0.f));
  sg = a >= 0.f ? r : t * r;
}

// byte offset of the 16-byte unit (row r, k octet cu) inside one K-major SWIZZLE_128B chunk tile
__device__ __forceinline__ uint32_t unit_off(int r, int cu) { return (uint32_t)r * 128u + (((uint32_t)cu ^ ((uint32_t)r & 7u)) << 4); }
// address of element (batch row r, column k) in a row-major activation mirror [k chunk][hi, lo][128 x 128 B]
__device__ __forceinline__ uint8_t* km_addr(uint8_t* base, int r, int k) {
  return base + (size_t)(k >> 6) * 2 * TBA + tc::sw128_offset(r, k & 63);
}
// address of element (row of feature tile `tile`, batch row b) in a transposed mirror
// [feature tile][batch chunk (2)][hi, lo][tile rows x 128 B]; half = tile rows * 128
__device__ __forceinline__ uint8_t* t_addr(uint8_t* base, int tile, int half, int row, int b) {
  return base + ((size_t)tile * 2 + (b >> 6)) * 2 * half + tc::sw128_offset(row, b & 63);
}

// ---- software producers for the minibatch x ------------------------------------------------------------------------
// Two-phase: every global load of a batch is issued before the first shared-memory store (one L2 round trip per batch).
// A tile of enc1: rows = batch rows, k in [64 c0, 64 (c0 + nch)), zero beyond D and beyond M rows.
__device__ __forceinline__ void stage_x_rows(uint8_t* sm, const float* __restrict__ x, int D, int M, int c0, int nch) {
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    float v[4][8];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int u = threadIdx.x + (half * 4 + b) * NT;          // 128 rows x 32 slots (4 chunks x 8 octets)
      const int r = u >> 5, ku = u & 31;
      const int k = (c0 + (ku >> 3)) * 64 + (ku & 7) * 8;
      if (ku < nch * 8 && r < M && k < D) {
        const float* s = x + (size_t)r * D + k;
        const float4 a0 = __ldcg(reinterpret_cast<const float4*>(s)), a1 = __ldcg(reinterpret_cast<const float4*>(s + 4));
        v[b][0] = a0.x; v[b][1] = a0.y; v[b][2] = a0.z; v[b][3] = a0.w;
        v[b][4] = a1.x; v[b][5] = a1.y; v[b][6] = a1.z; v[b][7] = a1.w;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[b][e] = 0.f;
      }
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int u = threadIdx.x + (half * 4 + b) * NT;
      const int r = u >> 5, ku = u & 31;
      if (ku < nch * 8) put_unit(sm + SM_A + (size_t)(ku >> 3) * 2 * TBA + unit_off(r, ku & 7), TBA, v[b]);
    }
  }
}
// The minibatch as tensor-core operands, written to global memory (P2, by the clusters without a latent-head item):
// x_km of the NEXT step (rows = batch rows, k = pixel: the A operand of enc1) and x_t of THIS step (rows = pixels, k =
// batch rows: the A operand of the W3 gradient; the row of pixel D is the constant 1 that yields the bias gradient).
// part / nparts: this CTA's share.  Rows >= M and pixels >= D are never written (zero since the mirrors were cleared).
__device__ __forceinline__ void item_xmirrors(const Params& p, const float* __restrict__ x_next, const float* __restrict__ x_cur,
                                              int part, int nparts) {
  const int D = p.D, M = p.M, D8 = D >> 3;
  if (x_next) {
    const int nu = M * D8;                                       // (batch row, pixel octet): lanes along the pixels
    for (int u = part * NT + threadIdx.x; u < nu; u += nparts * NT) {
      const int r = u / D8, ku = u - r * D8;
      const float* s = x_next + (size_t)r * D + ku * 8;
      const float4 a0 = __ldcg(reinterpret_cast<const float4*>(s)), a1 = __ldcg(reinterpret_cast<const float4*>(s + 4));
      const float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      put_unit(p.x_km + (size_t)(ku >> 3) * 2 * TBA + unit_off(r, ku & 7), TBA, v);
    }
  }
  {
    const int nbo = (M + 7) >> 3, nu = nbo * D;                  // (batch octet, pixel): lanes along the pixels
    for (int u = part * NT + threadIdx.x; u < nu; u += nparts * NT) {
      const int bo = u / D, f = u - bo * D;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = bo * 8 + e < M ? __ldcg(x_cur + (size_t)(bo * 8 + e) * D + f) : 0.f;
      put_unit(p.x_t + ((size_t)(f >> 7) * 2 + (bo >> 3)) * 2 * TBA + unit_off(f & 127, bo & 7), TBA, v);
    }
  }
}

// ---- MMA ---------------------------------------------------------------------------------------------------------
// thread 0: announce `bytes` of operand traffic on the operand barrier (the bulk copies follow)
// (the generic-proxy writes the copies read were fenced towards the async proxy by their WRITERS, before the grid
// barrier that ordered them before this thread: grid_barrier)
__device__ __forceinline__ void ops_begin(Ctx& c, uint32_t bytes) { tc::mbar_expect_tx(c.op_bar, bytes); }
// acc[128 x N] = sum over nch chunks / k16_total k steps of A.B^T (three MMAs per k step).  Called by EVERY thread; `wait_ops`: the
// issuing thread first waits for the bulk copies announced by ops_begin.  Returns when the accumulator is complete.
// fa / fb = 1: the A / B operand is a delta tensor (put_dl): the products with its H half go to the accumulator at
// DH_COL, the product with its L half to the main one.
__device__ __forceinline__ void mma_run(Ctx& c, int nch, int k16_total, int TBB, int N, bool wait_ops, uint32_t acc0 = 0u,
                                        int fa = 0, int fb = 0) {
  tc::fence_proxy_async();            // this thread's shared-memory stores -> visible to the tensor core (async proxy)
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  if (threadIdx.x == 0) {
    if (wait_ops) {
      tc::mbar_wait(c.op_bar, c.op_phase);
      c.op_phase ^= 1u;
      tc::tc_fence_after();
    }
    if (nch > 0) {
      const uint32_t idesc = tc::make_idesc_f16(MP, N, 0, 0);
      // descriptor = constant fields | (address >> 4); the address field (14 bits) never overflows: smem < 256 KB
      const uint64_t d0 = tc::make_smem_desc(0u, 16u, 1024u);
      const uint64_t a0 = d0 | (uint64_t)(tc::smem_u32(c.sm + SM_A) >> 4), b0 = d0 | (uint64_t)(tc::smem_u32(c.sm + SM_B) >> 4);
      const uint32_t a_lo = TBA >> 4, b_lo = (uint32_t)TBB >> 4;
      const uint32_t dL = c.tmem, dH = c.tmem + DH_COL;
      uint32_t acc = acc0;                 // != 0: a later pass of a contraction that does not fit the A region at once
      int k16 = 0;
#pragma unroll 1
      for (int ci = 0; ci < nch; ++ci) {
        const uint64_t a = a0 + (uint64_t)((uint32_t)ci * 2u * a_lo), b = b0 + (uint64_t)((uint32_t)ci * 2u * b_lo);
#pragma unroll
        for (int k = 0; k < 4; ++k, ++k16) {
          if (k16 >= k16_total) break;
          if (fa) {                        // A = (H, L)
            tc::umma_bf16(dH, a + 2 * k, b + 2 * k, idesc, acc);
            tc::umma_bf16(dH, a + 2 * k, b + b_lo + 2 * k, idesc, 1u);
            tc::umma_bf16(dL, a + a_lo + 2 * k, b + 2 * k, idesc, acc);
          } else if (fb) {                 // B = (H, L)
            tc::umma_bf16(dH, a + 2 * k, b + 2 * k, idesc, acc);
            tc::umma_bf16(dL, a + 2 * k, b + b_lo + 2 * k, idesc, acc);
            tc::umma_bf16(dH, a + a_lo + 2 * k, b + 2 * k, idesc, 1u);
          } else {
            tc::umma_bf16(dL, a + 2 * k, b + 2 * k, idesc, acc);
            tc::umma_bf16(dL, a + 2 * k, b + b_lo + 2 * k, idesc, 1u);
            tc::umma_bf16(dL, a + a_lo + 2 * k, b + 2 * k, idesc, 1u);
          }
          acc = 1u;
        }
      }
      tc::umma_commit(c.mma_bar);
    }
  }
  if (nch > 0) {
    tc::mbar_wait(c.mma_bar, c.mma_phase);
    c.mma_phase ^= 1u;
    tc::tc_fence_after();
  }
}
// eight accumulator columns of this thread's TMEM lane; delta: combined with the accumulator of the H products
__device__ __forceinline__ void acc_ld8(const Ctx& c, int q, uint32_t col, float* v, bool delta) {
  tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + col, v);
  if (delta) {
    float h[8];
    tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + DH_COL + col, h);
    tc::tmem_ld_wait();
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = fmaf(h[e], DSCALE, v[e]);
  } else {
    tc::tmem_ld_wait();
  }
}

// Partial accumulator [128 x N] -> the four CTAs of the cluster by row quarter: rows 32q..32q+31 go to CTA q, slot
// `rank` of its receive buffer, as asynchronous remote stores counted by the receiver's mbarrier (every CTA expects
// CL x 32 x N floats per item).  `have` == false sends zeros (this CTA had no k chunk).  Returns when this CTA's own
// receive buffer is complete.
__device__ __forceinline__ void reduce_scatter(Ctx& c, int N, bool have, bool delta = false) {
  const int q = c.warp & 3;
  if (threadIdx.x == 0) tc::mbar_expect_tx(c.rs_bar, (uint32_t)(CL * 32 * N * 4));
  const uint32_t dst0 = mapa(tc::smem_u32(c.sm + SM_RECV), (uint32_t)q);
  const uint32_t dbar = mapa(tc::smem_u32(c.rs_bar), (uint32_t)q);
  for (int u = c.warp >> 2; u < N / 8; u += 4) {
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (have) acc_ld8(c, q, (uint32_t)(u * 8), v, delta);
    const uint32_t d = dst0 + (uint32_t)(((c.rank * 32 + c.lane) * N + u * 8) * 4);
    st_async_v4(d, dbar, v[0], v[1], v[2], v[3]);
    st_async_v4(d + 16, dbar, v[4], v[5], v[6], v[7]);
  }
  tc::tc_fence_before();
  tc::mbar_wait(c.rs_bar, c.rs_phase);
  c.rs_phase ^= 1u;
}
__device__ __forceinline__ float recv_sum(const float* recv, int N, int row, int col) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < CL; ++k) s += recv[(k * 32 + row) * N + col];
  return s;
}

struct Hyper { float lr, eps, prior, p2, w; };   // w: the factor of the data term (1, or 1/M for the mean objective)
// Adagrad on the (up to) eight parameters one epilogue thread owns: every load is issued before the first store
// (one L2 round trip per unit), 16-byte accesses when the eight are contiguous and aligned.  nv = the new values.
__device__ __forceinline__ void adagrad8(float* P, float* ada, const size_t* off, const bool* ok, const float* g,
                                         const Hyper& hy, float* nv) {
  bool vec = (off[0] & 3) == 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) vec = vec && ok[e] && off[e] == off[0] + e;
  float p[8], a[8];
  if (vec) {
    const float4 p0 = __ldcg(reinterpret_cast<const float4*>(P + off[0])), p1 = __ldcg(reinterpret_cast<const float4*>(P + off[0] + 4));
    const float4 a0 = __ldcg(reinterpret_cast<const float4*>(ada + off[0])), a1 = __ldcg(reinterpret_cast<const float4*>(ada + off[0] + 4));
    p[0] = p0.x; p[1] = p0.y; p[2] = p0.z; p[3] = p0.w; p[4] = p1.x; p[5] = p1.y; p[6] = p1.z; p[7] = p1.w;
    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      p[e] = ok[e] ? __ldcg(P + off[e]) : 0.f;
      a[e] = ok[e] ? __ldcg(ada + off[e]) : 0.f;
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float gg = fmaf(g[e], hy.w, -hy.prior * p[e]);     // VAEB.py:389-390
    a[e] += gg * gg;                                      // VAEB.py:439
    float q = p[e] + hy.lr * gg / (sqrtf(a[e]) + hy.eps); // VAEB.py:441
    if (hy.p2 != 0.f) q -= hy.p2 * p[e] * p[e];           // VAEBfullbayes.py:183-184
    nv[e] = q;
  }
  if (vec) {
    *reinterpret_cast<float4*>(P + off[0]) = make_float4(nv[0], nv[1], nv[2], nv[3]);
    *reinterpret_cast<float4*>(P + off[0] + 4) = make_float4(nv[4], nv[5], nv[6], nv[7]);
    *reinterpret_cast<float4*>(ada + off[0]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(ada + off[0] + 4) = make_float4(a[4], a[5], a[6], a[7]);
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e)
      if (ok[e]) { P[off[e]] = nv[e]; ada[off[e]] = a[e]; }
  }
}
// one element of a weight mirror: tiles of TR rows (tile index nt, row r inside it), KC chunks per tile
__device__ __forceinline__ void mirror_put(uint8_t* m, int TR, int KC, int nt, int r, int k, float v) {
  const int TB = TR * 128;
  put_hl(m + ((size_t)nt * KC + (k >> 6)) * 2 * TB + tc::sw128_offset(r, k & 63), TB, v * WSCALE);
}

// ---- grid barrier (monotonic counter, release / acquire at gpu scope) --------------------------------------------
__device__ __forceinline__ void grid_barrier(unsigned long long* bar, unsigned long long target) {
  fence_proxy_async_all();            // this thread's global stores -> ordered before later async-proxy (bulk copy) reads
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(bar) : "memory");
    unsigned long long v;
    uint32_t spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(bar) : "memory");
      if (++spins > 20000000u) __trap();     // a lost CTA must abort the launch, not hang the GPU
    } while (v < target);
    __threadfence();
  }
  __syncthreads();
}

// =================================================================================================================
// cluster items
// =================================================================================================================
// P1: h_e[:, 16t .. 16t+15] = tanh(x.W3 + b3)                                               VAEB.py:246
// a_mode: where the A tile (this rank's k chunks of x) comes from
enum { A_BULK = 0,       // one bulk copy from x_km (written in P2 of the previous step), issued here
       A_PREFETCHED = 1, // that bulk copy was issued before the grid barrier that opened the phase (x_bar)
       A_STAGED = 2,     // already converted into shared memory by this CTA (first step of a launch)
       A_SOFTWARE = 3 }; // convert from the fp32 rows now (first step of a launch, second item of a cluster)
__device__ __forceinline__ void item_enc1(Ctx& c, const Params& p, const float* x, float* he, uint8_t* he_t, int t, int a_mode, bool more) {
  const int c0 = c.rank * p.KD / CL, c1 = (c.rank + 1) * p.KD / CL, nch = c1 - c0;
  constexpr int TB = TR_ENC1 * 128;
  if (threadIdx.x == 0 && nch > 0) {
    ops_begin(c, (uint32_t)(nch * 2 * TB + (a_mode == A_BULK ? nch * 2 * TBA : 0)));
    if (a_mode == A_BULK) bulk_g2s(c.sm + SM_A, p.x_km + (size_t)c0 * 2 * TBA, (uint32_t)(nch * 2 * TBA), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.m_enc1 + ((size_t)t * p.KD + c0) * 2 * TB, (uint32_t)(nch * 2 * TB), c.op_bar);
    if (a_mode == A_PREFETCHED) { tc::mbar_wait(c.x_bar, c.x_phase); c.x_phase ^= 1u; }
  }
  if (a_mode == A_SOFTWARE) stage_x_rows(c.sm, x, p.D, p.M, c0, nch);
  const int row = threadIdx.x >> 4, col = threadIdx.x & 15;
  const int gr = c.rank * 32 + row, j = t * 16 + col;
  const float bias = j < p.H ? __ldcg(p.P + p.ob3 + j) : 0.f;
  mma_run(c, nch, min(nch * 4, (p.D - c0 * 64 + 15) / 16), TB, TR_ENC1, nch > 0);
  reduce_scatter(c, TR_ENC1, nch > 0);
  const float* recv = reinterpret_cast<const float*>(c.sm + SM_RECV);
  if (gr < p.M) {
    const float v = j < p.H ? tanh_fast(fmaf(recv_sum(recv, TR_ENC1, row, col), WUNSCALE, bias)) : 0.f;
    he[(size_t)gr * p.HP + j] = v;
    put_hl(km_addr(p.he_km, gr, j), TBA, v);
    if (j < p.H) put_hl(t_addr(he_t, j >> 7, TBA, j & 127, gr), TBA, v);
  }
  if (more) cluster_sync();          // the receive buffer is reused by this cluster's next item of the phase
  else __syncthreads();
}

// P2: (mu, ls) = h_e.[W4|W5] + b, eps, z = mu + exp(ls/2) eps, the KL / L^A row term        VAEB.py:248-249,41-47,343,322-325
__device__ __forceinline__ void item_heads(Ctx& c, const Params& p, uint32_t step, bool more) {
  const int c0 = c.rank * p.KH / CL, c1 = (c.rank + 1) * p.KH / CL, nch = c1 - c0;
  const int TB = p.NH * 128, Z = p.Z, N = p.NH;
  if (threadIdx.x == 0 && nch > 0) {
    ops_begin(c, (uint32_t)(nch * 2 * (TBA + TB)));
    bulk_g2s(c.sm + SM_A, p.he_km + (size_t)c0 * 2 * TBA, (uint32_t)(nch * 2 * TBA), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.m_heads + (size_t)c0 * 2 * TB, (uint32_t)(nch * 2 * TB), c.op_bar);
  }
  // while the operands are in flight: this thread's noise (drawn in P1 by the spare cluster, or injected) and biases
  const float* eps_src = p.eps_inj ? p.eps_inj : p.eps;
  float e_[2], b4_[2], b5_[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    const int row = it / Z, j = it - row * Z;
    const int gr = c.rank * 32 + row;
    e_[i] = b4_[i] = b5_[i] = 0.f;
    if (it < 32 * Z && gr < p.M) {
      e_[i] = __ldcg(eps_src + (size_t)gr * Z + j);
      b4_[i] = __ldcg(p.P + p.ob4 + j); b5_[i] = __ldcg(p.P + p.ob5 + j);
    }
  }
  mma_run(c, nch, nch * 4, TB, N, nch > 0);
  reduce_scatter(c, N, nch > 0);
  const float* recv = reinterpret_cast<const float*>(c.sm + SM_RECV);
  float* term = reinterpret_cast<float*>(c.sm + SM_B);          // [32][Z] (the B tiles are dead)
  const int zt_half = p.NZ * 128;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    if (it >= 32 * Z) break;
    const int row = it / Z, j = it - row * Z;
    const int gr = c.rank * 32 + row;
    float tv = 0.f;
    if (gr < p.M) {
      const float am = fmaf(recv_sum(recv, N, row, j), WUNSCALE, b4_[i]);
      const float al = fmaf(recv_sum(recv, N, row, Z + j), WUNSCALE, b5_[i]);
      const size_t o = (size_t)gr * Z + j;
      const float e = e_[i];
      const float zv = am + expf(0.5f * al) * e;
      p.mu[o] = am; p.ls[o] = al; p.z[o] = zv;
      put_hl(km_addr(p.z_km, gr, j), TBA, zv);
      if (p.eps_inj) p.eps[o] = e;
      put_hl(t_addr(p.z_t, 0, zt_half, j, gr), zt_half, zv);
      tv = p.la ? (-0.5f * zv * zv + 0.5f * al + 0.5f * e * e) : 0.5f * (1.0f + al - am * am - expf(al));
    }
    term[it] = tv;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int gr = c.rank * 32 + threadIdx.x;
    if (gr < p.M) {
      float s = 0.f;
      for (int j = 0; j < Z; ++j) s += term[threadIdx.x * Z + j];
      p.aux[gr] = s;
    }
  }
  if (more) cluster_sync();          // the receive buffer is reused by this cluster's next item of the phase
  else __syncthreads();
}

// P3: h_d = tanh(z.W1 + b1) recomputed into the A tile, a = h_d.W2 + b2, x a - softplus(a), da2 = x - sigmoid a
//                                                                                           VAEB.py:254,263,311
// Gaussian decoder: the tile holds [W2 | W6] for 32 pixels; mu = sigmoid(a), lv = h_d.W6 + b6, the log-density of
// VAEB.py:306-307 and its two deltas.
__device__ __forceinline__ void item_dec2(Ctx& c, const Params& p, const float* x, int t, bool more, bool publish, int s) {
  const int c0 = c.rank * p.KH / CL, c1 = (c.rank + 1) * p.KH / CL, nch = c1 - c0;
  const int TR = p.TR3, TB = TR * 128;
  const int H = p.H, M = p.M;
  // Operands of BOTH GEMMs of the item in one transaction: [z|1] (A of the hidden layer) into the last chunk slot of
  // the A region, this rank's 64-unit tiles of [W1^T|b1] into the slot before it (nch <= 2: H <= 512).
  constexpr int T1 = 64 * 128;                                  // one half (hi or lo) of a [W1^T|b1] tile
  uint8_t* z_sm = c.sm + SM_A + 3 * 2 * TBA;
  uint8_t* w1_sm = c.sm + SM_A + 2 * 2 * TBA;
  if (threadIdx.x == 0 && nch > 0) {
    ops_begin(c, (uint32_t)(nch * 2 * TB + 2 * TBA + nch * 2 * T1));
    bulk_g2s(z_sm, p.z_km, (uint32_t)(2 * TBA), c.op_bar);
    bulk_g2s(w1_sm, p.m_dec1 + (size_t)c0 * 2 * T1, (uint32_t)(nch * 2 * T1), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.m_dec2 + ((size_t)t * p.KH + c0) * 2 * TB, (uint32_t)(nch * 2 * TB), c.op_bar);
  }
  // this thread's two elements of the final stage: x and the output biases (in flight during both GEMMs)
  float xv_[2], b2_[2], b6_[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    const int gr = c.rank * 32 + (it >> 5), n = t * 32 + (it & 31);
    const bool ok = gr < M && n < p.D;
    xv_[i] = ok ? __ldcg(x + (size_t)gr * p.D + n) : 0.f;
    b2_[i] = ok ? __ldcg(p.P + p.ob2 + n) : 0.f;
    b6_[i] = (ok && p.cont) ? __ldcg(p.P + p.ob6 + n) : 0.f;
  }
  // ---- hidden layer on the tensor cores: D1[128 x 64 nch] = [z|1] . [W1^T|b1]^T (K = 32: latent code + bias) --------
  tc::tc_fence_before();
  __syncthreads();                                              // the previous item's TMEM reads are complete
  tc::tc_fence_after();
  if (threadIdx.x == 0 && nch > 0) {
    tc::mbar_wait(c.op_bar, c.op_phase);
    c.op_phase ^= 1u;
    tc::tc_fence_after();
    const uint32_t idesc = tc::make_idesc_f16(MP, 64, 0, 0);
    const uint64_t d0 = tc::make_smem_desc(0u, 16u, 1024u);
    const uint64_t a = d0 | (uint64_t)(tc::smem_u32(z_sm) >> 4);
    const uint32_t a_lo = TBA >> 4, b_lo = T1 >> 4;
    for (int ci = 0; ci < nch; ++ci) {
      const uint64_t b = d0 | (uint64_t)((tc::smem_u32(w1_sm) + (uint32_t)ci * 2u * T1) >> 4);
      const uint32_t dcol = c.tmem + 64u + (uint32_t)ci * 64u;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        tc::umma_bf16(dcol, a + 2 * k, b + 2 * k, idesc, k ? 1u : 0u);
        tc::umma_bf16(dcol, a + 2 * k, b + b_lo + 2 * k, idesc, 1u);
        tc::umma_bf16(dcol, a + a_lo + 2 * k, b + 2 * k, idesc, 1u);
      }
    }
    tc::umma_commit(c.mma_bar);
  }
  if (nch > 0) {
    tc::mbar_wait(c.mma_bar, c.mma_phase);
    c.mma_phase ^= 1u;
    tc::tc_fence_after();
  }
  {
    // h_d = tanh(D1) (the bias rode along as latent column Z) -> the A tile of the output layer; thread = batch row,
    // eight consecutive hidden units per TMEM read = one 16-byte unit of the tile
    const int q = c.warp & 3, cg = c.warp >> 2;                 // lane quarter; 32-column group of the (up to) 128 columns
    const int r = q * 32 + c.lane;
    if (cg * 32 < nch * 64) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float v[8];
        tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + 64u + (uint32_t)(cg * 32 + u * 8), v);
        tc::tmem_ld_wait();
        const int kl = cg * 32 + u * 8;                          // column inside this rank's slice
        const int k0 = c0 * 64 + kl;
        if (r < M && k0 + 8 <= H) {                              // the common case, without per-element predicates
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = tanh_fast(v[e] * WUNSCALE);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = (r < M && k0 + e < H) ? tanh_fast(v[e] * WUNSCALE) : 0.f;
        }
        if (publish && r < M && r % p.n_tiles3 == t) {           // no spare cluster: every cluster publishes a few rows of h_d
          float* o = p.hd + (size_t)r * p.HP + k0;
          *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(o + 4) = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
          for (int e = 0; e < 8; ++e)
            if (k0 + e < H) put_hl(t_addr(p.hd_t, (k0 + e) >> 7, TBA, (k0 + e) & 127, r), TBA, v[e]);
        }
        put_unit(c.sm + SM_A + (size_t)(kl >> 6) * 2 * TBA + unit_off(r, (kl & 63) >> 3), TBA, v);
      }
    }
  }
  mma_run(c, nch, nch * 4, TB, TR, false);
  reduce_scatter(c, TR, nch > 0);
  const float* recv = reinterpret_cast<const float*>(c.sm + SM_RECV);
  float* term = reinterpret_cast<float*>(c.sm + SM_B);          // [32][32]
  float* dtile = term + 32 * 32;                                // [32][33] (+ a second one for the Gaussian lv deltas)
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    const int row = it >> 5, col = it & 31;
    const int gr = c.rank * 32 + row, n = t * 32 + col;
    float tv = 0.f, dval = 0.f, dval2 = 0.f;
    if (gr < M && n < p.D) {
      const float a = fmaf(recv_sum(recv, TR, row, col), WUNSCALE, b2_[i]);
      const float xv = xv_[i];
      float sp, sg;
      softplus_sigmoid(a, sp, sg);
      if (!p.cont) {
        dval = xv - sg;                                          // deltas are carried without the factor w (applied with the weight gradients)
        put_dl(km_addr(p.da2_km, gr, n), TBA, dval);
        tv = xv * a - sp;
      } else {
        const float lv = fmaf(recv_sum(recv, TR, row, 32 + col), WUNSCALE, b6_[i]);
        float iv;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(iv) : "f"(-1.4426950408889634f * lv));   // exp(-lv)
        const float d = xv - sg, r_ = d * iv;
        dval = r_ * sg * (1.0f - sg);                            // d/da   of VAEB.py:306-307 through mu = sigmoid(a)
        dval2 = fmaf(0.5f * d, r_, -0.5f);                       // d/dlv
        if (!(fmaxf(fabsf(dval), fabsf(dval2)) <= DLIMIT)) *p.status = s;   // (also NaN) -> the launch stops before P5
        put_dl(km_addr(p.da2_km, gr, t * 64 + col), TBA, dval);
        put_dl(km_addr(p.da2_km, gr, t * 64 + 32 + col), TBA, dval2);
        tv = -0.91893853320467274178f - 0.5f * lv - 0.5f * d * r_;
      }
    }
    term[it] = tv;
    dtile[row * 33 + col] = dval;
    if (p.cont) dtile[32 * 33 + row * 33 + col] = dval2;
  }
  __syncthreads();
  // the transposed mirror (operand of the W2 gradient) with the lanes along the batch rows: 64 contiguous bytes per store
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    const int col = it >> 5, row = it & 31;
    const int gr = c.rank * 32 + row, n = t * 32 + col;
    if (gr < M && n < p.D) {
      put_dl(t_addr(p.da2_t, t, TB, col, gr), TB, dtile[row * 33 + col]);
      if (p.cont) put_dl(t_addr(p.da2_t, t, TB, 32 + col, gr), TB, dtile[32 * 33 + row * 33 + col]);
    }
  }
  if (threadIdx.x < 32) {
    const int gr = c.rank * 32 + threadIdx.x;
    if (gr < M) {
      float s = 0.f;
      for (int j = 0; j < 32; ++j) s += term[threadIdx.x * 32 + j];
      p.partial[(size_t)gr * p.n_tiles3 + t] = s;
    }
  }
  if (more) cluster_sync();          // the receive buffer is reused by this cluster's next item of the phase
  else __syncthreads();
}

// P3, spare clusters: h_d = tanh([z|1].[W1^T|b1]^T) for 16 hidden units per CTA, published for P4 (fp32, the tanh'
// factor) and P5 (transposed operand of the W2 gradient).  The dec2 items recompute h_d for themselves.
__device__ __forceinline__ void item_hd(Ctx& c, const Params& p, int g) {
  constexpr int T1 = 64 * 128;
  uint8_t* z_sm = c.sm + SM_A;
  uint8_t* w_sm = c.sm + SM_B;                                  // [hi 16 rows x 128 B][lo]
  const uint8_t* src = p.m_dec1 + (size_t)(g >> 2) * 2 * T1 + (size_t)(g & 3) * 2048;
  if (threadIdx.x == 0) {
    ops_begin(c, (uint32_t)(2 * TBA + 4096));
    bulk_g2s(z_sm, p.z_km, (uint32_t)(2 * TBA), c.op_bar);
    bulk_g2s(w_sm, src, 2048u, c.op_bar);
    bulk_g2s(w_sm + 2048, src + T1, 2048u, c.op_bar);
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  if (threadIdx.x == 0) {
    tc::mbar_wait(c.op_bar, c.op_phase);
    c.op_phase ^= 1u;
    tc::tc_fence_after();
    const uint32_t idesc = tc::make_idesc_f16(MP, 16, 0, 0);
    const uint64_t d0 = tc::make_smem_desc(0u, 16u, 1024u);
    const uint64_t a = d0 | (uint64_t)(tc::smem_u32(z_sm) >> 4), b = d0 | (uint64_t)(tc::smem_u32(w_sm) >> 4);
    const uint32_t a_lo = TBA >> 4, b_lo = 2048u >> 4;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      tc::umma_bf16(c.tmem, a + 2 * k, b + 2 * k, idesc, k ? 1u : 0u);
      tc::umma_bf16(c.tmem, a + 2 * k, b + b_lo + 2 * k, idesc, 1u);
      tc::umma_bf16(c.tmem, a + a_lo + 2 * k, b + 2 * k, idesc, 1u);
    }
    tc::umma_commit(c.mma_bar);
  }
  tc::mbar_wait(c.mma_bar, c.mma_phase);
  c.mma_phase ^= 1u;
  tc::tc_fence_after();
  const int q = c.warp & 3, u = c.warp >> 2;
  if (u < 2) {
    float v[8];
    tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(u * 8), v);
    tc::tmem_ld_wait();
    const int r = q * 32 + c.lane, k0 = g * 16 + u * 8;
    if (r < p.M) {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = k0 + e < p.H ? tanh_fast(v[e] * WUNSCALE) : 0.f;
      float* o = p.hd + (size_t)r * p.HP + k0;
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(v[4], v[5], v[6], v[7]);
#pragma unroll
      for (int e = 0; e < 8; ++e)                               // lanes = consecutive batch rows: 64 contiguous bytes per store
        if (k0 + e < p.H) put_hl(t_addr(p.hd_t, (k0 + e) >> 7, TBA, (k0 + e) & 127, r), TBA, v[e]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
}

// P4: da1[:, 16t..] = (da2.W2^T) * (1 - h_d^2)                                              T.grad, VAEB.py:397
// (Gaussian decoder: K runs over the virtual columns [da | dlv] against [W2 | W6]^T.)  A rank's share of K may exceed
// the A region (Frey Face: 18 chunks over 4 ranks): further passes accumulate into the same TMEM columns.
__device__ __forceinline__ void item_dgrad(Ctx& c, const Params& p, int t, bool more, int s) {
  const int c0 = c.rank * p.KV / CL, c1 = (c.rank + 1) * p.KV / CL, nch = c1 - c0;
  constexpr int TB = TR_DGRAD * 128;
  const int row = threadIdx.x >> 4, col = threadIdx.x & 15;
  const int gr = c.rank * 32 + row, j = t * 16 + col;
  const float hv = gr < p.M ? __ldcg(p.hd + (size_t)gr * p.HP + j) : 0.f;
  for (int base = 0; base < nch || base == 0; base += A_MAXCH) {
    const int n = min(nch - base, A_MAXCH);
    if (threadIdx.x == 0 && n > 0) {
      ops_begin(c, (uint32_t)(n * 2 * (TBA + TB)));
      bulk_g2s(c.sm + SM_A, p.da2_km + (size_t)(c0 + base) * 2 * TBA, (uint32_t)(n * 2 * TBA), c.op_bar);
      bulk_g2s(c.sm + SM_B, p.m_dgrad + ((size_t)t * p.KV + c0 + base) * 2 * TB, (uint32_t)(n * 2 * TB), c.op_bar);
    }
    const int k16 = p.cont ? n * 4 : min(n * 4, (p.D - (c0 + base) * 64 + 15) / 16);
    mma_run(c, max(n, 0), k16, TB, TR_DGRAD, n > 0, base ? 1u : 0u, 1, 0);
  }
  reduce_scatter(c, TR_DGRAD, nch > 0, true);
  const float* recv = reinterpret_cast<const float*>(c.sm + SM_RECV);
  if (gr < p.M) {
    const float d = recv_sum(recv, TR_DGRAD, row, col) * WUNSCALE * (1.0f - hv * hv);
    if (p.cont && !(fabsf(d) <= DLIMIT)) *p.status = s;
    put_dl(km_addr(p.da1_km, gr, j), TBA, d);
    if (j < p.H) put_dl(t_addr(p.da1_t, j >> 7, TBA, j & 127, gr), TBA, d);
  }
  if (more) cluster_sync();          // the receive buffer is reused by this cluster's next item of the phase
  else __syncthreads();
}

// P5: dz = da1.W1^T -> dmu, dls (SURVEY.md 8a backward formulas).  kb = the step's KL weight: its three terms carry it,
// and the weight-gradient epilogues scale the whole gradient by w, so the update ascends w (grad loglik + kb grad aux)
__device__ __forceinline__ void item_dz(Ctx& c, const Params& p, bool more, float kb) {
  const int c0 = c.rank * p.KH / CL, c1 = (c.rank + 1) * p.KH / CL, nch = c1 - c0;
  const int TB = p.NZ * 128, Z = p.Z, N = p.NZ;
  if (threadIdx.x == 0 && nch > 0) {
    ops_begin(c, (uint32_t)(nch * 2 * (TBA + TB)));
    bulk_g2s(c.sm + SM_A, p.da1_km + (size_t)c0 * 2 * TBA, (uint32_t)(nch * 2 * TBA), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.m_dz + (size_t)c0 * 2 * TB, (uint32_t)(nch * 2 * TB), c.op_bar);
  }
  float ls_[2], ev_[2], zm_[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    const int row = it / Z, j = it - row * Z;
    const int gr = c.rank * 32 + row;
    ls_[i] = ev_[i] = zm_[i] = 0.f;
    if (it < 32 * Z && gr < p.M) {
      const size_t o = (size_t)gr * Z + j;
      ls_[i] = __ldcg(p.ls + o); ev_[i] = __ldcg(p.eps + o);
      zm_[i] = p.la ? __ldcg(p.z + o) : __ldcg(p.mu + o);
    }
  }
  mma_run(c, nch, nch * 4, TB, N, nch > 0, 0u, 1, 0);
  reduce_scatter(c, N, nch > 0, true);
  const float* recv = reinterpret_cast<const float*>(c.sm + SM_RECV);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int it = threadIdx.x + i * NT;
    if (it >= 32 * Z) break;
    const int row = it / Z, j = it - row * Z;
    const int gr = c.rank * 32 + row;
    if (gr < p.M) {
      float d = recv_sum(recv, N, row, j) * WUNSCALE;
      if (p.la) d -= kb * zm_[i];
      float a = d, b = d * (0.5f * expf(0.5f * ls_[i]) * ev_[i]);
      if (p.la) {
        b += kb * 0.5f;
      } else {
        a -= kb * zm_[i];
        b += kb * 0.5f * (1.0f - expf(ls_[i]));
      }
      put_dl(km_addr(p.dd_km, gr, j), TBA, a);                                   // A operand of the dh_e GEMMs (P6)
      put_dl(km_addr(p.dd_km, gr, Z + j), TBA, b);
      put_dl(t_addr(p.dd_t, j >> 4, 2048, j & 15, gr), 2048, a);                 // [dmu|dls]^T in tiles of 16 columns
      put_dl(t_addr(p.dd_t, (Z + j) >> 4, 2048, (Z + j) & 15, gr), 2048, b);
    }
  }
  if (more) cluster_sync();          // the receive buffer is reused by this cluster's next item of the phase
  else __syncthreads();
}

// =================================================================================================================
// CTA items: weight gradients with Adagrad (+ prior) in the epilogue                        VAEB.py:397,389-390,426-444
// =================================================================================================================
// epilogue driver: fn(row in the 128-row tile, first column of an 8-column unit, the eight sums)
template <class F>
__device__ __forceinline__ void wgrad_epilogue(Ctx& c, int N, F fn) {
  const int q = c.warp & 3;
  for (int u = c.warp >> 2; u < N / 8; u += 4) {
    float v[8];
    tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(u * 8), v);
    tc::tmem_ld_wait();
    fn(q * 32 + c.lane, u * 8, v);
  }
  tc::tc_fence_before();
  __syncthreads();
}

// Coalesced form.  The accumulator tile [128 x N] (N = 16 or 32) goes through shared memory twice:
//   A  thread = accumulator row (TMEM lane): the sums are parked in a [128][33] fp32 tile;
//   B  lane = column: a warp instruction reads / writes ONE contiguous row segment of the parameters and of the
//      accumulators (the uncoalesced form touches 32 lines per instruction and is bound by L1 request processing:
//      3.6 us per tile measured), Adagrad, the new values go back into the tile;
//   C  thread = row again: `mir(row, col0, nv[8])` writes the fp16 mirrors (their k index runs along the rows).
// off(row, col) = flat offset of the parameter behind accumulator element (row, col), or -1.
// ---- sampled full VB (VAEB.py:127-129 live inside getFVBL) ------------------------------------------------------------
// The update epilogues are issue bound (per parameter: thetaPrior, two Adagrad rules, a Philox draw), so they use the
// MUFU forms: relative error ~2^-22 each, far inside the parity tier; zeta' is stored and the stored value is what
// both theta' and the next step's d/dsigma use, so nothing has to reproduce it bit for bit.
__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_lg2(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// the four N(0,1) draws of Philox group g (flat parameters 4g .. 4g+3): philox_normal4 with MUFU log / sqrt / sin / cos
__device__ __forceinline__ void zeta_group(const Params& p, uint32_t step, uint64_t g, float n[4]) {
  uint32_t r[4];
  philox4x32_10((uint32_t)g, ((uint32_t)(g >> 32) & 0x00FFFFFFu) | ((VAEB_STREAM_ZETA & 0xFFu) << 24), 0u, step,
                (uint32_t)p.seed, (uint32_t)(p.seed >> 32), r);
  const float u0 = ((float)(r[0] >> 8) + 0.5f) * 5.9604644775390625e-8f, u1 = ((float)(r[1] >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float u2 = ((float)(r[2] >> 8) + 0.5f) * 5.9604644775390625e-8f, u3 = ((float)(r[3] >> 8) + 0.5f) * 5.9604644775390625e-8f;
  const float rad0 = fast_sqrt(-1.3862943611198906f * fast_lg2(u0)), rad1 = fast_sqrt(-1.3862943611198906f * fast_lg2(u2));
  // angles in (-pi, pi): the same point of the circle as 2 pi u, where sin.approx / cos.approx are most accurate
  const float a0 = 6.283185307179586f * (u1 - (u1 >= 0.5f ? 1.0f : 0.0f)), a1 = 6.283185307179586f * (u3 - (u3 >= 0.5f ? 1.0f : 0.0f));
  n[0] = rad0 * __cosf(a0); n[1] = rad0 * __sinf(a0); n[2] = rad1 * __cosf(a1); n[3] = rad1 * __sinf(a1);
}
// One parameter.  g = d(data term)/d theta, (m, sg) = (mu, sigma), zt = this step's zeta, z1 = the next step's.
// VAEB.py:359-363 (thetaPrior), :391-393 (its gradient), :426-444 (Adagrad).  Returns theta' of the next step.
__device__ __forceinline__ float fvb_math(Ctx& c, const Hyper& hy, float g, float m, float sg, float am0, float as0, float zt,
                                         float z1, float& m1, float& s1, float& am, float& as) {
  c.tp += 0.5f * (1.0f + 0.6931471805599453f * fast_lg2(sg * sg) - m * m - sg * sg);
  const float sn = (sg > 0.f) ? 1.f : ((sg < 0.f) ? -1.f : 0.f);
  const float gm = g - m - hy.prior * m;
  const float gs = fast_rcp(sg) - sg - hy.prior * sg + g * zt * sn;
  am = am0 + gm * gm; as = as0 + gs * gs;
  m1 = m + hy.lr * gm * fast_rcp(fast_sqrt(am) + hy.eps);
  s1 = sg + hy.lr * gs * fast_rcp(fast_sqrt(as) + hy.eps);
  return m1 + fabsf(s1) * z1;
}
// scalar form (the thin tensors, whose rows are not 16-byte aligned runs): one Philox group per parameter
__device__ __forceinline__ float fvb_element(Ctx& c, const Params& p, const Hyper& hy, long long o, float g, float m, float sg,
                                             float am0, float as0, float zt) {
  float zn[4];
  zeta_group(p, c.step + 1u, (uint64_t)o >> 2, zn);
  const uint32_t q = (uint32_t)o & 3u;
  const float z1 = q == 0 ? zn[0] : (q == 1 ? zn[1] : (q == 2 ? zn[2] : zn[3]));
  float m1, s1, am, as;
  const float th = fvb_math(c, hy, g, m, sg, am0, as0, zt, z1, m1, s1, am, as);
  p.vmu[o] = m1; p.vsig[o] = s1; p.ada_mu[o] = am; p.ada_sig[o] = as; p.zeta[o] = z1;
  return th;
}

template <int N>
struct WgPre {                                                     // parameters / accumulators of phase B, loaded early
  static constexpr int RPP = 32 / N, NP = 8 / RPP;                 // rows per warp pass; passes (a warp owns 8 rows)
  long long o[NP]; float pv[NP], av[NP];
};
// issue the phase-B loads (they do not depend on the GEMM): called BEFORE waiting for the operands and the MMAs
// vec4 (sampled full VB, N = 32, rows of the tensor are 16-byte aligned runs): a thread owns FOUR consecutive
// parameters = one Philox group, 16-byte accesses; pv / av then hold (mu, sigma) of its two groups, o their offsets.
// SV: the sampled-weights full-VB instantiation of the kernel (its epilogues need ~30 more registers: kept out of the
// code of the plain step)
template <int N, bool SV, class OffF>
__device__ __forceinline__ void wgrad_prefetch(Ctx& c, const Params& p, OffF off, WgPre<N>& w, bool vec4 = false) {
  if (SV && N == 32 && vec4) {
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {
      const int row = c.warp * 8 + ps * 4 + (c.lane >> 3), col = (c.lane & 7) * 4;
      const long long o = off(row, col);
      w.o[ps] = o;
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 m4 = o >= 0 ? __ldcg(reinterpret_cast<const float4*>(p.vmu + o)) : z4;
      const float4 s4 = o >= 0 ? __ldcg(reinterpret_cast<const float4*>(p.vsig + o)) : z4;
      w.pv[ps * 4] = m4.x; w.pv[ps * 4 + 1] = m4.y; w.pv[ps * 4 + 2] = m4.z; w.pv[ps * 4 + 3] = m4.w;
      w.av[ps * 4] = s4.x; w.av[ps * 4 + 1] = s4.y; w.av[ps * 4 + 2] = s4.z; w.av[ps * 4 + 3] = s4.w;
    }
    return;
  }
  const int col = c.lane % N, rsub = c.lane / N;
#pragma unroll
  for (int r = 0; r < WgPre<N>::NP; ++r) {
    const int row = c.warp * 8 + r * WgPre<N>::RPP + rsub;
    w.o[r] = off(row, col);
    w.pv[r] = w.o[r] >= 0 ? __ldcg((SV ? p.vmu : p.P) + w.o[r]) : 0.f;       // sampled full VB: (mu, sigma)
    w.av[r] = w.o[r] >= 0 ? __ldcg((SV ? p.vsig : p.ada) + w.o[r]) : 0.f;
  }
}
template <int N, bool SV, class MirF>
__device__ __forceinline__ void wgrad_epilogue_coalesced(Ctx& c, const Params& p, const Hyper& hy, const WgPre<N>& w, MirF mir,
                                                         bool vec4 = false) {
  // (every weight-gradient GEMM has a delta operand: the two accumulators are combined while they are parked)
  constexpr int GP = 33;
  float* gt = reinterpret_cast<float*>(c.sm + SM_RECV);            // 128 x 33 floats = 16.5 KB (no cluster item is active)
  const int q = c.warp & 3;
  for (int u = c.warp >> 2; u < N / 8; u += 4) {
    float v[8];
    acc_ld8(c, q, (uint32_t)(u * 8), v, true);
#pragma unroll
    for (int e = 0; e < 8; ++e) gt[(q * 32 + c.lane) * GP + u * 8 + e] = v[e];
  }
  tc::tc_fence_before();
  __syncthreads();
  if (SV && N == 32 && vec4) {
    // sampled full VB, one Philox group per thread and pass (see wgrad_prefetch)
    float4 am4[2], as4[2], zt4[2];
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {                               // every load before the first store
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const long long o = w.o[ps];
      am4[ps] = o >= 0 ? __ldcg(reinterpret_cast<const float4*>(p.ada_mu + o)) : z4;
      as4[ps] = o >= 0 ? __ldcg(reinterpret_cast<const float4*>(p.ada_sig + o)) : z4;
      zt4[ps] = o >= 0 ? __ldcg(reinterpret_cast<const float4*>(p.zeta + o)) : z4;
    }
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {
      const long long o = w.o[ps];
      if (o >= 0) {
        const int row = c.warp * 8 + ps * 4 + (c.lane >> 3), col = (c.lane & 7) * 4;
        float zn[4], m1[4], s1[4], am[4], as[4], th[4];
        zeta_group(p, c.step + 1u, (uint64_t)o >> 2, zn);
        const float a0[4] = {am4[ps].x, am4[ps].y, am4[ps].z, am4[ps].w}, b0[4] = {as4[ps].x, as4[ps].y, as4[ps].z, as4[ps].w};
        const float z0[4] = {zt4[ps].x, zt4[ps].y, zt4[ps].z, zt4[ps].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          th[j] = fvb_math(c, hy, gt[row * GP + col + j] * hy.w, w.pv[ps * 4 + j], w.av[ps * 4 + j], a0[j], b0[j], z0[j], zn[j],
                           m1[j], s1[j], am[j], as[j]);
          gt[row * GP + col + j] = th[j];
        }
        *reinterpret_cast<float4*>(p.vmu + o) = make_float4(m1[0], m1[1], m1[2], m1[3]);
        *reinterpret_cast<float4*>(p.vsig + o) = make_float4(s1[0], s1[1], s1[2], s1[3]);
        *reinterpret_cast<float4*>(p.ada_mu + o) = make_float4(am[0], am[1], am[2], am[3]);
        *reinterpret_cast<float4*>(p.ada_sig + o) = make_float4(as[0], as[1], as[2], as[3]);
        *reinterpret_cast<float4*>(p.zeta + o) = make_float4(zn[0], zn[1], zn[2], zn[3]);
        *reinterpret_cast<float4*>(p.P + o) = make_float4(th[0], th[1], th[2], th[3]);
      }
    }
  } else if (SV) {
    const int col = c.lane % N, rsub = c.lane / N;
    float am0[WgPre<N>::NP], as0[WgPre<N>::NP], zt[WgPre<N>::NP];
#pragma unroll
    for (int r = 0; r < WgPre<N>::NP; ++r) {                       // every load before the first store
      const bool ok = w.o[r] >= 0;
      am0[r] = ok ? __ldcg(p.ada_mu + w.o[r]) : 0.f;
      as0[r] = ok ? __ldcg(p.ada_sig + w.o[r]) : 0.f;
      zt[r] = ok ? __ldcg(p.zeta + w.o[r]) : 0.f;
    }
#pragma unroll
    for (int r = 0; r < WgPre<N>::NP; ++r) {
      const int row = c.warp * 8 + r * WgPre<N>::RPP + rsub;
      if (w.o[r] >= 0) {
        const float nv = fvb_element(c, p, hy, w.o[r], gt[row * GP + col] * hy.w, w.pv[r], w.av[r], am0[r], as0[r], zt[r]);
        p.P[w.o[r]] = nv;
        gt[row * GP + col] = nv;
      }
    }
  } else {
    const int col = c.lane % N, rsub = c.lane / N;
#pragma unroll
    for (int r = 0; r < WgPre<N>::NP; ++r) {
      const int row = c.warp * 8 + r * WgPre<N>::RPP + rsub;
      if (w.o[r] >= 0) {
        const float gg = fmaf(gt[row * GP + col], hy.w, -hy.prior * w.pv[r]);  // VAEB.py:389-390
        const float a = w.av[r] + gg * gg;                         // VAEB.py:439
        float nv = w.pv[r] + hy.lr * gg / (sqrtf(a) + hy.eps);     // VAEB.py:441
        if (hy.p2 != 0.f) nv -= hy.p2 * w.pv[r] * w.pv[r];         // VAEBfullbayes.py:183-184
        p.P[w.o[r]] = nv;
        p.ada[w.o[r]] = a;
        gt[row * GP + col] = nv;
      }
    }
  }
  __syncthreads();
  for (int u = c.warp >> 2; u < N / 8; u += 4) {
    float nv[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) nv[e] = gt[(q * 32 + c.lane) * GP + u * 8 + e];
    mir(q * 32 + c.lane, u * 8, nv);
  }
  __syncthreads();
}

// W2, b2 <- Adagrad([h_d | 1]^T . da2); tile = 128 hidden units x 32 pixels.  Gaussian decoder: `which` = 1 selects
// the W6 / b6 half of the tile (rows 32..63 of the transposed delta mirror, virtual columns 32..63 of the chunk).
template <bool SV>
__device__ __forceinline__ void item_wg2(Ctx& c, const Params& p, const Hyper& hy, int mt, int nt, int which) {
  constexpr int TB = 32 * 128;                                  // the B tile of the item: 32 rows
  const int TBM = p.TR3 * 128;                                  // one half (hi or lo) of a delta-mirror tile
  if (threadIdx.x == 0) {
    ops_begin(c, (uint32_t)(4 * TBA + 4 * TB));
    bulk_g2s(c.sm + SM_A, p.hd_t + (size_t)mt * 4 * TBA, (uint32_t)(4 * TBA), c.op_bar);
    const uint8_t* src = p.da2_t + (size_t)nt * 4 * TBM + (size_t)which * TB;
#pragma unroll
    for (int q = 0; q < 4; ++q)                                 // (batch chunk, hi / lo): 32 rows of each
      bulk_g2s(c.sm + SM_B + q * TB, src + (size_t)q * TBM, (uint32_t)TB, c.op_bar);
  }
  const int H = p.H, D = p.D;
  const long long oW = which ? p.oW6 : p.oW2, ob = which ? p.ob6 : p.ob2;
  WgPre<32> pre;
  const bool vec4 = SV && ((oW | ob | (long long)D) & 3) == 0;     // rows are 16-byte aligned runs
  wgrad_prefetch<32, SV>(c, p, [&](int row, int col) -> long long {
    const int i = mt * MP + row, n = nt * 32 + col;
    if (i > H || n >= D) return -1;
    return i < H ? oW + (long long)i * D + n : ob + n;
  }, pre, vec4);
  mma_run(c, 2, (p.M + 15) / 16, TB, 32, true, 0u, 0, 1);
  wgrad_epilogue_coalesced<32, SV>(
      c, p, hy, pre,
      [&](int row, int col0, float* nv) {
        const int i = mt * MP + row, n0 = nt * 32 + col0;
        if (i >= H || n0 >= D) return;
        const int vr = which * 32 + col0;                        // row of the dec2 tile = virtual column inside the chunk
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (n0 + e < D) mirror_put(p.m_dec2, p.TR3, p.KH, nt, vr + e, i, nv[e]);
          else nv[e] = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) nv[e] *= WSCALE;
        // dgrad mirror: row = hidden unit i, k = (virtual) output column: eight consecutive k = one 16-byte unit
        constexpr int TG = TR_DGRAD * 128;
        const int kv = p.cont ? nt * 64 + vr : n0;
        put_unit<true>(p.m_dgrad + ((size_t)(i >> 4) * p.KV + (kv >> 6)) * 2 * TG + unit_off(i & 15, (kv & 63) >> 3), TG, nv);
      }, vec4);
}

// W3, b3 <- Adagrad([x | 1]^T . da3), da3 = ([dmu|dls].[W4|W5]^T) * (1 - h_e^2) recomputed on the tensor cores (K = one
// chunk) and written, transposed, into the B tile; tile = 128 pixels x 32 hidden units
template <bool SV>
__device__ __forceinline__ void item_wg3(Ctx& c, const Params& p, const Hyper& hy, const float* he, int mt, int nt, int par) {
  const int H = p.H, M = p.M, D = p.D;
  constexpr int TB = 32 * 128;                                  // one half (hi or lo) of a 32-row tile
  uint8_t* dd_sm = c.sm + SM_A + 2 * 2 * TBA;                   // [dmu|dls]: the chunk slot behind the two chunks of x^T
  uint8_t* w45_sm = c.sm + SM_B + 16384;                        // this tile's rows of [W4|W5] behind the B tile
  if (threadIdx.x == 0) {
    ops_begin(c, (uint32_t)(4 * TBA + 2 * TBA + 2 * TB));
    bulk_g2s(dd_sm, p.dd_km, (uint32_t)(2 * TBA), c.op_bar);
    bulk_g2s(w45_sm, p.m_w45k + (size_t)par * p.w45k_bytes + (size_t)nt * 2 * TB, (uint32_t)(2 * TB), c.op_bar);
    bulk_g2s(c.sm + SM_A, p.x_t + (size_t)mt * 4 * TBA, (uint32_t)(4 * TBA), c.op_bar);
  }
  // this thread's share of the tanh' factors: batch row = TMEM lane, eight hidden units
  const int q = c.warp & 3, cg = c.warp >> 2;
  const int b = q * 32 + c.lane, j0 = nt * 32 + cg * 8;
  float hv[8];
  {
    const bool ok = b < M;
    const float4 h0 = ok ? __ldcg(reinterpret_cast<const float4*>(he + (size_t)b * p.HP + j0)) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 h1 = ok ? __ldcg(reinterpret_cast<const float4*>(he + (size_t)b * p.HP + j0 + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    hv[0] = h0.x; hv[1] = h0.y; hv[2] = h0.z; hv[3] = h0.w; hv[4] = h1.x; hv[5] = h1.y; hv[6] = h1.z; hv[7] = h1.w;
  }
  WgPre<32> pre;
  const bool vec4 = SV && ((p.oW3 | p.ob3 | (long long)H) & 3) == 0;   // rows are 16-byte aligned runs
  wgrad_prefetch<32, SV>(c, p, [&](int row, int col) -> long long {
    const int i = mt * MP + row, jc = nt * 32 + col;
    if (i > D || jc >= H) return -1;
    return i < D ? p.oW3 + (long long)i * H + jc : p.ob3 + jc;
  }, pre, vec4);
  // ---- dh_e pre-activation on the tensor cores: D1[128 x 32] = [dmu|dls] . [W4|W5]^T (tile rows) -----------------
  tc::tc_fence_before();
  __syncthreads();                                              // the previous item's TMEM reads are complete
  tc::tc_fence_after();
  if (threadIdx.x == 0) {
    tc::mbar_wait(c.op_bar, c.op_phase);
    c.op_phase ^= 1u;
    tc::tc_fence_after();
    const uint32_t idesc = tc::make_idesc_f16(MP, 32, 0, 0);    // A = a delta tensor: H products at +96, L product at +64
    const uint64_t d0 = tc::make_smem_desc(0u, 16u, 1024u);
    const uint64_t a = d0 | (uint64_t)(tc::smem_u32(dd_sm) >> 4), bdesc = d0 | (uint64_t)(tc::smem_u32(w45_sm) >> 4);
    const uint32_t a_lo = TBA >> 4, b_lo = TB >> 4;
    const int ks = (2 * p.Z + 15) / 16;
    for (int k = 0; k < ks; ++k) {
      tc::umma_bf16(c.tmem + 96u, a + 2 * k, bdesc + 2 * k, idesc, k ? 1u : 0u);
      tc::umma_bf16(c.tmem + 96u, a + 2 * k, bdesc + b_lo + 2 * k, idesc, 1u);
      tc::umma_bf16(c.tmem + 64u, a + a_lo + 2 * k, bdesc + 2 * k, idesc, k ? 1u : 0u);
    }
    tc::umma_commit(c.mma_bar);
  }
  tc::mbar_wait(c.mma_bar, c.mma_phase);
  c.mma_phase ^= 1u;
  tc::tc_fence_after();
  {
    float v[8], vh[8];
    tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + 64u + (uint32_t)(cg * 8), v);
    tmem_ld8(c.tmem + ((uint32_t)(q * 32) << 16) + 96u + (uint32_t)(cg * 8), vh);
    tc::tmem_ld_wait();
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = fmaf(vh[e], DSCALE, v[e]);
    // B tile of the weight gradient: row = hidden unit, k = batch row -> 2-byte stores, a warp writes 64 contiguous bytes
    uint8_t* bt = c.sm + SM_B + (size_t)(b >> 6) * 2 * TB;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float d = (b < M && j0 + e < H) ? v[e] * WUNSCALE * (1.0f - hv[e] * hv[e]) : 0.f;
      put_dl(bt + tc::sw128_offset(cg * 8 + e, b & 63), TB, d);
    }
  }
  mma_run(c, 2, (M + 15) / 16, TB, 32, false, 0u, 0, 1);
  wgrad_epilogue_coalesced<32, SV>(
      c, p, hy, pre,
      [&](int row, int col0, float* nv) {
        const int i = mt * MP + row, j0_ = nt * 32 + col0;
        if (i >= D) return;
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (j0_ + e < H) mirror_put(p.m_enc1, TR_ENC1, p.KD, (j0_ + e) >> 4, (j0_ + e) & 15, i, nv[e]);
      }, vec4);
}

// W1, b1 <- Adagrad([z | 1]^T . da1), computed transposed: tile = 128 hidden units x (Z + 1) latent columns.  W1 is
// [Z][H]: with the thread = hidden unit mapping of the accumulator every access below is coalesced along the lanes.
template <bool SV>
__device__ __forceinline__ void item_wg1(Ctx& c, const Params& p, const Hyper& hy, int mt) {
  const int Z = p.Z, H = p.H, N = p.NZ;
  const int TB = N * 128;
  if (threadIdx.x == 0) {
    ops_begin(c, (uint32_t)(4 * TBA + 4 * TB));
    bulk_g2s(c.sm + SM_A, p.da1_t + (size_t)mt * 4 * TBA, (uint32_t)(4 * TBA), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.z_t, (uint32_t)(4 * TB), c.op_bar);
  }
  // this thread's unit: hidden unit i, latent columns col0 .. col0 + 7 (column Z = the bias); loads before the GEMM
  const int qq = c.warp & 3, u = c.warp >> 2;
  const int i = mt * MP + qq * 32 + c.lane, col0 = u * 8;
  const bool mine = u < N / 8 && i < H && col0 <= Z;
  size_t off[8]; bool ok[8]; float pv[8], av[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int q = col0 + e;
    ok[e] = mine && q <= Z;
    off[e] = q < Z ? (size_t)p.oW1 + (size_t)q * H + i : (size_t)p.ob1 + i;
    pv[e] = ok[e] ? __ldcg((SV ? p.vmu : p.P) + off[e]) : 0.f;
    av[e] = ok[e] ? __ldcg((SV ? p.vsig : p.ada) + off[e]) : 0.f;
  }
  mma_run(c, 2, (p.M + 15) / 16, TB, N, true, 0u, 1, 0);
  if (u < N / 8) {
    float v[8], nv[8];
    acc_ld8(c, qq, (uint32_t)col0, v, true);
    if (SV && mine) {
      float am0[8], as0[8], zt[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        am0[e] = ok[e] ? __ldcg(p.ada_mu + off[e]) : 0.f;
        as0[e] = ok[e] ? __ldcg(p.ada_sig + off[e]) : 0.f;
        zt[e] = ok[e] ? __ldcg(p.zeta + off[e]) : 0.f;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        nv[e] = 0.f;
        if (ok[e]) {
          nv[e] = fvb_element(c, p, hy, (long long)off[e], v[e] * hy.w, pv[e], av[e], am0[e], as0[e], zt[e]);
          p.P[off[e]] = nv[e];
          if (col0 + e < Z) mirror_put(p.m_dz, N, p.KH, 0, col0 + e, i, nv[e]);
        }
      }
      constexpr int T1 = 64 * 128;
#pragma unroll
      for (int e = 0; e < 8; ++e) nv[e] *= WSCALE;
      put_unit<true>(p.m_dec1 + (size_t)(i >> 6) * 2 * T1 + unit_off(i & 63, col0 >> 3), T1, nv);
    } else if (mine) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        nv[e] = 0.f;
        if (ok[e]) {
          const float gg = fmaf(v[e], hy.w, -hy.prior * pv[e]);   // VAEB.py:389-390
          const float a = av[e] + gg * gg;                        // VAEB.py:439
          float n_ = pv[e] + hy.lr * gg / (sqrtf(a) + hy.eps);    // VAEB.py:441
          if (hy.p2 != 0.f) n_ -= hy.p2 * pv[e] * pv[e];          // VAEBfullbayes.py:183-184
          p.P[off[e]] = n_;
          p.ada[off[e]] = a;
          nv[e] = n_;
          if (col0 + e < Z) mirror_put(p.m_dz, N, p.KH, 0, col0 + e, i, n_);
        }
      }
      // [W1^T | b1] of the decoder hidden layer: row = hidden unit, the eight latent columns are one 16-byte unit
      constexpr int T1 = 64 * 128;
#pragma unroll
      for (int e = 0; e < 8; ++e) nv[e] *= WSCALE;
      put_unit<true>(p.m_dec1 + (size_t)(i >> 6) * 2 * T1 + unit_off(i & 63, col0 >> 3), T1, nv);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
}

// W4, b4, W5, b5 <- Adagrad([h_e | 1]^T . [dmu | dls]); tile = 128 hidden units x 16 columns of [dmu | dls]
template <bool SV>
__device__ __forceinline__ void item_wg45(Ctx& c, const Params& p, const Hyper& hy, int mt, int nt, int par) {
  const int Z = p.Z, H = p.H;
  constexpr int N = 16, TB = N * 128;
  if (threadIdx.x == 0) {
    ops_begin(c, (uint32_t)(4 * TBA + 4 * TB));
    bulk_g2s(c.sm + SM_A, p.he_t + (size_t)mt * 4 * TBA, (uint32_t)(4 * TBA), c.op_bar);
    bulk_g2s(c.sm + SM_B, p.dd_t + (size_t)nt * 4 * TB, (uint32_t)(4 * TB), c.op_bar);
  }
  WgPre<N> pre;
  wgrad_prefetch<N, SV>(c, p, [&](int row, int col) -> long long {
    const int i = mt * MP + row, cc = nt * N + col;
    if (i > H || cc >= 2 * Z) return -1;
    const int jc = cc < Z ? cc : cc - Z;
    if (i < H) return (cc < Z ? p.oW4 : p.oW5) + (long long)i * Z + jc;
    return (cc < Z ? p.ob4 : p.ob5) + jc;
  }, pre);
  mma_run(c, 2, (p.M + 15) / 16, TB, N, true, 0u, 0, 1);
  wgrad_epilogue_coalesced<N, SV>(
      c, p, hy, pre,
      [&](int row, int col0, float* nv) {
        const int i = mt * MP + row, cc0 = nt * N + col0;
        if (i >= H) return;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if (cc0 + e < 2 * Z) mirror_put(p.m_heads, p.NH, p.KH, 0, cc0 + e, i, nv[e]);
          nv[e] = cc0 + e < 2 * Z ? nv[e] * WSCALE : 0.f;
        }
        // the copy the NEXT step's dh_e GEMMs read (row = hidden unit, k = column of [dmu|dls]: one 16-byte unit)
        constexpr int T32 = 32 * 128;
        put_unit<true>(p.m_w45k + (size_t)(par ^ 1) * p.w45k_bytes + (size_t)(i >> 5) * 2 * T32 + unit_off(i & 31, cc0 >> 3), T32, nv);
      });
}

// noise of the step: eps[M, Z] ~ N(0, 1) from Philox (VAEB.py:42's srng.normal, on the device); one CTA per quarter
__device__ __forceinline__ void item_eps(const Params& p, uint32_t step, int part) {
  const int e = part * NT + threadIdx.x;
  if (e < p.M * p.Z)
    p.eps[e] = philox_normal1(p.seed, VAEB_STREAM_TRAIN, step, 0u, (uint64_t)(p.row_offset * p.Z + e));
  if (part == 0)
    for (int e2 = CL * NT + threadIdx.x; e2 < p.M * p.Z; e2 += NT)
      p.eps[e2] = philox_normal1(p.seed, VAEB_STREAM_TRAIN, step, 0u, (uint64_t)(p.row_offset * p.Z + e2));
}

// the bound of step s: fixed-order sum of the row partials (VAEB.py:340-344) / Mg
__device__ __forceinline__ void item_bound(Ctx& c, const Params& p, int s) {
  float* red = reinterpret_cast<float*>(c.sm + SM_MISC + 256);
  float t = 0.f;
  for (int r = threadIdx.x; r < p.M; r += NT) {
    float rs = __ldcg(p.aux + r);
    for (int q = 0; q < p.n_tiles3; ++q) rs += __ldcg(p.partial + (size_t)r * p.n_tiles3 + q);
    t += rs;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  __syncthreads();
  if (c.lane == 0) red[c.warp] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = 0.f;
    for (int w = 0; w < NT / 32; ++w) b += red[w];
    float tp = 0.f;                                  // thetaPrior (full VB), fixed order
    if (p.fvb) {
      const float* part = p.tprior_part + (size_t)(s & 1) * gridDim.x;
      for (int q = 0; q < (int)gridDim.x; ++q) tp += __ldcg(part + q);
    }
    p.scalars[s] = (p.bmult * b + tp) / p.Mg;        // VAEB.py:364,412
  }
  __syncthreads();
}

// this CTA's partial sum of thetaPrior (fixed order) into the step's half of tprior_part
__device__ __forceinline__ void store_tprior(Ctx& c, const Params& p, int s, float tp) {
  float* red = reinterpret_cast<float*>(c.sm + SM_MISC + 256);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tp += __shfl_xor_sync(0xffffffffu, tp, o);
  __syncthreads();
  if (c.lane == 0) red[c.warp] = tp;
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = 0.f;
    for (int w = 0; w < NT / 32; ++w) b += red[w];
    p.tprior_part[(size_t)(s & 1) * gridDim.x + blockIdx.x] = b;
  }
  __syncthreads();
}

// Full VB, reference-faithful: thetaPrior (VAEB.py:359-363) and the whole (mu, sigma) update in one pass over the flat
// buffers -- d/dmu = -mu - prior mu, d/dsigma = 1/s - s - prior s (VAEB.py:391-393), Adagrad (:426-444)
// part / nparts: this CTA's share (the CTAs of cluster 0 run the latent heads meanwhile and contribute 0)
__device__ __forceinline__ void item_fvb_prior(Ctx& c, const Params& p, const Hyper& hy, int s, int part, int nparts) {
  float tp = 0.f;
  for (int64_t g4 = (int64_t)part * NT + threadIdx.x; part >= 0 && 4 * g4 < p.total; g4 += (int64_t)nparts * NT) {
    float4 m4 = __ldcg(reinterpret_cast<const float4*>(p.vmu) + g4);
    float4 s4 = __ldcg(reinterpret_cast<const float4*>(p.vsig) + g4);
    float4 am4 = __ldcg(reinterpret_cast<const float4*>(p.ada_mu) + g4);
    float4 as4 = __ldcg(reinterpret_cast<const float4*>(p.ada_sig) + g4);
    float* mm = &m4.x; float* ss = &s4.x; float* am = &am4.x; float* as = &as4.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (4 * g4 + j < p.total) {
        const float m = mm[j], sg = ss[j];
        tp += 0.5f * (1.0f + logf(sg * sg) - m * m - sg * sg);
        const float gm = -m - hy.prior * m, gs = 1.0f / sg - sg - hy.prior * sg;
        am[j] += gm * gm; as[j] += gs * gs;
        mm[j] = m + hy.lr * gm / (sqrtf(am[j]) + hy.eps);
        ss[j] = sg + hy.lr * gs / (sqrtf(as[j]) + hy.eps);
      }
    }
    reinterpret_cast<float4*>(p.vmu)[g4] = m4;
    reinterpret_cast<float4*>(p.vsig)[g4] = s4;
    reinterpret_cast<float4*>(p.ada_mu)[g4] = am4;
    reinterpret_cast<float4*>(p.ada_sig)[g4] = as4;
  }
  store_tprior(c, p, s, tp);
}

// =================================================================================================================
template <bool SV>
__global__ void __launch_bounds__(NT, 1) step_tc_kernel(const __grid_constant__ Params p) {
  Ctx c;
  c.sm = smem_base();
  c.mma_bar = reinterpret_cast<uint64_t*>(c.sm + SM_MISC);
  c.op_bar = c.mma_bar + 1;
  c.x_bar = c.mma_bar + 3;
  c.rs_bar = c.mma_bar + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(c.sm + SM_MISC + 16);
  c.mma_phase = 0; c.op_phase = 0; c.x_phase = 0; c.rs_phase = 0;
  c.rank = (int)cluster_ctarank(); c.cid = (int)cluster_idx(); c.ncl = (int)cluster_count();
  c.warp = threadIdx.x >> 5; c.lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tc::mbar_init(c.mma_bar, 1);
    tc::mbar_init(c.op_bar, 1);
    tc::mbar_init(c.x_bar, 1);
    tc::mbar_init(c.rs_bar, 1);
    tc::fence_barrier_init();
  }
  if (c.warp == 1) tc::tmem_alloc(tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  c.tmem = *tmem_slot;
  cluster_sync();                                   // every CTA of the cluster is resident before any remote store

  const int G = gridDim.x;
  unsigned long long target = p.bar_base;
  const Hyper hy{p.lr, p.ada_eps, p.prior, p.p2, p.w};
  const bool rec = p.timing != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  const int n1 = p.HP / 16;                         // enc1 / dgrad tiles
  const int n3 = p.n_tiles3;                        // dec2 tiles
  const int m_h1 = (p.H + 1 + MP - 1) / MP;         // 128-row tiles over the hidden units + the ones row
  const int m_h = (p.H + MP - 1) / MP;
  const int m_d1 = (p.D + 1 + MP - 1) / MP;
  const int n_h32 = p.HP / 32;
  const int n3w = m_d1 * n_h32;                     // W3 gradient tiles
  const int n45t = p.NH / 16;                       // 16-column tiles of [dmu|dls] in the W4/W5 gradient
  // a phase's item list: cluster items first, then CTA items in groups of four (one per rank of a cluster)
  auto n_groups = [](int n_cta_items) { return (n_cta_items + CL - 1) / CL; };
  auto x_of = [&](int s) { return p.batch_order ? p.x_base + (size_t)__ldg(p.batch_order + s) * p.M * p.D : p.x_direct; };
  const int kd0 = c.rank * p.KD / CL, kdn = (c.rank + 1) * p.KD / CL - kd0;

  // the A tile of this CTA's first enc1 item: converted from the fp32 rows for the first step of a launch (x depends
  // on nothing), one bulk copy of x_km -- issued before the barrier that closes the previous step -- afterwards
  const bool has_p1 = c.cid < n1;
  if (has_p1) stage_x_rows(c.sm, x_of(0), p.D, p.M, kd0, kdn);
  const int n_spare = c.ncl - n3;                   // clusters without a dec2 item: they publish h_d in P3
  int last_done = -1;                               // last step whose updates were applied (a Gaussian launch may stop early)

  for (int s = 0; s < p.n_steps; ++s) {
    const float* x = x_of(s);
    const int par = (p.w45_par0 + s) & 1;                        // which copy of the k-major [W4|W5] mirror this step reads
    c.step = p.step0 + (uint32_t)s; c.tp = 0.f;
    // sampled full VB: the bound of the previous step needs the thetaPrior sums of ITS update epilogues (P5, P6): it is
    // summed here, by a CTA that has no enc1 item, before P2 / P3 overwrite the row partials
    if (SV && s > 0 && (int)blockIdx.x == G - 1) item_bound(c, p, s - 1);
    long long* tm = rec ? p.timing + (size_t)s * (N_PHASES + 1) : nullptr;
    if (tm) tm[0] = gtime();

    // ---- P1: encoder hidden layer | this step's noise ----------------------------------------------------------
    {
      const int n_e = p.eps_inj ? 0 : CL;
      for (int it = c.cid; it < n1 + n_groups(n_e); it += c.ncl) {
        if (it < n1) {
          const int mode = it == c.cid ? (s == 0 ? A_STAGED : A_PREFETCHED) : (s == 0 ? A_SOFTWARE : A_BULK);
          item_enc1(c, p, x, p.he, p.he_t, it, mode, it + c.ncl < n1);
          continue;
        }
        item_eps(p, p.step0 + (uint32_t)s, c.rank);
      }
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[1] = gtime();
    // ---- P2: latent heads | the minibatch operands of P6 and of the next step's P1 ---------------------------------
    if (c.cid == 0) item_heads(c, p, p.step0 + (uint32_t)s, false);
    else item_xmirrors(p, s + 1 < p.n_steps ? x_of(s + 1) : nullptr, x, (c.cid - 1) * CL + c.rank, (c.ncl - 1) * CL);
    if (p.fvb == 1) item_fvb_prior(c, p, hy, s, c.cid == 0 ? -1 : (c.cid - 1) * CL + c.rank, (c.ncl - 1) * CL);   // nothing downstream reads (mu, sigma)
    grid_barrier(p.bar, target += G);
    if (tm) tm[2] = gtime();
    // ---- P3: decoder + log-likelihood | h_d published by the spare clusters ------------------------------------------
    for (int it = c.cid; it < n3; it += c.ncl) item_dec2(c, p, x, it, it + c.ncl < n3, n_spare <= 0, s);
    if (c.cid >= n3)
      for (int g = (c.cid - n3) * CL + c.rank; g < p.HP / 16; g += n_spare * CL) item_hd(c, p, g);
    grid_barrier(p.bar, target += G);
    if (tm) tm[3] = gtime();
    if (p.fvb == 1) {
      // reference-faithful full VB: the bound is all the layers are needed for.  One CTA (rotating) sums it; the
      // partials it reads are overwritten two barriers into the next step at the earliest.
      if ((int)blockIdx.x == (c.ncl > n1 ? G - 1 - (s & 3) : s % G)) item_bound(c, p, s);   // a CTA without an enc1 item
      if (s + 1 < p.n_steps && has_p1 && threadIdx.x == 0 && kdn > 0) {
        tc::mbar_expect_tx(c.x_bar, (uint32_t)(kdn * 2 * TBA));
        bulk_g2s(c.sm + SM_A, p.x_km + (size_t)kd0 * 2 * TBA, (uint32_t)(kdn * 2 * TBA), c.x_bar);
      }
      continue;
    }
    // ---- P4: back through the decoder output layer ---------------------------------------------------------------
    for (int it = c.cid; it < n1; it += c.ncl) item_dgrad(c, p, it, it + c.ncl < n1, s);
    grid_barrier(p.bar, target += G);
    if (tm) tm[4] = gtime();
    // Gaussian decoder: a delta left the operand range -> every CTA leaves before the first parameter update of step s
    if (p.cont && __syncthreads_or(threadIdx.x == 0 && __ldcg(p.status) >= 0)) break;
    // ---- P5: dz | W2 update | the bound ---------------------------------------------------------------------------
    {
      const int nw = p.cont ? 2 : 1;                              // Gaussian decoder: W2 and W6
      const int n2 = m_h1 * n3 * nw;
      const int g2 = n_groups(n2 + 1);
      for (int it = c.cid; it < 1 + g2; it += c.ncl) {
        if (it == 0) { item_dz(c, p, false, p.kl_beta ? __ldg(p.kl_beta + s) : 1.f); continue; }
        const int i = (it - 1) * CL + c.rank;
        if (i < n2) item_wg2<SV>(c, p, hy, i / (n3 * nw), (i / nw) % n3, i % nw);
        else if (i == n2 && !SV) item_bound(c, p, s);
      }
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[5] = gtime();
    // ---- P6: W3 update | W1 update | W4, W5 update -----------------------------------------------------------------
    {
      const int n45 = m_h1 * n45t;
      for (int it = c.cid; it < n_groups(n3w + m_h + n45); it += c.ncl) {
        const int i = it * CL + c.rank;
        if (i < n3w) item_wg3<SV>(c, p, hy, p.he, i / n_h32, i % n_h32, par);
        else if (i < n3w + m_h) item_wg1<SV>(c, p, hy, i - n3w);
        else if (i < n3w + m_h + n45) item_wg45<SV>(c, p, hy, (i - n3w - m_h) / n45t, (i - n3w - m_h) % n45t, par);
      }
    }
    if (SV) store_tprior(c, p, s, c.tp);
    // the A tile of this CTA's first enc1 item of the next step (x_km was written in P2): in flight across the barrier
    if (s + 1 < p.n_steps && has_p1 && threadIdx.x == 0 && kdn > 0) {
      tc::mbar_expect_tx(c.x_bar, (uint32_t)(kdn * 2 * TBA));
      bulk_g2s(c.sm + SM_A, p.x_km + (size_t)kd0 * 2 * TBA, (uint32_t)(kdn * 2 * TBA), c.x_bar);
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[6] = gtime();
    last_done = s;
  }
  if (SV && last_done >= 0 && (int)blockIdx.x == G - 1) item_bound(c, p, last_done);
  tc::tc_fence_before();
  __syncthreads();
  cluster_sync();                                   // no CTA leaves while a peer may still write its shared memory
  if (c.warp == 1) tc::tmem_dealloc(c.tmem, TMEM_COLS);
}

// ---- mirrors from the fp32 master parameters (after set_tensors / load / an update by another path) ----------------
struct MirrorArgs {
  const float* P; int64_t oW3, oW4, oW5, oW1, oW2, ob1, oW6; int cont, TR3, KV;
  uint8_t *m_enc1, *m_heads, *m_dec2, *m_dgrad, *m_dz, *m_dec1, *m_w45k;
  int D, H, Z, HP, KD, KH, NH, NZ;
};
__global__ void __launch_bounds__(256) build_mirrors_kernel(MirrorArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int D = a.D, H = a.H, Z = a.Z;
  switch (blockIdx.y) {
    case 0: {   // enc1: n = hidden (HP rows), k = pixel (KD chunks)
      const int K = a.KD * 64;
      if (i >= (int64_t)a.HP * K) return;
      const int n = (int)(i / K), k = (int)(i % K);
      mirror_put(a.m_enc1, TR_ENC1, a.KD, n / TR_ENC1, n % TR_ENC1, k, (n < H && k < D) ? a.P[a.oW3 + (size_t)k * H + n] : 0.f);
      break;
    }
    case 1: {   // heads: n = [W4 cols | W5 cols] (NH rows), k = hidden
      const int K = a.KH * 64;
      if (i >= (int64_t)a.NH * K) return;
      const int n = (int)(i / K), k = (int)(i % K);
      float v = 0.f;
      if (k < H && n < 2 * Z) v = n < Z ? a.P[a.oW4 + (size_t)k * Z + n] : a.P[a.oW5 + (size_t)k * Z + n - Z];
      mirror_put(a.m_heads, a.NH, a.KH, 0, n, k, v);
      break;
    }
    case 2: {   // dec2: n = (virtual) output column (tiles of TR3), k = hidden
      const int K = a.KH * 64, NR = (D + 31) / 32 * a.TR3;
      if (i >= (int64_t)NR * K) return;
      const int n = (int)(i / K), k = (int)(i % K);
      const int r = n % a.TR3, px = (n / a.TR3) * 32 + (r & 31);           // r >= 32: the W6 half (Gaussian decoder)
      mirror_put(a.m_dec2, a.TR3, a.KH, n / a.TR3, r, k, (px < D && k < H) ? a.P[(r < 32 ? a.oW2 : a.oW6) + (size_t)k * D + px] : 0.f);
      break;
    }
    case 3: {   // dgrad: n = hidden (HP rows), k = (virtual) output column
      const int K = a.KV * 64;
      if (i >= (int64_t)a.HP * K) return;
      const int n = (int)(i / K), k = (int)(i % K);
      const int px = a.cont ? (k >> 6) * 32 + (k & 31) : k;
      const int64_t oW = (a.cont && (k & 32)) ? a.oW6 : a.oW2;
      mirror_put(a.m_dgrad, TR_DGRAD, a.KV, n / TR_DGRAD, n % TR_DGRAD, k, (n < H && px < D) ? a.P[oW + (size_t)n * D + px] : 0.f);
      break;
    }
    case 6: {   // [W4|W5] with the hidden unit as the row (tiles of 32), k = column of [dmu|dls]; both parity copies
      if (i >= (int64_t)a.HP * 64) return;
      const int n = (int)(i / 64), k = (int)(i % 64);
      float v = 0.f;
      if (n < H && k < 2 * Z) v = k < Z ? a.P[a.oW4 + (size_t)n * Z + k] : a.P[a.oW5 + (size_t)n * Z + k - Z];
      mirror_put(a.m_w45k, 32, 1, n >> 5, n & 31, k, v);
      mirror_put(a.m_w45k + (size_t)a.HP * 64 * 4, 32, 1, n >> 5, n & 31, k, v);
      break;
    }
    case 5: {   // dec1: n = hidden (tiles of 64), k = latent index, k = Z: the bias
      if (i >= (int64_t)a.HP * 64) return;
      const int n = (int)(i / 64), k = (int)(i % 64);
      float v = 0.f;
      if (n < H) v = k < Z ? a.P[a.oW1 + (size_t)k * H + n] : (k == Z ? a.P[a.ob1 + n] : 0.f);
      mirror_put(a.m_dec1, 64, 1, n >> 6, n & 63, k, v);
      break;
    }
    default: {  // dz: n = latent (NZ rows), k = hidden
      const int K = a.KH * 64;
      if (i >= (int64_t)a.NZ * K) return;
      const int n = (int)(i / K), k = (int)(i % K);
      mirror_put(a.m_dz, a.NZ, a.KH, 0, n, k, (n < Z && k < H) ? a.P[a.oW1 + (size_t)n * H + k] : 0.f);
      break;
    }
  }
}

// constant rows of the transposed activation mirrors: the "ones" feature that turns a weight-gradient GEMM's extra row /
// column into the bias gradient (h_e and h_d: feature H; z: feature Z).  Everything else starts as zero.
struct OnesArgs { uint8_t *he_t, *hd_t, *z_t, *z_km, *x_t; int H, Z, NZ, D; };
__global__ void __launch_bounds__(128) init_ones_kernel(OnesArgs a) {
  const int b = threadIdx.x;                       // batch column 0..127
  const __half one = __float2half_rn(1.0f);
  uint8_t* m[2] = {a.he_t, a.hd_t};
  for (int q = 0; q < 2; ++q)
    *reinterpret_cast<__half*>(t_addr(m[q], a.H >> 7, TBA, a.H & 127, b)) = one;
  *reinterpret_cast<__half*>(t_addr(a.z_t, 0, a.NZ * 128, a.Z, b)) = one;
  *reinterpret_cast<__half*>(km_addr(a.z_km, b, a.Z)) = one;      // [z | 1]: batch row b, column Z
  *reinterpret_cast<__half*>(t_addr(a.x_t, a.D >> 7, TBA, a.D & 127, b)) = one;   // [x | 1]^T: the row of pixel D
}

}  // namespace st2

// =====================================================================================================================
// host side
// =====================================================================================================================
void step_tc_free(StepTcState& s) {
  void* ptrs[] = {s.bar, s.m_enc1, s.m_heads, s.m_dec2, s.m_dgrad, s.m_dz, s.m_dec1, s.act, s.he, s.hd, s.mu, s.ls,
                  s.eps, s.z, s.m_w45k, s.partial, s.aux, s.d_timing, s.d_status, s.tprior_part};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  s = StepTcState();
}

static int step_tc_init(vaeb_handle* h) {
  using namespace st2;
  StepTcState& s = h->steptc;
  const int D = h->D, H = h->H, Z = h->Z;
  const int HP = (H + 63) / 64 * 64, KD = (D + 63) / 64, KH = HP / 64;
  const int NH = (2 * Z + 15) / 16 * 16, NZ = (Z + 1 + 15) / 16 * 16;
  const int n3 = (D + 31) / 32;
  const int TR3 = h->cont ? 64 : 32, KV = h->cont ? n3 : KD;
  const int m_h1 = (H + 1 + MP - 1) / MP;
  VAEB_CUDA(cudaFuncSetAttribute(step_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  VAEB_CUDA(cudaFuncSetAttribute(step_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  // how many clusters of four fit at once: the grid must be co-resident (grid barriers)
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(CL * 64); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = SMEM_BYTES;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = CL; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
  cfg.attrs = &at; cfg.numAttrs = 1;
  int ncl = 0;
  VAEB_CUDA(cudaOccupancyMaxActiveClusters(&ncl, step_tc_kernel<true>, &cfg));
  if (ncl < 8) { s.unavailable = true; return VAEB_OK; }
  s.n_cta = CL * std::min(ncl, 33);
  auto alloc = [](void** q, size_t bytes) -> cudaError_t {
    cudaError_t e = cudaMalloc(q, bytes);
    if (e == cudaSuccess) e = cudaMemset(*q, 0, bytes);
    return e;
  };
  VAEB_CUDA(alloc((void**)&s.bar, sizeof(unsigned long long)));
  VAEB_CUDA(alloc((void**)&s.m_enc1, (size_t)HP * KD * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_dgrad, (size_t)HP * KV * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_heads, (size_t)NH * KH * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_dec2, (size_t)n3 * TR3 * KH * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_dz, (size_t)NZ * KH * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_dec1, (size_t)HP * 64 * 4));
  VAEB_CUDA(alloc((void**)&s.m_w45k, (size_t)2 * HP * 64 * 4));       // two copies (step parity)
  // activation mirrors in one allocation (cleared together when the minibatch size changes)
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at_ = o; o += (bytes + 1023) / 1024 * 1024; return at_; };
  s.o_he_km = take((size_t)KH * 2 * TBA);
  s.o_he_t = take((size_t)m_h1 * 4 * TBA);
  s.o_hd_t = take((size_t)m_h1 * 4 * TBA);
  s.o_da2_km = take((size_t)KV * 2 * TBA);
  s.o_da2_t = take((size_t)n3 * 4 * TR3 * 128);
  s.o_da1_km = take((size_t)KH * 2 * TBA);
  s.o_da1_t = take((size_t)m_h1 * 4 * TBA);
  s.o_dd_t = take((size_t)4 * NH * 128);
  s.o_z_t = take((size_t)4 * NZ * 128);
  s.o_z_km = take((size_t)2 * TBA);
  s.o_dd_km = take((size_t)2 * TBA);
  s.o_x_km = take((size_t)KD * 2 * TBA);
  s.o_x_t = take((size_t)((D + 1 + MP - 1) / MP) * 4 * TBA);
  s.act_bytes = o;
  VAEB_CUDA(alloc((void**)&s.act, s.act_bytes));
  VAEB_CUDA(alloc((void**)&s.he, (size_t)MP * HP * 4));
  VAEB_CUDA(alloc((void**)&s.hd, (size_t)MP * HP * 4));
  VAEB_CUDA(alloc((void**)&s.mu, (size_t)MP * Z * 4));
  VAEB_CUDA(alloc((void**)&s.ls, (size_t)MP * Z * 4));
  VAEB_CUDA(alloc((void**)&s.eps, (size_t)MP * Z * 4));
  VAEB_CUDA(alloc((void**)&s.z, (size_t)MP * Z * 4));
  VAEB_CUDA(alloc((void**)&s.partial, (size_t)MP * n3 * 4));
  VAEB_CUDA(alloc((void**)&s.aux, (size_t)MP * 4));
  VAEB_CUDA(alloc((void**)&s.d_status, 2 * sizeof(int)));
  VAEB_CUDA(alloc((void**)&s.tprior_part, (size_t)2 * s.n_cta * sizeof(float)));
  s.ready = true;
  return VAEB_OK;
}

int step_tc_launch(vaeb_handle* h, const int* d_order, const float* d_kl, const float* d_xrows, int rows, int n_steps,
                   const float* d_eps, int slot0, long long* d_timing) {
  using namespace st2;
  StepTcState& s = h->steptc;
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  if (!s.ready) {
    VAEB_TRY(step_tc_init(h));
    if (s.unavailable) { vaeb_set_error("step_tc: thread-block clusters of 4 are not available on this device"); return VAEB_ESTATE; }
  }
  Params p{};
  p.D = D; p.H = H; p.Z = Z; p.M = rows;
  p.HP = (H + 63) / 64 * 64; p.KD = (D + 63) / 64; p.KH = p.HP / 64;
  p.NH = (2 * Z + 15) / 16 * 16; p.NZ = (Z + 1 + 15) / 16 * 16;
  p.n_tiles3 = (D + 31) / 32;
  p.cont = h->cont ? 1 : 0; p.TR3 = h->cont ? 64 : 32; p.KV = h->cont ? p.n_tiles3 : p.KD;
  p.oW6 = h->cont ? l.off[l.iW6] : 0; p.ob6 = h->cont ? l.off[l.ib6] : 0;
  p.la = h->cfg.estimator == VAEB_EST_LA ? 1 : 0;
  const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES;
  p.w = fb ? 1.0f / (float)rows : 1.0f;
  p.kl_beta = d_kl;
  p.lr = h->cfg.learning_rate; p.ada_eps = h->cfg.adagrad_eps;
  p.prior = fb ? 0.f : h->cfg.prior_scale;
  p.p2 = fb ? h->cfg.learning_rate * 1e-6f : 0.f;
  p.P = h->d_params; p.ada = h->d_ada;
  p.oW3 = l.off[l.iW3]; p.oW4 = l.off[l.iW4]; p.oW5 = l.off[l.iW5]; p.oW1 = l.off[l.iW1]; p.oW2 = l.off[l.iW2];
  p.ob3 = l.off[l.ib3]; p.ob4 = l.off[l.ib4]; p.ob5 = l.off[l.ib5]; p.ob1 = l.off[l.ib1]; p.ob2 = l.off[l.ib2];
  p.m_enc1 = s.m_enc1; p.m_heads = s.m_heads; p.m_dec2 = s.m_dec2; p.m_dgrad = s.m_dgrad; p.m_dz = s.m_dz;
  p.m_dec1 = s.m_dec1;
  p.he_km = s.act + s.o_he_km; p.he_t = s.act + s.o_he_t; p.hd_t = s.act + s.o_hd_t;
  p.da2_km = s.act + s.o_da2_km; p.da2_t = s.act + s.o_da2_t; p.da1_km = s.act + s.o_da1_km; p.da1_t = s.act + s.o_da1_t;
  p.dd_t = s.act + s.o_dd_t; p.z_t = s.act + s.o_z_t; p.z_km = s.act + s.o_z_km;
  p.x_base = (d_order && d_xrows) ? d_xrows : h->d_x; p.batch_order = d_order; p.x_direct = d_xrows;
  p.eps_inj = d_eps;
  p.seed = h->cfg.seed; p.step0 = h->step; p.row_offset = 0;
  p.w45_par0 = s.w45_par;
  p.he = s.he; p.hd = s.hd; p.mu = s.mu; p.ls = s.ls; p.eps = s.eps; p.z = s.z;
  p.dd_km = s.act + s.o_dd_km; p.x_km = s.act + s.o_x_km; p.x_t = s.act + s.o_x_t;
  p.m_w45k = s.m_w45k; p.w45k_bytes = p.HP * 64 * 4;
  p.partial = s.partial; p.aux = s.aux;
  p.scalars = h->d_scalars + slot0; p.Mg = (float)rows; p.bmult = 1.0f;
  p.n_steps = n_steps;
  p.bar = s.bar; p.bar_base = s.bar_count;
  p.timing = d_timing;
  p.status = s.d_status;
  p.fvb = h->cfg.estimator == VAEB_EST_FVB ? 1 : (h->cfg.estimator == VAEB_EST_FVB_SAMPLED ? 2 : 0);
  if (p.fvb == 2) {
    // the layers run on the sampled theta; the data term of the gradient carries the factor M of VAEB.py:364
    p.P = h->d_theta; p.zeta = h->d_zeta; p.w = (float)rows;
    // theta and zeta of this step: drawn by the previous launch's epilogues (MUFU forms), restored with
    // vaeb_set_tensors(10, 11), or drawn here; the operand mirrors are rebuilt from the fp32 theta below when stale
    if (s.theta_step != (long long)h->step) {
      VAEB_CUDA(launch_sample_theta(h->stream, &h->launches, h->d_vmu, h->d_vsig, nullptr, h->cfg.seed, h->step, l.total,
                                    h->d_theta, h->d_zeta));
      invalidate_weight_mirrors(h);
    }
  }
  if (p.fvb) {
    // SGVB = x.shape[0] * (sum logp + sum KL) + thetaPrior, update returns SGVB / M (VAEB.py:364,412)
    p.bmult = (float)rows; p.prior = h->cfg.prior_scale; p.p2 = 0.f;
    p.vmu = h->d_vmu; p.vsig = h->d_vsig; p.ada_mu = h->d_ada_mu; p.ada_sig = h->d_ada_sig; p.total = l.total;
    p.tprior_part = s.tprior_part;
  }
  const bool can_abort = h->cont && p.fvb != 1;           // forward-only full VB writes no deltas
  if (can_abort) VAEB_CUDA(cudaMemsetAsync(s.d_status, 0xFF, sizeof(int), h->stream));      // -1
  if (rows != s.rows_init) {
    // batch columns >= rows of every activation mirror must read as zero (they are contraction rows of the weight
    // gradients): clear everything when the minibatch size changes, then restore the constant "ones" features
    VAEB_CUDA(cudaMemsetAsync(s.act, 0, s.act_bytes, h->stream));
    OnesArgs oa{p.he_t, p.hd_t, p.z_t, p.z_km, p.x_t, H, Z, p.NZ, D};
    init_ones_kernel<<<1, 128, 0, h->stream>>>(oa);
    VAEB_CUDA(cudaGetLastError());
    ++h->launches;
    s.rows_init = rows;
  }
  if (!s.mirrors_valid) {
    MirrorArgs a{p.P, p.oW3, p.oW4, p.oW5, p.oW1, p.oW2, p.ob1, p.oW6, p.cont, p.TR3, p.KV, s.m_enc1, s.m_heads, s.m_dec2, s.m_dgrad, s.m_dz,
                 s.m_dec1, s.m_w45k, D, H, Z, p.HP, p.KD, p.KH, p.NH, p.NZ};
    int64_t most = (int64_t)p.HP * p.KD * 64;
    most = std::max<int64_t>(most, (int64_t)p.n_tiles3 * p.TR3 * p.KH * 64);
    most = std::max<int64_t>(most, (int64_t)p.HP * p.KV * 64);
    most = std::max<int64_t>(most, (int64_t)p.NH * p.KH * 64);
    build_mirrors_kernel<<<dim3((unsigned)((most + 255) / 256), 7), 256, 0, h->stream>>>(a);
    VAEB_CUDA(cudaGetLastError());
    ++h->launches;
    s.mirrors_valid = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(s.n_cta); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = h->stream;
  cudaLaunchAttribute at[2]{};
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeCooperative; at[1].val.cooperative = 1;
  cfg.attrs = at; cfg.numAttrs = 2;
  if (p.fvb == 2) VAEB_CUDA(cudaLaunchKernelEx(&cfg, step_tc_kernel<true>, p));
  else VAEB_CUDA(cudaLaunchKernelEx(&cfg, step_tc_kernel<false>, p));
  ++h->launches;
  h->grads_have_prior = false;
  invalidate_weight_mirrors(h);
  s.mirrors_valid = true;             // the kernel keeps its own mirrors current with the parameters it updates
  int done = n_steps;
  if (can_abort) {
    // the Gaussian decoder's deltas are unbounded: did a step leave the range of the fp16 operand pairs?
    int st = -1;
    VAEB_CUDA(cudaMemcpyAsync(&st, s.d_status, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    if (st >= 0) done = st;
  }
  // an aborted launch passed 4 of the grid barriers of step `done`
  s.bar_count += (unsigned long long)s.n_cta * ((unsigned long long)(p.fvb == 1 ? 3 : N_PHASES) * (unsigned long long)done + (done < n_steps ? 4ull : 0ull));
  h->step += (uint32_t)done;
  s.w45_par ^= done & 1;              // each completed step wrote the other copy
  s.theta_step = (long long)h->step;
  if (done < n_steps) {
    // steps done .. n_steps-1 through the fp32 FFMA kernel (same contract; it invalidates the operand mirrors)
    VAEB_REQUIRE(fused_step_supported(h, rows), "step_tc: delta overflow and no fp32 single-launch kernel for this configuration");
    return fused_step_launch(h, d_order ? d_order + done : nullptr, d_kl ? d_kl + done : nullptr, d_xrows, rows, n_steps - done, d_eps, slot0 + done, nullptr);
  }
  return VAEB_OK;
}
