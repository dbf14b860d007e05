// Epilogues of the tcgen05 layers (one thread owns one accumulator row, 16 columns per call) and the 16-/32-byte
// access helpers they share.  Included by tc_layers.cu.
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"
#include "launchers.h"
#include "tc_common.cuh"
#include "philox.cuh"

namespace {

constexpr int BM = 128, BK = 64;
constexpr int EPI_WARPS = 16, TC_THREADS = 128 + EPI_WARPS * 32;

__device__ __forceinline__ void put_split(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t o, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[o] = h;
  if (lo) lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// ---- epilogues: one thread owns one accumulator row, 16 columns per call --------------------
// A thread's 16 columns are contiguous in every operand it touches, but neighbouring lanes are different
// ROWS: scalar accesses would touch 32 cache lines per instruction, 4 (or 2) bytes each.  The fast paths move
// 16 bytes per access (full 32-byte sectors per row), the scalar paths handle ragged edges.
__device__ __forceinline__ bool vec_ok(const void* p, int col0, int N) {
  return col0 + 16 <= N && (((uintptr_t)p) & 15u) == 0;
}
// 32-byte (whole-sector) accesses, sm_100: one request per sector instead of two half-sector ones
__device__ __forceinline__ void st32B(void* p, const uint32_t* w) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
               "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}
__device__ __forceinline__ void ld32B(const void* p, uint32_t* w) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
               : "l"(p));
}
__device__ __forceinline__ void ld16f(const float* p, float* d) {
  if ((((uintptr_t)p) & 31u) == 0) {
    ld32B(p, reinterpret_cast<uint32_t*>(d));
    ld32B(p + 8, reinterpret_cast<uint32_t*>(d) + 8);
    return;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 t = *reinterpret_cast<const float4*>(p + 4 * q);
    d[4 * q] = t.x; d[4 * q + 1] = t.y; d[4 * q + 2] = t.z; d[4 * q + 3] = t.w;
  }
}
__device__ __forceinline__ void unpack16bf(const uint32_t* w, float* d) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    d[2 * q] = __uint_as_float(w[q] << 16);
    d[2 * q + 1] = __uint_as_float(w[q] & 0xffff0000u);
  }
}
__device__ __forceinline__ void ld16bf(const __nv_bfloat16* p, float* d) {
  uint32_t w[8];
  if ((((uintptr_t)p) & 31u) == 0) {
    ld32B(p, w);
  } else {
    const uint4 a = reinterpret_cast<const uint4*>(p)[0], b = reinterpret_cast<const uint4*>(p)[1];
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    d[2 * q] = __uint_as_float(w[q] << 16);
    d[2 * q + 1] = __uint_as_float(w[q] & 0xffff0000u);
  }
}
__device__ __forceinline__ void st16f(float* p, const float* d) {
  if ((((uintptr_t)p) & 31u) == 0) {
    st32B(p, reinterpret_cast<const uint32_t*>(d));
    st32B(p + 8, reinterpret_cast<const uint32_t*>(d) + 8);
    return;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(p + 4 * q) = make_float4(d[4 * q], d[4 * q + 1], d[4 * q + 2], d[4 * q + 3]);
}
// packed conversions (F2FP.BF16.PACK_AB, full rate) instead of one quarter-rate F2F per element
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&t);
}
__device__ __forceinline__ void st16_split(__nv_bfloat16* hi, __nv_bfloat16* lo, const float* d) {
  uint32_t h[8], l[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    h[q] = pack_bf16x2(d[2 * q], d[2 * q + 1]);
    if (lo) l[q] = pack_bf16x2(d[2 * q] - __uint_as_float(h[q] << 16), d[2 * q + 1] - __uint_as_float(h[q] & 0xffff0000u));
  }
  if ((((uintptr_t)hi | (uintptr_t)lo) & 31u) == 0) {
    st32B(hi, h);
    if (lo) st32B(lo, l);
    return;
  }
  reinterpret_cast<uint4*>(hi)[0] = make_uint4(h[0], h[1], h[2], h[3]);
  reinterpret_cast<uint4*>(hi)[1] = make_uint4(h[4], h[5], h[6], h[7]);
  if (lo) {
    reinterpret_cast<uint4*>(lo)[0] = make_uint4(l[0], l[1], l[2], l[3]);
    reinterpret_cast<uint4*>(lo)[1] = make_uint4(l[4], l[5], l[6], l[7]);
  }
}

// tanh on the epilogue's critical path: 16 warps finish a 128 x 256 tile = 32768 activations, and libdevice's tanhf
// (~40 instructions, a divergent branch) alone costs ~5 us per tile.  fast = 1 (plain bf16 tier, the result is
// rounded to bf16 anyway): MUFU tanh.approx (|err| <= 2^-10.99).  fast = 0 (bf16x3, fp32 tier): branch-free --
// 1 - 2/(e^{2|x|}+1) from ex2.approx / rcp.approx (|err| < 4e-7) for |x| >= 0.1, the odd Taylor polynomial through
// x^9 below (truncation < 1e-13 at 0.1); relative error < 5e-6 everywhere.
__device__ __forceinline__ float tanh_tc(float x, int fast) {
  if (fast) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
  }
  const float ax = fabsf(x), x2 = x * x;
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * 2.8853900817779268f));   // e^{2|x|}
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  const float big = copysignf(fmaf(-2.0f, r, 1.0f), x);
  const float poly = fmaf(x * x2, fmaf(x2, fmaf(x2, fmaf(x2, 0.021869488536155203f, -0.053968253968253971f),
                                                0.13333333333333333f), -0.33333333333333331f), x);
  return ax < 0.1f ? poly : big;
}

// out == nullptr: only the mirror is written (large-batch path: every consumer reads the bf16 mirrors)
struct EpiTanh {            // out[row, col] = tanh(acc + bias[col]) (+ optional bf16 hi/lo mirror of it)
  static constexpr bool PREFETCH = true;   // persistent kernel: unrolled epilogue with the next chunk's operand in flight
  const float* bias; float* out; int ld;
  __nv_bfloat16* mh; __nv_bfloat16* ml; int ldm; int fast;
  __device__ __forceinline__ void begin() {}
  __device__ __forceinline__ void split(int) {}
  __device__ __forceinline__ bool preload(int, bool, int, int, uint32_t*) const { return false; }   // bias only: L1 hits
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* = nullptr) {
    if (!ok) return;
    float* o = out ? out + (size_t)row * ld + col0 : nullptr;
    __nv_bfloat16* m = mh ? mh + (size_t)row * ldm + col0 : nullptr;
    if (vec_ok(o, col0, N) && vec_ok(bias + col0, col0, N) && vec_ok(m, col0, N)) {
      float r[16];
      ld16f(bias + col0, r);
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] += v[j];
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] = tanh_tc(r[j], fast);
      if (out) st16f(o, r);
      if (mh) st16_split(m, ml ? ml + (size_t)row * ldm + col0 : nullptr, r);
      return;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) {
        const float t = tanh_tc(v[j] + bias[col0 + j], fast);
        if (out) o[j] = t;
        if (mh) put_split(mh, ml, (size_t)row * ldm + col0 + j, t);
      }
  }
  __device__ __forceinline__ void end(int, bool, int, int) {}
};

struct EpiBernoulliTc {     // VAEB.py:263,311: term = x*a - softplus(a); da = scale*(x - sigmoid(a))
  static constexpr bool PREFETCH = false;   // persistent kernel: unrolled epilogue with the next chunk's operand in flight
  const float* bias; const float* x; int ldx; int x_div; int x_mod; float scale;
  __nv_bfloat16* da_hi; __nv_bfloat16* da_lo; int ldda; float* partial;
  // x == nullptr: x is read from its bf16 mirror (hi + lo when present), row offset xm_off, leading dimension ldxm
  const __nv_bfloat16* xm_hi; const __nv_bfloat16* xm_lo; int ldxm; int xm_off;
  float acc;
  __device__ __forceinline__ void begin() { acc = 0.f; }
  __device__ __forceinline__ void split(int) {}
  // one exponential serves both: t = e^-|a|; softplus = max(a,0) + log(1+t); sigmoid = {1, t}/(1+t)
  // (three MUFU ops -- ex2, rcp, lg2 -- and ~12 FP32 instructions per element: this epilogue is issue bound, ncu shows
  // the schedulers 48 % active against 19-28 % in the other layers)
  __device__ __forceinline__ float one(float a, float xv) {
    float t, r, lg;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-1.4426950408889634f * fabsf(a)));     // e^-|a|
    const float u = 1.0f + t;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(u));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u));
    acc += fmaf(xv, a, -fmaf(lg, 0.6931471805599453f, fmaxf(a, 0.f)));
    return scale * (xv - (a >= 0.f ? r : t * r));
  }
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* pre = nullptr) {
    if (!ok) return;
    const int xrow = (row / x_div) % x_mod;
    const float* xr = x ? x + (size_t)xrow * ldx + col0 : nullptr;
    const size_t oxm = (size_t)(xm_off + xrow) * ldxm + col0;
    __nv_bfloat16* dh = da_hi ? da_hi + (size_t)row * ldda + col0 : nullptr;
    __nv_bfloat16* dl = da_lo ? da_lo + (size_t)row * ldda + col0 : nullptr;
    if (vec_ok(xr, col0, N) && vec_ok(bias + col0, col0, N) && vec_ok(dh, col0, N) && vec_ok(dl, col0, N) &&
        vec_ok(x ? nullptr : xm_hi + oxm, col0, N)) {
      float b[16], xv[16], d[16];
      ld16f(bias + col0, b);
      if (x) {
        ld16f(xr, xv);
      } else {
        if (pre) unpack16bf(pre, xv); else ld16bf(xm_hi + oxm, xv);
        if (xm_lo) {
          float lo[16];
          ld16bf(xm_lo + oxm, lo);
#pragma unroll
          for (int j = 0; j < 16; ++j) xv[j] += lo[j];
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) d[j] = one(v[j] + b[j], xv[j]);
      if (dh) st16_split(dh, dl, d);
      return;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int c = col0 + j;
      if (c < N) {
        float xj;
        if (x) xj = xr[j];
        else xj = __bfloat162float(xm_hi[oxm + j]) + (xm_lo ? __bfloat162float(xm_lo[oxm + j]) : 0.f);
        const float d = one(v[j] + bias[c], xj);
        if (dh) put_split(dh, dl, (size_t)j, d);
      }
    }
  }
  __device__ __forceinline__ void end(int row, bool ok, int tile_n, int n_tiles) {
    if (ok) partial[(size_t)row * n_tiles + tile_n] = acc;
  }
};

// Gaussian decoder on the tensor cores (VAEB.py:257-258, 306-307): the output layer is ONE GEMM over the interleaved
// columns [W2|W6]' (column 2d = W2[:, d], 2d + 1 = W6[:, d]), so the thread that owns an accumulator row holds
// (a_d, lv_d) of eight pixels per 16-column chunk.  term = -log(2 pi)/2 - lv/2 - (x - mu)^2 e^{-lv} / 2, mu = sigmoid(a);
// deltas scale * (x - mu) e^{-lv} mu (1 - mu) and scale * (-1/2 + (x - mu)^2 e^{-lv} / 2) go to the interleaved mirror
// [rows, ldda] that the backward GEMMs (dgrad over K = 2D, the [W2|W6]' weight gradient) read.
struct EpiGaussianTc {
  static constexpr bool PREFETCH = false;
  const float* b2; const float* b6; const float* x; int ldx; int x_div; int x_mod; float scale;
  __nv_bfloat16* da_hi; __nv_bfloat16* da_lo; int ldda; float* partial;
  const __nv_bfloat16* xm_hi; const __nv_bfloat16* xm_lo; int ldxm; int xm_off;      // x == nullptr: x from its bf16 mirror
  float acc;
  __device__ __forceinline__ void begin() { acc = 0.f; }
  __device__ __forceinline__ void split(int) {}
  __device__ __forceinline__ void one(float a, float lv, float xv, float& d_a, float& d_lv) {
    const float mu = 1.0f / (1.0f + __expf(-a));
    const float d = xv - mu;
    const float r = d * __expf(-lv);
    acc += -0.91893853320467274178f - 0.5f * lv - 0.5f * d * r;
    d_a = scale * r * mu * (1.0f - mu);
    d_lv = scale * (-0.5f + 0.5f * d * r);
  }
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* = nullptr) {
    if (!ok) return;
    const int xrow = (row / x_div) % x_mod;
    const int d0 = col0 >> 1;                               // first pixel of the chunk; N = 2 D
    float out[16];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int d = d0 + j;
      out[2 * j] = out[2 * j + 1] = 0.f;
      if (2 * d + 1 < N) {
        float xv;
        if (x) xv = x[(size_t)xrow * ldx + d];
        else xv = __bfloat162float(xm_hi[(size_t)(xm_off + xrow) * ldxm + d]) +
                  (xm_lo ? __bfloat162float(xm_lo[(size_t)(xm_off + xrow) * ldxm + d]) : 0.f);
        one(v[2 * j] + b2[d], v[2 * j + 1] + b6[d], xv, out[2 * j], out[2 * j + 1]);
      }
    }
    if (!da_hi) return;
    __nv_bfloat16* dh = da_hi + (size_t)row * ldda + col0;
    __nv_bfloat16* dl = da_lo ? da_lo + (size_t)row * ldda + col0 : nullptr;
    if (vec_ok(dh, col0, N) && vec_ok(dl, col0, N)) { st16_split(dh, dl, out); return; }
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) put_split(dh, dl, (size_t)j, out[j]);
  }
  __device__ __forceinline__ void end(int row, bool ok, int tile_n, int n_tiles) {
    if (ok) partial[(size_t)row * n_tiles + tile_n] = acc;
  }
};

struct EpiWgradTc {         // rows < Hreal -> gW[Hreal, N]; row == Hreal (the ones column of A) -> gb
  float* gW; float* gb; int Hreal; int ld;
  float* scratch; size_t split_stride;   // split-K: slice z writes [gW | gb] at scratch + z * split_stride
  __device__ __forceinline__ void begin() {}
  __device__ __forceinline__ void split(int z) {
    if (scratch) { gW = scratch + (size_t)z * split_stride; gb = gW + (size_t)Hreal * ld; }
  }
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* = nullptr) {
    if (!ok) return;
    float* dst = (row < Hreal ? gW + (size_t)row * ld : gb) + col0;
    if (vec_ok(dst, col0, N)) { st16f(dst, v); return; }
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) dst[j] = v[j];
  }
  __device__ __forceinline__ void end(int, bool, int, int) {}
};

// h comes in fp32 (h != nullptr) or as its bf16 mirror hh (+ hl: hi + lo carries 16 mantissa bits); out == nullptr:
// only the mirror of the result is written (large-batch path)
struct EpiDgradTanh {       // out = acc * (1 - h^2) (+ optional bf16 hi/lo mirror of it)
  static constexpr bool PREFETCH = true;   // persistent kernel: unrolled epilogue with the next chunk's operand in flight
  const float* h; float* out; int ld;
  __nv_bfloat16* mh; __nv_bfloat16* ml; int ldm;
  const __nv_bfloat16* hh; const __nv_bfloat16* hl;      // mirror of h, leading dimension ldm
  __device__ __forceinline__ void begin() {}
  __device__ __forceinline__ void split(int) {}
  __device__ __forceinline__ float hval(int row, int c) const {
    if (h) return h[(size_t)row * ld + c];
    float t = __bfloat162float(hh[(size_t)row * ldm + c]);
    if (hl) t += __bfloat162float(hl[(size_t)row * ldm + c]);
    return t;
  }
  __device__ __forceinline__ bool preload(int row, bool ok, int col0, int N, uint32_t* w) const {
    if (!ok || h || col0 + 16 > N) return false;
    const __nv_bfloat16* p = hh + (size_t)row * ldm + col0;
    if (((uintptr_t)p) & 31u) return false;
    ld32B(p, w);
    return true;
  }
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* pre = nullptr) {
    if (!ok) return;
    const float* hp = h ? h + (size_t)row * ld + col0 : nullptr;
    float* o = out ? out + (size_t)row * ld + col0 : nullptr;
    const size_t om = (size_t)row * ldm + col0;
    if (vec_ok(hp, col0, N) && vec_ok(o, col0, N) && vec_ok(mh ? mh + om : nullptr, col0, N) &&
        vec_ok(hh ? hh + om : nullptr, col0, N)) {
      float hv[16], r[16];
      if (h) {
        ld16f(hp, hv);
      } else {
        if (pre) unpack16bf(pre, hv); else ld16bf(hh + om, hv);
        if (hl) {
          float lo[16];
          ld16bf(hl + om, lo);
#pragma unroll
          for (int j = 0; j < 16; ++j) hv[j] += lo[j];
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] = v[j] * (1.0f - hv[j] * hv[j]);
      if (out) st16f(o, r);
      if (mh) st16_split(mh + om, ml ? ml + om : nullptr, r);
      return;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) {
        const float hvj = hval(row, col0 + j);
        const float t = v[j] * (1.0f - hvj * hvj);
        if (out) o[j] = t;
        if (mh) put_split(mh, ml, om + j, t);
      }
  }
  __device__ __forceinline__ void end(int, bool, int, int) {}
};

// (mu_j, ls_j) = columns (2j, 2j+1) of h_e.[W4|W5]_interleaved + bias -> eps, z, row term, z mirror (L = 1)
struct EpiHeads {
  static constexpr bool PREFETCH = false;   // persistent kernel: unrolled epilogue with the next chunk's operand in flight
  const float* b4; const float* b5; int Z; int la; EpsSource src;
  float* mu; float* ls; float* eps; float* z; __nv_bfloat16* z_hi; __nv_bfloat16* z_lo; int ldz; float* aux_part;
  float acc;
  __device__ __forceinline__ void begin() { acc = 0.f; }
  __device__ __forceinline__ void split(int) {}
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* = nullptr) {
    if (!ok) return;
    // one Philox counter yields four draws: elements (row, 4g..4g+3) share one when Z is a multiple of 4
    float e8[8];
    const int j0 = col0 >> 1;
    if (!src.injected && (Z & 3) == 0) {
#pragma unroll
      for (int g = 0; g < 2; ++g)
        if (j0 + 4 * g < Z)
          philox_normal4(src.seed, src.stream, src.step, 0u,
                         (uint64_t)(((src.row_offset + row) * Z + j0 + 4 * g) >> 2), e8 + 4 * g);
    } else {
#pragma unroll
      for (int jj = 0; jj < 8; ++jj)
        if (j0 + jj < Z)
          e8[jj] = src.injected ? src.injected[(size_t)row * Z + j0 + jj]
                                : philox_normal1(src.seed, src.stream, src.step, 0u,
                                                 (uint64_t)((src.row_offset + row) * Z + j0 + jj));
    }
    float am8[8], al8[8], z8[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      const int j = j0 + jj;
      am8[jj] = al8[jj] = z8[jj] = 0.f;
      if (j < Z) {
        const float am = v[2 * jj] + b4[j], al = v[2 * jj + 1] + b5[j];
        const float e = e8[jj];
        const float zv = am + expf(0.5f * al) * e;
        am8[jj] = am; al8[jj] = al; z8[jj] = zv;
        acc += la ? (-0.5f * zv * zv + 0.5f * al + 0.5f * e * e) : 0.5f * (1.0f + al - am * am - expf(al));
      } else {
        e8[jj] = 0.f;
      }
    }
    // a thread's eight latent units are contiguous in every output: 16-byte stores where a whole quad is valid
    const size_t o2 = (size_t)row * Z + j0;
    const bool al16 = ((Z & 3) == 0) && ((((uintptr_t)mu | (uintptr_t)ls | (uintptr_t)eps | (uintptr_t)z) & 15u) == 0);
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const int jq = j0 + 4 * g;
      if (al16 && jq + 4 <= Z) {
        *reinterpret_cast<float4*>(mu + o2 + 4 * g) = make_float4(am8[4 * g], am8[4 * g + 1], am8[4 * g + 2], am8[4 * g + 3]);
        *reinterpret_cast<float4*>(ls + o2 + 4 * g) = make_float4(al8[4 * g], al8[4 * g + 1], al8[4 * g + 2], al8[4 * g + 3]);
        *reinterpret_cast<float4*>(eps + o2 + 4 * g) = make_float4(e8[4 * g], e8[4 * g + 1], e8[4 * g + 2], e8[4 * g + 3]);
        *reinterpret_cast<float4*>(z + o2 + 4 * g) = make_float4(z8[4 * g], z8[4 * g + 1], z8[4 * g + 2], z8[4 * g + 3]);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (jq + q < Z) {
            mu[o2 + 4 * g + q] = am8[4 * g + q]; ls[o2 + 4 * g + q] = al8[4 * g + q];
            eps[o2 + 4 * g + q] = e8[4 * g + q]; z[o2 + 4 * g + q] = z8[4 * g + q];
          }
      }
    }
    // z mirror: the row is ldz wide (a multiple of 8: 16-byte aligned octets), columns >= Z stay as initialised
    __nv_bfloat16* zh = z_hi + (size_t)row * ldz + j0;
    __nv_bfloat16* zl = z_lo ? z_lo + (size_t)row * ldz + j0 : nullptr;
    if (j0 + 8 <= Z && (((uintptr_t)zh) & 15u) == 0 && (!zl || (((uintptr_t)zl) & 15u) == 0)) {
      uint32_t hq[4], lq[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        hq[q] = pack_bf16x2(z8[2 * q], z8[2 * q + 1]);
        lq[q] = pack_bf16x2(z8[2 * q] - __uint_as_float(hq[q] << 16), z8[2 * q + 1] - __uint_as_float(hq[q] & 0xffff0000u));
      }
      *reinterpret_cast<uint4*>(zh) = make_uint4(hq[0], hq[1], hq[2], hq[3]);
      if (zl) *reinterpret_cast<uint4*>(zl) = make_uint4(lq[0], lq[1], lq[2], lq[3]);
    } else {
#pragma unroll
      for (int jj = 0; jj < 8; ++jj)
        if (j0 + jj < Z) put_split(z_hi, z_lo, (size_t)row * ldz + j0 + jj, z8[jj]);
    }
  }
  __device__ __forceinline__ void end(int row, bool ok, int tile_n, int n_tiles) {
    if (ok) aux_part[(size_t)row * n_tiles + tile_n] = acc;
  }
};

// dz = da1.W1^T -> dmu, dls (L = 1; formulas of SURVEY.md 8a, as launch_dprep / lb_latent_bwd) + bf16 mirror [dmu|dls];
// w_aux weights the latent term (the data weight times the KL weight of vaeb_set_kl_weight)
struct EpiDzPrep {
  static constexpr bool PREFETCH = false;   // persistent kernel: unrolled epilogue with the next chunk's operand in flight
  const float* z; const float* eps; const float* mu; const float* ls; int Z; int la; float w_aux;
  float* dmu; float* dls; __nv_bfloat16* dd_hi; __nv_bfloat16* dd_lo; int ldq;
  __device__ __forceinline__ void begin() {}
  __device__ __forceinline__ void split(int) {}
  __device__ __forceinline__ void chunk(int row, bool ok, int col0, int N, const float* v, const uint32_t* = nullptr) {
    if (!ok) return;
    const size_t o0 = (size_t)row * Z + col0;
    const bool al16 = ((Z & 3) == 0) &&
                      ((((uintptr_t)z | (uintptr_t)eps | (uintptr_t)mu | (uintptr_t)ls | (uintptr_t)dmu | (uintptr_t)dls) & 15u) == 0);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int c = col0 + 4 * g;
      if (c >= N) break;
      float lsv[4], zv[4], ev[4], mv[4], a[4], b[4];
      const bool vec = al16 && c + 4 <= N;
      if (vec) {
        const float4 t0 = *reinterpret_cast<const float4*>(ls + o0 + 4 * g), t1 = *reinterpret_cast<const float4*>(eps + o0 + 4 * g);
        lsv[0] = t0.x; lsv[1] = t0.y; lsv[2] = t0.z; lsv[3] = t0.w;
        ev[0] = t1.x; ev[1] = t1.y; ev[2] = t1.z; ev[3] = t1.w;
        const float4 t2 = *reinterpret_cast<const float4*>((la ? z : mu) + o0 + 4 * g);
        zv[0] = mv[0] = t2.x; zv[1] = mv[1] = t2.y; zv[2] = mv[2] = t2.z; zv[3] = mv[3] = t2.w;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          lsv[q] = ev[q] = zv[q] = mv[q] = 0.f;
          if (c + q < N) {
            lsv[q] = ls[o0 + 4 * g + q]; ev[q] = eps[o0 + 4 * g + q];
            zv[q] = mv[q] = (la ? z : mu)[o0 + 4 * g + q];
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float d = v[4 * g + q];
        if (la) d -= w_aux * zv[q];
        a[q] = d; b[q] = d * (0.5f * expf(0.5f * lsv[q]) * ev[q]);
        if (la) {
          b[q] += w_aux * 0.5f;
        } else {
          a[q] -= w_aux * mv[q];
          b[q] += w_aux * 0.5f * (1.0f - expf(lsv[q]));
        }
      }
      if (vec) {
        *reinterpret_cast<float4*>(dmu + o0 + 4 * g) = make_float4(a[0], a[1], a[2], a[3]);
        *reinterpret_cast<float4*>(dls + o0 + 4 * g) = make_float4(b[0], b[1], b[2], b[3]);
      }
      // [dmu | dls] mirror row: quads are 8-byte aligned when Z and ldq are multiples of 4
      const size_t oa = (size_t)row * ldq + c, ob = oa + Z;
      if (vec && (ldq & 3) == 0 && (((uintptr_t)dd_hi | (uintptr_t)dd_lo) & 7u) == 0) {
        uint32_t ha[2], la_[2], hb[2], lb[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          ha[q] = pack_bf16x2(a[2 * q], a[2 * q + 1]);
          hb[q] = pack_bf16x2(b[2 * q], b[2 * q + 1]);
          la_[q] = pack_bf16x2(a[2 * q] - __uint_as_float(ha[q] << 16), a[2 * q + 1] - __uint_as_float(ha[q] & 0xffff0000u));
          lb[q] = pack_bf16x2(b[2 * q] - __uint_as_float(hb[q] << 16), b[2 * q + 1] - __uint_as_float(hb[q] & 0xffff0000u));
        }
        *reinterpret_cast<uint2*>(dd_hi + oa) = make_uint2(ha[0], ha[1]);
        *reinterpret_cast<uint2*>(dd_hi + ob) = make_uint2(hb[0], hb[1]);
        if (dd_lo) {
          *reinterpret_cast<uint2*>(dd_lo + oa) = make_uint2(la_[0], la_[1]);
          *reinterpret_cast<uint2*>(dd_lo + ob) = make_uint2(lb[0], lb[1]);
        }
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (c + q < N) {
            if (!vec) { dmu[o0 + 4 * g + q] = a[q]; dls[o0 + 4 * g + q] = b[q]; }
            put_split(dd_hi, dd_lo, oa + q, a[q]);
            put_split(dd_hi, dd_lo, ob + q, b[q]);
          }
      }
    }
  }
  __device__ __forceinline__ void end(int, bool, int, int) {}
};

struct LayerMaps {            // hi/lo tensor maps of both operands (lo unused when NS == 1)
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
};

}  // namespace
