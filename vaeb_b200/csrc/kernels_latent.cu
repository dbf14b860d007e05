// Latent-layer kernels of the AEVB step: everything between the two wide hidden layers, where
// the contractions are too thin (N = 2Z, K = Z) for tiles and the work is latency-bound.
//   latent_fwd : mu, ls = h_e.W4+b4, h_e.W5+b5 (VAEB.py:248-249); eps, z = mu+exp(.5 ls) eps
//                (VAEB.py:41-47); KL / LA row terms (VAEB.py:343, :322-325);
//                h_d = tanh(z.W1+b1) (VAEB.py:254)            -- one warp per datapoint
//   latent_bwd : dz = da1.W1^T; dmu, dls (SURVEY.md 8a); da3 = (dmu.W4^T + dls.W5^T)*(1-h_e^2);
//                per-row bound and its deterministic total    -- one warp per datapoint
//   small_wgrad: gW1,gb1 = [z|1]^T.da1 ; gW4,gb4,gW5,gb5 = [h_e|1]^T.[dmu|dls]
// Optional bf16 hi/lo mirrors of h_d and da3 feed the tcgen05 GEMMs of the wide layers.
#include <cuda_bf16.h>

#include "activations.cuh"
#include "launchers.h"
#include "philox.cuh"

namespace {

constexpr int LB_MIN_ROWS = 1024;   // from here on the large-batch tilings below take over
__host__ __device__ inline bool latent_lb_supported(int rows, int H, int Z, int L) {
  return rows >= LB_MIN_ROWS && L == 1 && Z >= 1 && Z <= 23 && H >= 32;
}

constexpr int NWARPS = 16;          // 512 threads per block
constexpr int NTHREADS = NWARPS * 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void store_split(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t o, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[o] = h;
  if (lo) lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// W45T = [W4^T ; W5^T] ([2Z, H], H contiguous): both latent heads and their backward read the
// head weights with the hidden index contiguous (coalesced over lanes).
__global__ void __launch_bounds__(256)
transpose_heads_kernel(const float* __restrict__ W4, const float* __restrict__ W5, int H, int Z,
                       float* __restrict__ w45t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * Z * H) return;
  const int o = i / H, k = i % H;
  w45t[i] = (o < Z) ? W4[(size_t)k * Z + o] : W5[(size_t)k * Z + (o - Z)];
}

// A block owns RB datapoints.  Phase 1: the 2Z head pre-activations; warps split (chunk of 8
// outputs) x (slice of the hidden index), every weight is loaded once per block and reused for
// the RB rows.  Phase 2: reparameterisation + row terms (one thread per (row, j)).  Phase 3:
// decoder hidden layer, one thread per hidden unit, W1 column held in registers across the rows.
template <int RB>
__global__ void __launch_bounds__(NTHREADS)
latent_fwd_kernel(const float* __restrict__ h_e, int rows, int H, const float* __restrict__ w45t,
                  const float* __restrict__ b4, const float* __restrict__ b5, const float* __restrict__ W1,
                  const float* __restrict__ b1, int Z, int L, int la, EpsSource src, float* __restrict__ mu,
                  float* __restrict__ ls, float* __restrict__ eps, float* __restrict__ z,
                  float* __restrict__ row_aux, float* __restrict__ h_d, __nv_bfloat16* __restrict__ hd_hi,
                  __nv_bfloat16* __restrict__ hd_lo, int ld_mirror, int KS, int act) {
  extern __shared__ float sm[];
  const int Z2 = 2 * Z;
  float* part = sm;                         // [KS][RB][2Z]
  float* out = part + KS * RB * Z2;         // [RB][2Z] mu | ls
  float* zs = out + RB * Z2;                // [RB][Z]  z of the current sample
  float* terms = zs + RB * Z;               // [RB][Z]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * RB;
  const int nchunks = (Z2 + 7) / 8;
  for (int task = warp; task < nchunks * KS; task += NWARPS) {
    const int c0 = (task % nchunks) * 8, sl = task / nchunks;
    const int nq = min(8, Z2 - c0);
    const int k_lo = (int)(((long)H * sl) / KS), k_hi = (int)(((long)H * (sl + 1)) / KS);
    float acc[RB][8];
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[r][q] = 0.f;
    for (int k = k_lo + lane; k < k_hi; k += 32) {
      float wv[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) wv[q] = (q < nq) ? w45t[(size_t)(c0 + q) * H + k] : 0.f;
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const float hv = (m0 + r < rows) ? h_e[(size_t)(m0 + r) * H + k] : 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[r][q] = fmaf(hv, wv[q], acc[r][q]);
      }
    }
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float t = warp_sum(acc[r][q]);
        if (lane == 0 && q < nq) part[(sl * RB + r) * Z2 + c0 + q] = t;
      }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < RB * Z2; i += NTHREADS) {
    const int o = i % Z2;
    float t = (o < Z) ? b4[o] : b5[o - Z];
    for (int sl = 0; sl < KS; ++sl) t += part[sl * RB * Z2 + i];
    out[i] = t;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < RB * Z; i += NTHREADS) {
    const int r = i / Z, j = i % Z, m = m0 + r;
    float term = 0.f;
    if (m < rows) {
      const float am = out[r * Z2 + j], al = out[r * Z2 + Z + j];
      mu[(size_t)m * Z + j] = am;
      ls[(size_t)m * Z + j] = al;
      if (!la) term = 0.5f * (1.0f + al - am * am - expf(al));
    }
    terms[i] = term;
  }
  for (int l = 0; l < L; ++l) {
    for (int i = threadIdx.x; i < RB * Z; i += NTHREADS) {
      const int r = i / Z, j = i % Z, m = m0 + r;
      if (m < rows) {
        const float am = out[r * Z2 + j], al = out[r * Z2 + Z + j];
        const size_t o2 = ((size_t)l * rows + m) * Z + j;
        const float e = src.injected
                            ? src.injected[o2]
                            : philox_normal1(src.seed, src.stream, src.step, (uint32_t)l,
                                             (uint64_t)((src.row_offset + m) * Z + j));
        const float zv = am + expf(0.5f * al) * e;
        eps[o2] = e;
        z[o2] = zv;
        zs[i] = zv;
        if (la) terms[i] += (-0.5f * zv * zv + 0.5f * al + 0.5f * e * e) / (float)L;
      }
    }
    __syncthreads();
    for (int n = threadIdx.x; n < H; n += NTHREADS) {
      float a[RB];
      const float bn = b1[n];
#pragma unroll
      for (int r = 0; r < RB; ++r) a[r] = bn;
      for (int j = 0; j < Z; ++j) {
        const float wv = W1[(size_t)j * H + n];
#pragma unroll
        for (int r = 0; r < RB; ++r) a[r] = fmaf(zs[r * Z + j], wv, a[r]);
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        if (m0 + r < rows) {
          const size_t rr = (size_t)l * rows + m0 + r;
          const float hv = act_fwd(a[r], act);
          h_d[rr * H + n] = hv;
          if (hd_hi) store_split(hd_hi, hd_lo, rr * ld_mirror + n, hv);
        }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x < RB && m0 + threadIdx.x < rows) {
    float t = 0.f;
    for (int j = 0; j < Z; ++j) t += terms[threadIdx.x * Z + j];
    row_aux[m0 + threadIdx.x] = t;
  }
}

// deterministic sum of v[0..n) by one block (fixed strided partials + fixed tree)
__device__ float block_total(const float* __restrict__ v, int n, float* red) {
  float t = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) t += __ldcg(v + i);   // written by other blocks: bypass L1
  t = warp_sum(t);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = t;
  __syncthreads();
  float s = 0.f;
  if (wid == 0) {
    s = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.f;
    s = warp_sum(s);
  }
  return s;
}

// A block owns RB datapoints: dz (warps split latent chunks x hidden slices), dmu/dls, da3 (one
// thread per hidden unit, head weights held in registers across the rows), the per-row bound; the
// last block to finish totals the per-row bounds in a fixed order.
template <int RB>
__global__ void __launch_bounds__(NTHREADS)
latent_bwd_kernel(const float* __restrict__ da1, const float* __restrict__ W1, const float* __restrict__ w45t,
                  const float* __restrict__ h_e, const float* __restrict__ z, const float* __restrict__ eps,
                  const float* __restrict__ mu, const float* __restrict__ ls, int rows, int H, int Z, int L, int la,
                  float w_aux, float* __restrict__ dmu, float* __restrict__ dls, float* __restrict__ da3,
                  __nv_bfloat16* __restrict__ da3_hi, __nv_bfloat16* __restrict__ da3_lo, int ld_mirror,
                  const float* __restrict__ partial, int n_tiles, const float* __restrict__ row_aux,
                  float* __restrict__ per_row, unsigned int* __restrict__ counter, float* __restrict__ base_out,
                  float mult, const float* __restrict__ tprior, int n_tprior, float div,
                  float* __restrict__ scalar_out, int NSL, int act) {
  extern __shared__ float sm[];
  __shared__ float red[NWARPS];
  __shared__ int is_last;
  float* part = sm;                    // [NSL][RB][Z]
  float* dm = part + NSL * RB * Z;     // [RB][Z] dmu
  float* dl = dm + RB * Z;             // [RB][Z] dls
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * RB;
  const float s = w_aux / (float)L;
  const int nchunks = (Z + 7) / 8;
  for (int i = threadIdx.x; i < RB * Z; i += NTHREADS) { dm[i] = 0.f; dl[i] = 0.f; }
  for (int l = 0; l < L; ++l) {
    // dz[r][j] = sum_n da1[(l,m0+r), n] W1[j, n]
    for (int task = warp; task < nchunks * NSL; task += NWARPS) {
      const int c0 = (task % nchunks) * 8, sl = task / nchunks;
      const int nq = min(8, Z - c0);
      const int n_lo = (int)(((long)H * sl) / NSL), n_hi = (int)(((long)H * (sl + 1)) / NSL);
      float acc[RB][8];
#pragma unroll
      for (int r = 0; r < RB; ++r)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[r][q] = 0.f;
      for (int n = n_lo + lane; n < n_hi; n += 32) {
        float wv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) wv[q] = (q < nq) ? W1[(size_t)(c0 + q) * H + n] : 0.f;
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          const float dv = (m0 + r < rows) ? da1[((size_t)l * rows + m0 + r) * H + n] : 0.f;
#pragma unroll
          for (int q = 0; q < 8; ++q) acc[r][q] = fmaf(dv, wv[q], acc[r][q]);
        }
      }
#pragma unroll
      for (int r = 0; r < RB; ++r)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float t = warp_sum(acc[r][q]);
          if (lane == 0 && q < nq) part[(sl * RB + r) * Z + c0 + q] = t;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < RB * Z; i += NTHREADS) {
      const int r = i / Z, j = i % Z, m = m0 + r;
      if (m < rows) {
        float d = 0.f;
        for (int sl = 0; sl < NSL; ++sl) d += part[sl * RB * Z + i];
        const size_t o2 = ((size_t)l * rows + m) * Z + j;
        if (la) d -= s * z[o2];
        const float sd = expf(0.5f * ls[(size_t)m * Z + j]);
        dm[i] += d;
        dl[i] += d * (0.5f * sd * eps[o2]);
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < RB * Z; i += NTHREADS) {
    const int r = i / Z, j = i % Z, m = m0 + r;
    if (m < rows) {
      const float lsv = ls[(size_t)m * Z + j], muv = mu[(size_t)m * Z + j];
      float a = dm[i], b = dl[i];
      if (la) {
        b += w_aux * 0.5f;
      } else {
        a -= w_aux * muv;
        b += w_aux * 0.5f * (1.0f - expf(lsv));
      }
      dm[i] = a;
      dl[i] = b;
      dmu[(size_t)m * Z + j] = a;
      dls[(size_t)m * Z + j] = b;
    }
  }
  __syncthreads();
  // da3[m,n] = (sum_j dmu_j W4[n,j] + dls_j W5[n,j]) * (1 - h_e^2)
  for (int n = threadIdx.x; n < H; n += NTHREADS) {
    float a[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) a[r] = 0.f;
    for (int j = 0; j < Z; ++j) {
      const float w4 = w45t[(size_t)j * H + n], w5 = w45t[(size_t)(Z + j) * H + n];
#pragma unroll
      for (int r = 0; r < RB; ++r) a[r] = fmaf(dm[r * Z + j], w4, fmaf(dl[r * Z + j], w5, a[r]));
    }
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const int m = m0 + r;
      if (m < rows) {
        const float hv = h_e[(size_t)m * H + n];
        const float v = a[r] * act_bwd(hv, act);
        da3[(size_t)m * H + n] = v;
        if (da3_hi) store_split(da3_hi, da3_lo, (size_t)m * ld_mirror + n, v);
      }
    }
  }
  // per-datapoint bound: (1/L) sum_l sum_tiles partial + row_aux   (one warp per row, from the top)
  for (int r = NWARPS - 1 - warp; r < RB; r += NWARPS) {
    const int m = m0 + r;
    if (m < rows) {
      float t = 0.f;
      for (int l = 0; l < L; ++l) {
        const float* p = partial + ((size_t)l * rows + m) * n_tiles;
        for (int q = lane; q < n_tiles; q += 32) t += p[q];
      }
      t = warp_sum(t);
      if (lane == 0) per_row[m] = t / (float)L + row_aux[m];
    }
  }
  // the last block to finish totals the rows in a fixed order (deterministic)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  const float base = block_total(per_row, rows, red);
  float tp = 0.f;
  if (tprior) { __syncthreads(); tp = block_total(tprior, n_tprior, red); }
  if (threadIdx.x == 0) {
    *base_out = base;
    if (scalar_out) *scalar_out = (mult * base + tp) / div;
    *counter = 0u;
  }
}

// Thin weight gradients.  A block owns 64 outputs; its 4 thread groups each take a quarter of the
// row chunk (independent loads, unrolled) and are summed through shared memory in a fixed order.
//   part 0: gW1[j,n] (j<Z) and gb1[n] (j==Z)          = sum_r [z|1][r,j] * da1[r,n]        ((Z+1)*H outputs)
//   part 1: gW4[k,j], gW5[k,j] (k<H), gb4, gb5 (k==H) = sum_m [h_e|1][m,k] * dmu/dls[m,j]  ((H+1)*Z outputs x2)
__global__ void __launch_bounds__(256)
small_wgrad_kernel(const float* __restrict__ z, const float* __restrict__ da1, int R, const float* __restrict__ h_e,
                   const float* __restrict__ dmu, const float* __restrict__ dls, int rows, int H, int Z,
                   int rows_per_chunk, float* __restrict__ gW1, float* __restrict__ gb1, float* __restrict__ gW4,
                   float* __restrict__ gb4, float* __restrict__ gW5, float* __restrict__ gb5,
                   float* __restrict__ scratch) {
  __shared__ float red[2][4][64];
  const int nA = (Z + 1) * H, nB = (H + 1) * Z;
  const int oi = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int i = blockIdx.x * 64 + oi;
  const int chunk = blockIdx.y, nchunks = gridDim.y;
  float a4 = 0.f, a5 = 0.f;
  if (i < nA) {
    const int j = i / H, n = i % H;
    const int Lr = R / rows;
    const int c0 = chunk * rows_per_chunk * Lr, c1 = min(R, c0 + rows_per_chunk * Lr);
    const int per = (c1 - c0 + 3) / 4;
    const int r0 = c0 + grp * per, r1 = min(c1, r0 + per);
    if (j < Z) {
#pragma unroll 8
      for (int r = r0; r < r1; ++r) a4 = fmaf(z[(size_t)r * Z + j], da1[(size_t)r * H + n], a4);
    } else {
#pragma unroll 8
      for (int r = r0; r < r1; ++r) a4 += da1[(size_t)r * H + n];
    }
  } else if (i < nA + nB) {
    const int o = i - nA;
    const int k = o / Z, j = o % Z;
    const int c0 = chunk * rows_per_chunk, c1 = min(rows, c0 + rows_per_chunk);
    const int per = (c1 - c0 + 3) / 4;
    const int r0 = c0 + grp * per, r1 = min(c1, r0 + per);
    if (k < H) {
#pragma unroll 8
      for (int r = r0; r < r1; ++r) {
        const float hv = h_e[(size_t)r * H + k];
        a4 = fmaf(hv, dmu[(size_t)r * Z + j], a4);
        a5 = fmaf(hv, dls[(size_t)r * Z + j], a5);
      }
    } else {
#pragma unroll 8
      for (int r = r0; r < r1; ++r) { a4 += dmu[(size_t)r * Z + j]; a5 += dls[(size_t)r * Z + j]; }
    }
  }
  red[0][grp][oi] = a4;
  red[1][grp][oi] = a5;
  __syncthreads();
  if (grp != 0) return;
  a4 = (red[0][0][oi] + red[0][1][oi]) + (red[0][2][oi] + red[0][3][oi]);
  a5 = (red[1][0][oi] + red[1][1][oi]) + (red[1][2][oi] + red[1][3][oi]);
  if (i < nA) {
    const int j = i / H, n = i % H;
    if (nchunks > 1) scratch[(size_t)chunk * (nA + 2 * nB) + i] = a4;
    else if (j < Z) gW1[(size_t)j * H + n] = a4;
    else gb1[n] = a4;
  } else if (i < nA + nB) {
    const int o = i - nA;
    const int k = o / Z, j = o % Z;
    if (nchunks > 1) {
      scratch[(size_t)chunk * (nA + 2 * nB) + nA + o] = a4;
      scratch[(size_t)chunk * (nA + 2 * nB) + nA + nB + o] = a5;
    } else if (k < H) {
      gW4[(size_t)k * Z + j] = a4;
      gW5[(size_t)k * Z + j] = a5;
    } else {
      gb4[j] = a4;
      gb5[j] = a5;
    }
  }
}

__global__ void __launch_bounds__(256)
small_wgrad_reduce_kernel(const float* __restrict__ scratch, int nchunks, int H, int Z, float* __restrict__ gW1,
                          float* __restrict__ gb1, float* __restrict__ gW4, float* __restrict__ gb4,
                          float* __restrict__ gW5, float* __restrict__ gb5) {
  const int nA = (Z + 1) * H, nB = (H + 1) * Z, tot = nA + 2 * nB;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tot) return;
  float a = 0.f;
  for (int c = 0; c < nchunks; ++c) a += scratch[(size_t)c * tot + i];
  if (i < nA) {
    const int j = i / H, n = i % H;
    if (j < Z) gW1[(size_t)j * H + n] = a; else gb1[n] = a;
  } else {
    const int o = (i - nA) % nB;
    float* gW = (i - nA) < nB ? gW4 : gW5;
    float* gb = (i - nA) < nB ? gb4 : gb5;
    const int k = o / Z, j = o % Z;
    if (k < H) gW[(size_t)k * Z + j] = a; else gb[j] = a;
  }
}


// =====================================================================================================
// Large-batch variants (rows >= LB_MIN_ROWS, L == 1, 2Z <= 48, H <= 512: config c3, M = 16384).  The kernels
// above give one block a handful of rows, which is right for M = 100 and leaves the SMs idle at M = 16384;
// these tile 64 rows per block, stage operands through shared memory and keep 12-48 accumulators per thread.
// =====================================================================================================
constexpr int LB_ROWS = 64, LB_T = 256, LB_KC = 32, LB_WS = 52, LB_NC = 48, LB_ZP = 24;

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// mu|ls = h_e.[W4|W5] + b ; eps, z, row terms ; h_d = tanh(z.W1 + b1)        (VAEB.py:248-254, 41-47, 343)
// Three blocks per SM (80 registers): left to itself ptxas takes 99 and fits two.
__global__ void __launch_bounds__(LB_T, 3)
lb_latent_fwd_kernel(const float* __restrict__ h_e, int rows, int H, const float* __restrict__ w45t,
                     const float* __restrict__ b4, const float* __restrict__ b5, const float* __restrict__ W1,
                     const float* __restrict__ b1, int Z, int la, EpsSource src, float* __restrict__ mu,
                     float* __restrict__ ls, float* __restrict__ eps, float* __restrict__ z,
                     float* __restrict__ row_aux, float* __restrict__ h_d, __nv_bfloat16* __restrict__ hd_hi,
                     __nv_bfloat16* __restrict__ hd_lo, int ld_mirror, int act) {
  __shared__ __align__(16) float hs[LB_ROWS][LB_KC + 1];
  __shared__ __align__(16) float ws[LB_KC][LB_WS];
  __shared__ __align__(16) float outs[LB_ROWS][LB_NC];
  __shared__ __align__(16) float zs[LB_ROWS][LB_ZP];
  __shared__ float terms[LB_ROWS][8];
  const int t = threadIdx.x, m0 = blockIdx.x * LB_ROWS, Z2 = 2 * Z;
  const int r = t >> 2, g = t & 3;
  float acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.f;
  for (int i = t; i < LB_ROWS * LB_ZP; i += LB_T) (&zs[0][0])[i] = 0.f;
  // operand chunks go global -> registers -> shared; the loads of chunk k+1 are in flight while chunk k is contracted
  float hreg[LB_ROWS * LB_KC / LB_T], wreg[LB_KC * LB_NC / LB_T];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < LB_ROWS * LB_KC / LB_T; ++i) {
      const int rr = (t >> 5) + 8 * i, kk = t & 31;
      hreg[i] = (m0 + rr < rows && k0 + kk < H) ? h_e[(size_t)(m0 + rr) * H + k0 + kk] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < LB_KC * LB_NC / LB_T; ++i) {
      const int e = t + LB_T * i, kk = e & 31, c = e >> 5;
      wreg[i] = (c < Z2 && k0 + kk < H) ? w45t[(size_t)c * H + k0 + kk] : 0.f;
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < H; k0 += LB_KC) {
#pragma unroll
    for (int i = 0; i < LB_ROWS * LB_KC / LB_T; ++i) hs[(t >> 5) + 8 * i][t & 31] = hreg[i];
#pragma unroll
    for (int i = 0; i < LB_KC * LB_NC / LB_T; ++i) { const int e = t + LB_T * i; ws[e & 31][e >> 5] = wreg[i]; }
    __syncthreads();
    if (k0 + LB_KC < H) fetch(k0 + LB_KC);
#pragma unroll 8
    for (int kk = 0; kk < LB_KC; ++kk) {
      const float hv = hs[r][kk];
      const float4 w0 = lds4(&ws[kk][g * 12]), w1 = lds4(&ws[kk][g * 12 + 4]), w2 = lds4(&ws[kk][g * 12 + 8]);
      acc[0] = fmaf(hv, w0.x, acc[0]); acc[1] = fmaf(hv, w0.y, acc[1]); acc[2] = fmaf(hv, w0.z, acc[2]);
      acc[3] = fmaf(hv, w0.w, acc[3]); acc[4] = fmaf(hv, w1.x, acc[4]); acc[5] = fmaf(hv, w1.y, acc[5]);
      acc[6] = fmaf(hv, w1.z, acc[6]); acc[7] = fmaf(hv, w1.w, acc[7]); acc[8] = fmaf(hv, w2.x, acc[8]);
      acc[9] = fmaf(hv, w2.y, acc[9]); acc[10] = fmaf(hv, w2.z, acc[10]); acc[11] = fmaf(hv, w2.w, acc[11]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    const int c = g * 12 + i;
    outs[r][c] = acc[i] + (c < Z ? b4[c] : (c < Z2 ? b5[c - Z] : 0.f));
  }
  __syncthreads();
  // reparameterisation + row terms: one item = 4 latent coordinates of one row
  const int nq = (Z + 3) >> 2;
  const bool quad = (Z & 3) == 0 && !src.injected;
  for (int it = t; it < LB_ROWS * nq; it += LB_T) {
    const int rr = it / nq, qd = it - rr * nq, j0 = 4 * qd, m = m0 + rr;
    float term = 0.f;
    if (m < rows) {
      float nrm[4] = {0.f, 0.f, 0.f, 0.f};
      if (quad) philox_normal4(src.seed, src.stream, src.step, 0u, (uint64_t)((src.row_offset + m) * Z + j0) >> 2, nrm);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u;
        if (j < Z) {
          const float am = outs[rr][j], al = outs[rr][Z + j];
          const size_t o2 = (size_t)m * Z + j;
          const float e = src.injected ? src.injected[o2]
                                       : (quad ? nrm[u]
                                               : philox_normal1(src.seed, src.stream, src.step, 0u,
                                                                (uint64_t)((src.row_offset + m) * Z + j)));
          const float zv = am + expf(0.5f * al) * e;
          mu[o2] = am; ls[o2] = al; eps[o2] = e; z[o2] = zv;
          zs[rr][j] = zv;
          term += la ? (-0.5f * zv * zv + 0.5f * al + 0.5f * e * e) : 0.5f * (1.0f + al - am * am - expf(al));
        }
      }
    }
    terms[rr][qd] = term;
  }
  __syncthreads();
  if (t < LB_ROWS && m0 + t < rows) {
    float a = 0.f;
    for (int qd = 0; qd < nq; ++qd) a += terms[t][qd];
    row_aux[m0 + t] = a;
  }
  // decoder hidden layer: one thread per hidden unit, its W1 column in registers across the 64 rows
  for (int n = t; n < H; n += LB_T) {
    float w[LB_ZP];
#pragma unroll
    for (int j = 0; j < LB_ZP; ++j) w[j] = j < Z ? W1[(size_t)j * H + n] : 0.f;
    const float bn = b1[n];
    const int nrows = min(LB_ROWS, rows - m0);
#pragma unroll 2
    for (int rr = 0; rr < nrows; ++rr) {
      const int m = m0 + rr;
      float a = bn;
#pragma unroll
      for (int q = 0; q < LB_ZP / 4; ++q) {
        const float4 zq = lds4(&zs[rr][4 * q]);
        a = fmaf(zq.x, w[4 * q], a); a = fmaf(zq.y, w[4 * q + 1], a);
        a = fmaf(zq.z, w[4 * q + 2], a); a = fmaf(zq.w, w[4 * q + 3], a);
      }
      const float hv = act_fwd(a, act);
      h_d[(size_t)m * H + n] = hv;
      if (hd_hi) store_split(hd_hi, hd_lo, (size_t)m * ld_mirror + n, hv);
    }
  }
}

// dz = da1.W1^T ; dmu, dls ; da3 = ([dmu|dls].[W4|W5]^T) * (1 - h_e^2) ; per-row bound and its total
__global__ void __launch_bounds__(LB_T)
lb_latent_bwd_kernel(const float* __restrict__ da1, const float* __restrict__ W1, const float* __restrict__ w45t,
                     const float* __restrict__ h_e, const float* __restrict__ z, const float* __restrict__ eps,
                     const float* __restrict__ mu, const float* __restrict__ ls, int rows, int H, int Z, int la,
                     float w_aux, float* __restrict__ dmu, float* __restrict__ dls, float* __restrict__ da3,
                     const float* __restrict__ partial, int n_tiles, const float* __restrict__ row_aux,
                     float* __restrict__ per_row, unsigned int* __restrict__ counter, float* __restrict__ base_out,
                     float mult, const float* __restrict__ tprior, int n_tprior, float div,
                     float* __restrict__ scalar_out, int act) {
  __shared__ __align__(16) float ds[LB_ROWS][LB_KC + 1];
  __shared__ __align__(16) float ws[LB_KC][28];
  __shared__ __align__(16) float psum[2][LB_ROWS][LB_ZP];
  __shared__ __align__(16) float dd[LB_ROWS][LB_NC];
  __shared__ float red[LB_T / 32];
  __shared__ int is_last;
  const int t = threadIdx.x, m0 = blockIdx.x * LB_ROWS;
  const int r = t >> 2, g = (t >> 1) & 1, ks = t & 1;
  float acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.f;
  for (int i = t; i < LB_ROWS * LB_NC; i += LB_T) (&dd[0][0])[i] = 0.f;
  float dreg[LB_ROWS * LB_KC / LB_T], wreg[LB_KC * LB_ZP / LB_T];
  auto fetch = [&](int n0) {
#pragma unroll
    for (int i = 0; i < LB_ROWS * LB_KC / LB_T; ++i) {
      const int rr = (t >> 5) + 8 * i, kk = t & 31;
      dreg[i] = (m0 + rr < rows && n0 + kk < H) ? da1[(size_t)(m0 + rr) * H + n0 + kk] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < LB_KC * LB_ZP / LB_T; ++i) {
      const int e = t + LB_T * i, kk = e & 31, j = e >> 5;
      wreg[i] = (j < Z && n0 + kk < H) ? W1[(size_t)j * H + n0 + kk] : 0.f;
    }
  };
  fetch(0);
  for (int n0 = 0; n0 < H; n0 += LB_KC) {
#pragma unroll
    for (int i = 0; i < LB_ROWS * LB_KC / LB_T; ++i) ds[(t >> 5) + 8 * i][t & 31] = dreg[i];
#pragma unroll
    for (int i = 0; i < LB_KC * LB_ZP / LB_T; ++i) { const int e = t + LB_T * i; ws[e & 31][e >> 5] = wreg[i]; }
    __syncthreads();
    if (n0 + LB_KC < H) fetch(n0 + LB_KC);
#pragma unroll 8
    for (int q = 0; q < LB_KC / 2; ++q) {
      const int kk = ks * (LB_KC / 2) + q;
      const float dv = ds[r][kk];
      const float4 w0 = lds4(&ws[kk][g * 12]), w1 = lds4(&ws[kk][g * 12 + 4]), w2 = lds4(&ws[kk][g * 12 + 8]);
      acc[0] = fmaf(dv, w0.x, acc[0]); acc[1] = fmaf(dv, w0.y, acc[1]); acc[2] = fmaf(dv, w0.z, acc[2]);
      acc[3] = fmaf(dv, w0.w, acc[3]); acc[4] = fmaf(dv, w1.x, acc[4]); acc[5] = fmaf(dv, w1.y, acc[5]);
      acc[6] = fmaf(dv, w1.z, acc[6]); acc[7] = fmaf(dv, w1.w, acc[7]); acc[8] = fmaf(dv, w2.x, acc[8]);
      acc[9] = fmaf(dv, w2.y, acc[9]); acc[10] = fmaf(dv, w2.z, acc[10]); acc[11] = fmaf(dv, w2.w, acc[11]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) psum[ks][r][g * 12 + i] = acc[i];
  __syncthreads();
  for (int it = t; it < LB_ROWS * Z; it += LB_T) {
    const int rr = it / Z, j = it - rr * Z, m = m0 + rr;
    if (m < rows) {
      const size_t o2 = (size_t)m * Z + j;
      const float lsv = ls[o2], muv = mu[o2];
      float d = psum[0][rr][j] + psum[1][rr][j];
      if (la) d -= w_aux * z[o2];
      float a = d, b = d * (0.5f * expf(0.5f * lsv) * eps[o2]);
      if (la) {
        b += w_aux * 0.5f;
      } else {
        a -= w_aux * muv;
        b += w_aux * 0.5f * (1.0f - expf(lsv));
      }
      dmu[o2] = a; dls[o2] = b;
      dd[rr][j] = a; dd[rr][Z + j] = b;
    }
  }
  __syncthreads();
  for (int n = t; n < H; n += LB_T) {
    float wr[LB_NC];
#pragma unroll
    for (int c = 0; c < LB_NC; ++c) wr[c] = c < 2 * Z ? w45t[(size_t)c * H + n] : 0.f;
    const int nrows = min(LB_ROWS, rows - m0);
#pragma unroll 4
    for (int rr = 0; rr < nrows; ++rr) {
      const int m = m0 + rr;
      float a = 0.f;
#pragma unroll
      for (int q = 0; q < LB_NC / 4; ++q) {
        const float4 dq = lds4(&dd[rr][4 * q]);
        a = fmaf(dq.x, wr[4 * q], a); a = fmaf(dq.y, wr[4 * q + 1], a);
        a = fmaf(dq.z, wr[4 * q + 2], a); a = fmaf(dq.w, wr[4 * q + 3], a);
      }
      const float hv = h_e[(size_t)m * H + n];
      const float v = a * act_bwd(hv, act);
      da3[(size_t)m * H + n] = v;
    }
  }
  // per-datapoint bound: sum of the log-likelihood tile partials + the KL / LA row term
  if (t < LB_ROWS && m0 + t < rows) {
    const float* pp = partial + (size_t)(m0 + t) * n_tiles;
    float a = 0.f;
    for (int q = 0; q < n_tiles; ++q) a += pp[q];
    per_row[m0 + t] = a + row_aux[m0 + t];
  }
  __threadfence();
  __syncthreads();
  if (t == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  const float base = block_total(per_row, rows, red);
  float tp = 0.f;
  if (tprior) { __syncthreads(); tp = block_total(tprior, n_tprior, red); }
  if (t == 0) {
    *base_out = base;
    if (scalar_out) *scalar_out = (mult * base + tp) / div;
    *counter = 0u;
  }
}

// Thin weight gradients at large batch: split the rows into chunks of LB_WG_ROWS, every block reduces its
// chunk for 128 outputs rows x all columns, partials go to scratch[chunk] and small_wgrad_reduce_kernel sums
// them in a fixed order.  scratch layout per chunk = [(Z+1)*H | (H+1)*Z | (H+1)*Z] as above.
constexpr int LB_WG_ROWS = 128, LB_WG_T = 128, LB_WG_SUB = 32;

// gW4|gW5 (and gb4|gb5 as row k == H) = [h_e|1]^T.[dmu|dls]: thread = hidden index k, 48 accumulators
__global__ void __launch_bounds__(LB_WG_T)
lb_wgrad45_kernel(const float* __restrict__ h_e, const float* __restrict__ dmu, const float* __restrict__ dls, int rows,
                  int H, int Z, float* __restrict__ scratch) {
  __shared__ __align__(16) float dsm[LB_WG_SUB][LB_NC];
  const int t = threadIdx.x, k = blockIdx.x * LB_WG_T + t, chunk = blockIdx.y;
  const int r_lo = chunk * LB_WG_ROWS, r_hi = min(rows, r_lo + LB_WG_ROWS);
  float acc[LB_NC];
#pragma unroll
  for (int c = 0; c < LB_NC; ++c) acc[c] = 0.f;
  for (int r0 = r_lo; r0 < r_hi; r0 += LB_WG_SUB) {
    for (int i = t; i < LB_WG_SUB * LB_NC; i += LB_WG_T) {
      const int rr = i / LB_NC, c = i - rr * LB_NC, m = r0 + rr;
      float v = 0.f;
      if (m < r_hi) v = c < Z ? dmu[(size_t)m * Z + c] : (c < 2 * Z ? dls[(size_t)m * Z + c - Z] : 0.f);
      dsm[rr][c] = v;
    }
    __syncthreads();
    if (k <= H) {
      const int nr = min(LB_WG_SUB, r_hi - r0);
#pragma unroll 8
      for (int rr = 0; rr < nr; ++rr) {
        const float hv = k < H ? h_e[(size_t)(r0 + rr) * H + k] : 1.0f;
#pragma unroll
        for (int q = 0; q < LB_NC / 4; ++q) {
          const float4 d = lds4(&dsm[rr][4 * q]);
          acc[4 * q] = fmaf(hv, d.x, acc[4 * q]); acc[4 * q + 1] = fmaf(hv, d.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(hv, d.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(hv, d.w, acc[4 * q + 3]);
        }
      }
    }
    __syncthreads();
  }
  if (k > H) return;
  const int nA = (Z + 1) * H, nB = (H + 1) * Z;
  float* out = scratch + (size_t)chunk * (nA + 2 * nB) + nA;
#pragma unroll
  for (int c = 0; c < LB_NC; ++c) {
    if (c < Z) out[(size_t)k * Z + c] = acc[c];
    else if (c < 2 * Z) out[(size_t)nB + (size_t)k * Z + (c - Z)] = acc[c];
  }
}

// gW1 (and gb1 as row j == Z) = [z|1]^T.da1: thread = hidden index n, 24 accumulators
__global__ void __launch_bounds__(LB_WG_T)
lb_wgrad1_kernel(const float* __restrict__ z, const float* __restrict__ da1, int rows, int H, int Z,
                 float* __restrict__ scratch) {
  __shared__ __align__(16) float zsm[LB_WG_SUB][LB_ZP];
  const int t = threadIdx.x, n = blockIdx.x * LB_WG_T + t, chunk = blockIdx.y;
  const int r_lo = chunk * LB_WG_ROWS, r_hi = min(rows, r_lo + LB_WG_ROWS);
  float acc[LB_ZP];
#pragma unroll
  for (int j = 0; j < LB_ZP; ++j) acc[j] = 0.f;
  for (int r0 = r_lo; r0 < r_hi; r0 += LB_WG_SUB) {
    for (int i = t; i < LB_WG_SUB * LB_ZP; i += LB_WG_T) {
      const int rr = i / LB_ZP, j = i - rr * LB_ZP, m = r0 + rr;
      float v = 0.f;
      if (m < r_hi) v = j < Z ? z[(size_t)m * Z + j] : (j == Z ? 1.0f : 0.f);
      zsm[rr][j] = v;
    }
    __syncthreads();
    if (n < H) {
      const int nr = min(LB_WG_SUB, r_hi - r0);
#pragma unroll 8
      for (int rr = 0; rr < nr; ++rr) {
        const float dv = da1[(size_t)(r0 + rr) * H + n];
#pragma unroll
        for (int q = 0; q < LB_ZP / 4; ++q) {
          const float4 zq = lds4(&zsm[rr][4 * q]);
          acc[4 * q] = fmaf(dv, zq.x, acc[4 * q]); acc[4 * q + 1] = fmaf(dv, zq.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(dv, zq.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(dv, zq.w, acc[4 * q + 3]);
        }
      }
    }
    __syncthreads();
  }
  if (n >= H) return;
  const int nA = (Z + 1) * H, nB = (H + 1) * Z;
  float* out = scratch + (size_t)chunk * (nA + 2 * nB);
#pragma unroll
  for (int j = 0; j < LB_ZP; ++j)
    if (j <= Z) out[(size_t)j * H + n] = acc[j];
}

}  // namespace

cudaError_t launch_transpose_heads(cudaStream_t st, int64_t* launches, const float* W4, const float* W5, int H, int Z,
                                   float* w45t) {
  transpose_heads_kernel<<<(2 * Z * H + 255) / 256, 256, 0, st>>>(W4, W5, H, Z, w45t);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_latent_fwd(cudaStream_t st, int64_t* launches, const float* h_e, int rows, int H,
                              const float* w45t, const float* b4, const float* b5, const float* W1, const float* b1,
                              int Z, int L, int la, EpsSource src, float* mu, float* ls, float* eps, float* z,
                              float* row_aux, float* h_d, void* hd_hi, void* hd_lo, int ld_mirror, int act) {
  const int nchunks = (2 * Z + 7) / 8;
  const int KS = max(1, NWARPS / nchunks);
  ++*launches;
  if (latent_lb_supported(rows, H, Z, L)) {
    lb_latent_fwd_kernel<<<(rows + LB_ROWS - 1) / LB_ROWS, LB_T, 0, st>>>(
        h_e, rows, H, w45t, b4, b5, W1, b1, Z, la, src, mu, ls, eps, z, row_aux, h_d, (__nv_bfloat16*)hd_hi,
        (__nv_bfloat16*)hd_lo, ld_mirror, act);
  } else if (rows <= 512) {
    const size_t smem = (size_t)((KS + 1) * 2 * Z + 2 * Z) * sizeof(float);
    latent_fwd_kernel<1><<<rows, NTHREADS, smem, st>>>(h_e, rows, H, w45t, b4, b5, W1, b1, Z, L, la, src, mu, ls, eps,
                                                      z, row_aux, h_d, (__nv_bfloat16*)hd_hi, (__nv_bfloat16*)hd_lo,
                                                      ld_mirror, KS, act);
  } else {
    constexpr int RB = 8;
    const size_t smem = (size_t)RB * ((KS + 1) * 2 * Z + 2 * Z) * sizeof(float);
    latent_fwd_kernel<RB><<<(rows + RB - 1) / RB, NTHREADS, smem, st>>>(
        h_e, rows, H, w45t, b4, b5, W1, b1, Z, L, la, src, mu, ls, eps, z, row_aux, h_d, (__nv_bfloat16*)hd_hi,
        (__nv_bfloat16*)hd_lo, ld_mirror, KS, act);
  }
  return cudaGetLastError();
}

cudaError_t launch_latent_bwd(cudaStream_t st, int64_t* launches, const float* da1, const float* W1,
                              const float* w45t, const float* h_e, const float* z, const float* eps, const float* mu,
                              const float* ls, int rows, int H, int Z, int L, int la, float w_aux, float* dmu, float* dls,
                              float* da3, void* da3_hi, void* da3_lo, int ld_mirror, const float* partial,
                              int n_tiles, const float* row_aux, float* per_row, unsigned int* counter,
                              float* base_out, float mult, const float* tprior, int n_tprior, float div,
                              float* scalar_out, int act) {
  const int nchunks = (Z + 7) / 8;
  const int NSL = max(1, (NWARPS - 2) / nchunks);
  ++*launches;
  if (latent_lb_supported(rows, H, Z, L)) {
    lb_latent_bwd_kernel<<<(rows + LB_ROWS - 1) / LB_ROWS, LB_T, 0, st>>>(
        da1, W1, w45t, h_e, z, eps, mu, ls, rows, H, Z, la, w_aux, dmu, dls, da3, partial, n_tiles, row_aux, per_row,
        counter, base_out, mult, tprior, n_tprior, div, scalar_out, act);
  } else if (rows <= 512) {
    const size_t smem = (size_t)(NSL + 2) * Z * sizeof(float);
    latent_bwd_kernel<1><<<rows, NTHREADS, smem, st>>>(
        da1, W1, w45t, h_e, z, eps, mu, ls, rows, H, Z, L, la, w_aux, dmu, dls, da3, (__nv_bfloat16*)da3_hi,
        (__nv_bfloat16*)da3_lo, ld_mirror, partial, n_tiles, row_aux, per_row, counter, base_out, mult, tprior,
        n_tprior, div, scalar_out, NSL, act);
  } else {
    constexpr int RB = 8;
    const size_t smem = (size_t)RB * (NSL + 2) * Z * sizeof(float);
    latent_bwd_kernel<RB><<<(rows + RB - 1) / RB, NTHREADS, smem, st>>>(
        da1, W1, w45t, h_e, z, eps, mu, ls, rows, H, Z, L, la, w_aux, dmu, dls, da3, (__nv_bfloat16*)da3_hi,
        (__nv_bfloat16*)da3_lo, ld_mirror, partial, n_tiles, row_aux, per_row, counter, base_out, mult, tprior,
        n_tprior, div, scalar_out, NSL, act);
  }
  return cudaGetLastError();
}

bool latent_large_batch(int rows, int H, int Z, int L) { return latent_lb_supported(rows, H, Z, L); }

int small_wgrad_chunks(int rows) { return rows <= 512 ? 1 : (rows + 255) / 256; }
size_t small_wgrad_scratch_elems(int rows, int H, int Z) {
  const int c = rows >= LB_MIN_ROWS ? (rows + LB_WG_ROWS - 1) / LB_WG_ROWS : small_wgrad_chunks(rows);
  return c > 1 ? (size_t)c * ((size_t)(Z + 1) * H + 2 * (size_t)(H + 1) * Z) : 0;
}

cudaError_t launch_small_wgrad(cudaStream_t st, int64_t* launches, const float* z, const float* da1, int R,
                               const float* h_e, const float* dmu, const float* dls, int rows, int H, int Z,
                               float* gW1, float* gb1, float* gW4, float* gb4, float* gW5, float* gb5,
                               float* scratch) {
  if (latent_lb_supported(rows, H, Z, R / rows)) {
    const int chunks = (rows + LB_WG_ROWS - 1) / LB_WG_ROWS;
    lb_wgrad45_kernel<<<dim3((H + 1 + LB_WG_T - 1) / LB_WG_T, chunks), LB_WG_T, 0, st>>>(h_e, dmu, dls, rows, H, Z, scratch);
    lb_wgrad1_kernel<<<dim3((H + LB_WG_T - 1) / LB_WG_T, chunks), LB_WG_T, 0, st>>>(z, da1, rows, H, Z, scratch);
    const int all = (Z + 1) * H + 2 * (H + 1) * Z;
    small_wgrad_reduce_kernel<<<(all + 255) / 256, 256, 0, st>>>(scratch, chunks, H, Z, gW1, gb1, gW4, gb4, gW5, gb5);
    *launches += 3;
    return cudaGetLastError();
  }
  const int tot = (Z + 1) * H + (H + 1) * Z;
  const int chunks = small_wgrad_chunks(rows);
  const int rpc = chunks > 1 ? 256 : rows;
  dim3 grid((tot + 63) / 64, chunks);
  small_wgrad_kernel<<<grid, 256, 0, st>>>(z, da1, R, h_e, dmu, dls, rows, H, Z, rpc, gW1, gb1, gW4, gb4, gW5, gb5,
                                          scratch);
  ++*launches;
  if (chunks > 1) {
    const int all = (Z + 1) * H + 2 * (H + 1) * Z;
    small_wgrad_reduce_kernel<<<(all + 255) / 256, 256, 0, st>>>(scratch, chunks, H, Z, gW1, gb1, gW4, gb4, gW5, gb5);
    ++*launches;
  }
  return cudaGetLastError();
}
