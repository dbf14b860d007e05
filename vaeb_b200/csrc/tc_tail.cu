// The tail of a large-batch AEVB update as ONE launch (config C3): sum of the split-K weight-gradient slices, the
// minibatch bound, the cross-GPU gradient sum, prior + Adagrad (VAEB.py:389-390, 426-444) and the bf16 operand mirrors
// of the updated weights for the next step.  Round 1 spent five launches and an un-overlapped ncclAllReduce here.
//
// One GPU:   P1 slices -> g, Adagrad in place (a thread owns a parameter; fixed summation order) ‖ per-row bounds
//            -- grid barrier -- P3 mirrors of the new weights ‖ total bound (block 0, fixed order).
// N GPUs (data parallel, one process per GPU; the buffers below are mapped into every rank with CUDA IPC):
//            P1 slices -> this rank's gsum buffer ‖ per-row bounds       -- grid barrier, "staged" flag to every peer --
//            P2 rank r owns flat slice r: loads it from every rank's gsum over NVLink (fixed rank order: every rank
//               would get the same bits, but only the owner computes), Adagrad, STORES the new parameters and
//               accumulators into every rank's buffers (reduce-scatter + all-gather of a 3.26 MB buffer, no NCCL
//               kernel, no host)                                         -- grid barrier, "done" flag to every peer --
//            P3 after every peer's slice has landed: mirrors of the new weights.
// Flags are monotonic launch numbers written with st.release.sys into the PEER's flag array and polled locally.
// The rule is a template parameter: prior + Adagrad, or Adam (adam.cuh), whose owner of a slice also stores the two
// moments into every rank's buffers, so that they stay replicated and identical on all ranks.
#include <cuda_bf16.h>
#include <cstdlib>

#include "adam.cuh"
#include "common.cuh"
#include "launchers.h"
#include "tc_layers.h"

namespace {

constexpr int TAIL_THREADS = 256;

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// flag stores: ONE system-scope fence, then relaxed stores to every peer (a st.release.sys per peer would wait for the
// acknowledgement of the previous remote store each time: ~2.5 us x 8 peers, measured)
__device__ __forceinline__ void st_relaxed_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// another GPU's memory: system-scope relaxed loads (never served by L1; unlike ld.volatile they are not ordered among
// themselves, so eight of them overlap -- with ld.volatile the eight peers' loads of P2 took 8 x 2.2 us)
__device__ __forceinline__ float4 ld_peer4(const float* p) {
  float4 v;
  asm("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_peer1(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// every CTA of the (co-resident) grid arrives; monotonic counter, `target` = arrivals expected by now
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(bar), "r"(1u) : "memory");
    uint32_t spins = 0;
    while ((int)(ld_acquire_gpu(bar) - target) < 0) {
      if (++spins > 400000000u) __trap();
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = 0.f;
  if (w == 0) {
    t = l < (int)(blockDim.x >> 5) ? red[l] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;      // valid in warp 0
}

__device__ __forceinline__ void adagrad_one(float& p, float& a, float g, float lr, float eps, float prior, float p2) {
  g -= prior * p;                                  // VAEB.py:389-390
  a = a + g * g;                                   // VAEB.py:439
  float np_ = p + lr * g / (sqrtf(a) + eps);       // VAEB.py:441
  if (p2 != 0.f) np_ -= p2 * p * p;                // VAEBfullbayes.py:183-184
  p = np_;
}

__device__ __forceinline__ void put_pair(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t o, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[o] = h;
  if (lo) lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
}

template <bool ADAM>
__global__ void __launch_bounds__(TAIL_THREADS)
tc_tail_kernel(const TcTailArgs a) {
  __shared__ float red[32];
  // programmatic dependent launch: the grid is scheduled while the weight-gradient launch drains
  // (its CTAs fill the SMs: nothing of this grid becomes resident before they exit); nothing is read before this point
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  unsigned int bar_target = a.bar_base;
  const bool dp = a.world > 1;

  // ---- P1: split-K slices -> gradient (fixed order); one GPU: prior + Adagrad right here -----------------------
  // Four consecutive elements per thread (16-byte accesses) wherever a job's slices and its place in the flat buffers
  // are 16-byte aligned -- every tensor of the MNIST / Frey shapes is -- else one.
  for (int q = 0; q < a.jobs.n; ++q) {
    const TcReduceJob& j = a.jobs.job[q];
    const int n = j.n_w + j.n_b;
    int n_vec = 0;                                   // elements [0, n_vec) go four at a time
    if (j.kind == 0 && (j.n_w & 3) == 0 && (j.stride & 3) == 0 && ((((uintptr_t)j.scratch) | ((uintptr_t)j.gW)) & 15u) == 0 &&
        ((j.gW - a.grads) & 3) == 0)
      n_vec = j.n_w;
    for (int i4 = (int)tid; i4 < n_vec / 4; i4 += (int)nth) {
      const float4* sp = reinterpret_cast<const float4*>(j.scratch) + i4;
      const size_t st4 = j.stride / 4;
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      int z = 0;
      for (; z + 2 <= j.splits; z += 2) {
        const float4 t0 = __ldcg(sp + (size_t)z * st4), t1 = __ldcg(sp + (size_t)(z + 1) * st4);
        g.x += t0.x; g.y += t0.y; g.z += t0.z; g.w += t0.w;
        g.x += t1.x; g.y += t1.y; g.z += t1.z; g.w += t1.w;
      }
      for (; z < j.splits; ++z) {
        const float4 t0 = __ldcg(sp + (size_t)z * st4);
        g.x += t0.x; g.y += t0.y; g.z += t0.z; g.w += t0.w;
      }
      const size_t f4 = (size_t)(j.gW - a.grads) / 4 + i4;
      if (dp) {
        reinterpret_cast<float4*>(a.gsum[a.rank])[f4] = g;
      } else if constexpr (ADAM) {
        reinterpret_cast<float4*>(a.grads)[f4] = g;
        float4 p = reinterpret_cast<const float4*>(a.params)[f4], m = reinterpret_cast<const float4*>(a.ada)[f4],
               v = reinterpret_cast<const float4*>(a.v)[f4];
        adam1(p.x, m.x, v.x, g.x, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.y, m.y, v.y, g.y, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.z, m.z, v.z, g.z, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.w, m.w, v.w, g.w, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        reinterpret_cast<float4*>(a.params)[f4] = p;
        reinterpret_cast<float4*>(a.ada)[f4] = m;
        reinterpret_cast<float4*>(a.v)[f4] = v;
      } else {
        reinterpret_cast<float4*>(a.grads)[f4] = g;
        float4 p = reinterpret_cast<const float4*>(a.params)[f4], ac = reinterpret_cast<const float4*>(a.ada)[f4];
        adagrad_one(p.x, ac.x, g.x, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.y, ac.y, g.y, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.z, ac.z, g.z, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.w, ac.w, g.w, a.lr, a.eps, a.prior, a.p2);
        reinterpret_cast<float4*>(a.params)[f4] = p;
        reinterpret_cast<float4*>(a.ada)[f4] = ac;
      }
    }
    for (int i = n_vec + (int)tid; i < n; i += (int)nth) {
      // the slices are summed in slice order (deterministic); four loads in flight per thread
      float g = 0.f;
      const float* sp = j.scratch + i;
      int z = 0;
      for (; z + 4 <= j.splits; z += 4) {
        const float t0 = __ldcg(sp + (size_t)z * j.stride), t1 = __ldcg(sp + (size_t)(z + 1) * j.stride),
                    t2 = __ldcg(sp + (size_t)(z + 2) * j.stride), t3 = __ldcg(sp + (size_t)(z + 3) * j.stride);
        g += t0; g += t1; g += t2; g += t3;
      }
      for (; z < j.splits; ++z) g += __ldcg(sp + (size_t)z * j.stride);
      float* dst;      // the element's place in the flat gradient buffer
      if (j.kind == 0) {
        dst = i < j.n_w ? j.gW + i : j.gb + (i - j.n_w);
      } else if (j.kind == 2) {   // interleaved Gaussian head [(H+1) x 2D]: column 2d -> W2 / b2, 2d + 1 -> W6 / b6
        const int D = j.Z, H = j.H;
        const int k = i / (2 * D), c = i - k * 2 * D, d = c >> 1;
        dst = k < H ? ((c & 1) ? j.gW2 : j.gW) + (size_t)k * D + d : ((c & 1) ? j.gb2 : j.gb) + d;
      } else {         // interleaved heads slice [(H+1) x 2Z]: column c < Z -> W4 / b4, else W5 / b5
        const int Z = j.Z, H = j.H;
        const int k = i / (2 * Z), c = i - k * 2 * Z;
        const int jj = c < Z ? c : c - Z;
        dst = k < H ? (c < Z ? j.gW : j.gW2) + (size_t)k * Z + jj : (c < Z ? j.gb : j.gb2) + jj;
      }
      const size_t f = (size_t)(dst - a.grads);
      if (dp) {
        a.gsum[a.rank][f] = g;
      } else if constexpr (ADAM) {
        *dst = g;
        float p = a.params[f], m = a.ada[f], v = a.v[f];
        adam1(p, m, v, g, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        a.params[f] = p;
        a.ada[f] = m;
        a.v[f] = v;
      } else {
        *dst = g;
        float p = a.params[f], ac = a.ada[f];
        adagrad_one(p, ac, g, a.lr, a.eps, a.prior, a.p2);
        a.params[f] = p;
        a.ada[f] = ac;
      }
    }
  }
  // ---- per-row bounds (VAEB.py:343-347): row m = its log-likelihood partials + its KL / L^A term ----------------
  float v = 0.f;
  for (int64_t m = tid; m < a.rows; m += nth) {
    float t = 0.f;
    const float* p = a.partial + (size_t)m * a.n_tiles;
    for (int q = 0; q < a.n_tiles; ++q) t += p[q];
    float u = 0.f;
    if (a.aux_part) {
      for (int q = 0; q < a.n_aux; ++q) u += a.aux_part[(size_t)m * a.n_aux + q];
    } else {
      u = a.row_aux[m];
    }
    t += u;
    a.per_row[m] = t;
    v += t;
  }
  const float bs = block_sum(v, red);
  if (threadIdx.x == 0) a.block_part[blockIdx.x] = bs;
  bar_target += gridDim.x;
  grid_barrier(a.bar, bar_target);

  // total bound of this rank: block 0, fixed order
  float base = 0.f;
  if (blockIdx.x == 0) {
    float t = 0.f;
    for (int r = threadIdx.x; r < (int)gridDim.x; r += blockDim.x) t += __ldcg(a.block_part + r);
    base = block_sum(t, red);
    if (threadIdx.x == 0) {
      *a.base_out = base;
      if (!dp) {
        if (a.scalar_out) *a.scalar_out = (a.mult * base) / a.div;
      } else {
        a.gsum[a.rank][a.padded] = base;              // travels with the gradient
      }
    }
    if (dp) {                                         // "staged": thread r tells peer r
      __syncthreads();
      if (threadIdx.x < a.world) {
        __threadfence_system();
        st_relaxed_sys(a.flags[threadIdx.x] + a.rank, a.epoch);
      }
    }
  }

  if (dp) {
    // ---- P2: my slice of the flat buffer: sum over ranks, Adagrad, new parameters to every rank ------------------
    if (threadIdx.x == 0) {
      for (int r = 0; r < a.world; ++r) {
        uint32_t spins = 0;
        while ((int)(ld_acquire_sys(a.flags[a.rank] + r) - a.epoch) < 0) {
          if (++spins > 400000000u) __trap();
        }
      }
    }
    __syncthreads();
    const int64_t n4 = a.padded / 4;
    const int64_t per = (n4 + a.world - 1) / a.world;
    const int64_t lo = per * a.rank, hi = lo + per < n4 ? lo + per : n4;
    for (int64_t i = lo + tid; i < hi; i += nth) {
      // every peer's copy of the four elements is requested before the first one is used (a remote load is ~2.5 us)
      float4 t[TC_MAX_PEERS];
#pragma unroll
      for (int r = 0; r < TC_MAX_PEERS; ++r)
        if (r < a.world) t[r] = ld_peer4(a.gsum[r] + 4 * i);
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < TC_MAX_PEERS; ++r)
        if (r < a.world) { g.x += t[r].x; g.y += t[r].y; g.z += t[r].z; g.w += t[r].w; }
      if constexpr (ADAM) {
        float4 p = reinterpret_cast<const float4*>(a.params)[i], m = reinterpret_cast<const float4*>(a.ada)[i],
               v = reinterpret_cast<const float4*>(a.v)[i];
        adam1(p.x, m.x, v.x, g.x, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.y, m.y, v.y, g.y, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.z, m.z, v.z, g.z, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        adam1(p.w, m.w, v.w, g.w, a.alpha_t, a.s2_t, a.b1, a.b2, a.adam_eps, a.prior);
        for (int r = 0; r < a.world; ++r) {
          reinterpret_cast<float4*>(a.peer_params[r])[i] = p;
          reinterpret_cast<float4*>(a.peer_ada[r])[i] = m;
          reinterpret_cast<float4*>(a.peer_v[r])[i] = v;
        }
      } else {
        float4 p = reinterpret_cast<const float4*>(a.params)[i], ac = reinterpret_cast<const float4*>(a.ada)[i];
        adagrad_one(p.x, ac.x, g.x, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.y, ac.y, g.y, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.z, ac.z, g.z, a.lr, a.eps, a.prior, a.p2);
        adagrad_one(p.w, ac.w, g.w, a.lr, a.eps, a.prior, a.p2);
        for (int r = 0; r < a.world; ++r) {
          reinterpret_cast<float4*>(a.peer_params[r])[i] = p;
          reinterpret_cast<float4*>(a.peer_ada[r])[i] = ac;
        }
      }
    }
    if (tid == 0 && a.scalar_out) {       // the bound of the global minibatch (every rank sums the same values in rank order)
      float t = 0.f;
      for (int r = 0; r < a.world; ++r) t += ld_peer1(a.gsum[r] + a.padded);
      *a.scalar_out = (a.mult * t) / a.div;
    }
    __threadfence_system();
    bar_target += gridDim.x;
    grid_barrier(a.bar, bar_target);
    if (blockIdx.x == 0 && threadIdx.x < a.world) {      // "my slice is everywhere": thread r tells peer r
      __threadfence_system();
      st_relaxed_sys(a.flags[threadIdx.x] + a.world + a.rank, a.epoch);
    }
    if (threadIdx.x == 0) {
      for (int r = 0; r < a.world; ++r) {
        uint32_t spins = 0;
        while ((int)(ld_acquire_sys(a.flags[a.rank] + a.world + r) - a.epoch) < 0) {
          if (++spins > 400000000u) __trap();
        }
      }
    }
    __syncthreads();
  }

  // ---- P3: bf16 (hi, lo) operand mirrors of the new weights, in the layouts the TMA maps of the next step read --------
  if (!a.w3h) return;
  const int D = a.D, H = a.H, Z = a.Z;
  const float* W3 = a.params + a.oW3; const float* W4 = a.params + a.oW4; const float* W5 = a.params + a.oW5;
  const float* W1 = a.params + a.oW1; const float* W2 = a.params + a.oW2;
  __nv_bfloat16 *w3h = (__nv_bfloat16*)a.w3h, *w3l = (__nv_bfloat16*)a.w3l, *w2h = (__nv_bfloat16*)a.w2h,
                *w2l = (__nv_bfloat16*)a.w2l, *w45h = (__nv_bfloat16*)a.w45h, *w45l = (__nv_bfloat16*)a.w45l,
                *whh = (__nv_bfloat16*)a.whh, *whl = (__nv_bfloat16*)a.whl, *w1h = (__nv_bfloat16*)a.w1h,
                *w1l = (__nv_bfloat16*)a.w1l;
  const int t32 = (int)tid, n32 = (int)nth;
  // row-major fp32 [rows, cols] -> bf16 (hi, lo) mirror [rows, ld]: four elements per thread (16-byte loads, 8-byte
  // stores) when cols and ld are multiples of 4, else one
  auto mirror = [&](const float* W, __nv_bfloat16* hi, __nv_bfloat16* lo, int rows, int cols, int ld) {
    if ((cols & 3) == 0 && (ld & 3) == 0 && (((uintptr_t)W) & 15u) == 0 && ((((uintptr_t)hi) | ((uintptr_t)lo)) & 7u) == 0) {
      const int c4 = cols / 4;
      for (int i = t32; i < rows * c4; i += n32) {
        const int r = i / c4, c = (i - r * c4) * 4;
        const float4 v = __ldcg(reinterpret_cast<const float4*>(W) + i);
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
        const size_t o = (size_t)r * ld + c;
        *reinterpret_cast<uint2*>(hi + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
        if (lo) {
          const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - __low2float(h0), v.y - __high2float(h0));
          const __nv_bfloat162 l1 = __floats2bfloat162_rn(v.z - __low2float(h1), v.w - __high2float(h1));
          *reinterpret_cast<uint2*>(lo + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
        }
      }
    } else {
      for (int i = t32; i < rows * cols; i += n32) {
        const int r = i / cols, c = i - r * cols;
        put_pair(hi, lo, (size_t)r * ld + c, __ldcg(W + i));
      }
    }
  };
  mirror(W3, w3h, w3l, D, H, a.ldh);
  if (a.oW6 >= 0) {                  // Gaussian decoder: [W2|W6]' interleaved
    const float* W6 = a.params + a.oW6;
    for (int i = t32; i < H * D; i += n32) {
      const int r = i / D, c = i - r * D;
      put_pair(w2h, w2l, (size_t)r * a.ldd + 2 * c, __ldcg(W2 + i));
      put_pair(w2h, w2l, (size_t)r * a.ldd + 2 * c + 1, __ldcg(W6 + i));
    }
  } else {
    mirror(W2, w2h, w2l, H, D, a.ldd);
  }
  mirror(W1, w1h, w1l, Z, H, a.ldh);
  for (int i = t32; i < H * Z; i += n32) {      // W4[k, j], W5[k, j]
    const int k = i / Z, j = i - k * Z;
    const float v4 = __ldcg(W4 + i), v5 = __ldcg(W5 + i);
    a.w45t[(size_t)j * H + k] = v4;
    a.w45t[(size_t)(Z + j) * H + k] = v5;
    put_pair(w45h, w45l, (size_t)j * a.ldh + k, v4);
    put_pair(w45h, w45l, (size_t)(Z + j) * a.ldh + k, v5);
    put_pair(whh, whl, (size_t)k * a.ldq + 2 * j, v4);
    put_pair(whh, whl, (size_t)k * a.ldq + 2 * j + 1, v5);
  }
}

}  // namespace

cudaError_t tc_tail_launch(cudaStream_t st, int64_t* launches, const TcTailArgs& a, int grid, bool adam) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(TAIL_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  ++*launches;
  return adam ? cudaLaunchKernelEx(&cfg, tc_tail_kernel<true>, a) : cudaLaunchKernelEx(&cfg, tc_tail_kernel<false>, a);
}

// the grid must be co-resident (grid barriers): as many CTAs per SM as the kernel's registers allow
int tc_tail_grid(int n_sm, bool adam) {
  static int per_sm_of[2] = {0, 0};
  int& per_sm = per_sm_of[adam ? 1 : 0];
  if (per_sm == 0) {
    const cudaError_t oe = adam ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tc_tail_kernel<true>, TAIL_THREADS, 0)
                               : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tc_tail_kernel<false>, TAIL_THREADS, 0);
    if (oe != cudaSuccess || per_sm < 1) per_sm = 1;
    if (per_sm > 6) per_sm = 6;
  }
  return per_sm * n_sm;
}
