// Small fused fp32 kernels of the AEVB step: latent heads + reparameterisation + KL, gradient
// assembly at the latent layer, bound reduction, Adagrad over the flat buffer, full-VB pieces,
// importance-sampling reductions.
#include <cfloat>

#include "adam.cuh"
#include "launchers.h"
#include "philox.cuh"

namespace {

constexpr int ENC2_ROWS = 4;      // rows per block
constexpr int ENC2_THREADS = 128;

__device__ __forceinline__ float eps_at(const EpsSource& s, int64_t flat_injected, int64_t row, int j, int Z,
                                        uint32_t sample) {
  if (s.injected) return s.injected[flat_injected];
  return philox_normal1(s.seed, s.stream, s.step, sample, (uint64_t)((s.row_offset + row) * Z + j));
}

// One block: ENC2_ROWS rows.  Thread per (row, j): two dot products over H sharing the h loads
// (VAEB.py:248-249), then the reparameterisation for every sample (VAEB.py:41-47) and the row
// terms (VAEB.py:343 / :322-325).
__global__ void __launch_bounds__(ENC2_THREADS)
enc2_kernel(const float* __restrict__ h_e, int rows, int H, const float* __restrict__ W4,
            const float* __restrict__ b4, const float* __restrict__ W5, const float* __restrict__ b5, int Z, int L,
            int la, EpsSource src, float* __restrict__ mu, float* __restrict__ ls, float* __restrict__ eps,
            float* __restrict__ z, float* __restrict__ row_aux) {
  extern __shared__ float sm[];
  float* sh = sm;                       // [ENC2_ROWS][H]
  float* st = sm + ENC2_ROWS * H;       // [ENC2_ROWS][Z]
  const int m0 = blockIdx.x * ENC2_ROWS;
  for (int i = threadIdx.x; i < ENC2_ROWS * H; i += blockDim.x) {
    const int r = i / H, k = i % H;
    sh[i] = (m0 + r < rows) ? h_e[(size_t)(m0 + r) * H + k] : 0.f;
  }
  __syncthreads();
  for (int o = threadIdx.x; o < ENC2_ROWS * Z; o += blockDim.x) {
    const int r = o / Z, j = o % Z, m = m0 + r;
    float term = 0.f;
    if (m < rows) {
      float am = 0.f, al = 0.f;
      const float* hr = sh + r * H;
#pragma unroll 4
      for (int k = 0; k < H; ++k) {
        const float hv = hr[k];
        am = fmaf(hv, W4[(size_t)k * Z + j], am);
        al = fmaf(hv, W5[(size_t)k * Z + j], al);
      }
      am += b4[j];
      al += b5[j];
      mu[(size_t)m * Z + j] = am;
      ls[(size_t)m * Z + j] = al;
      const float sd = expf(0.5f * al);
      if (!la) term = 0.5f * (1.0f + al - am * am - expf(al));
      float la_acc = 0.f;
      for (int l = 0; l < L; ++l) {
        const int64_t o2 = ((int64_t)l * rows + m) * Z + j;
        const float e = eps_at(src, o2, m, j, Z, (uint32_t)l);
        const float zv = am + sd * e;
        eps[o2] = e;
        z[o2] = zv;
        la_acc += -0.5f * zv * zv + 0.5f * al + 0.5f * e * e;
      }
      if (la && L > 0) term = la_acc / (float)L;
    }
    st[o] = term;
  }
  __syncthreads();
  if (row_aux && threadIdx.x < ENC2_ROWS && m0 + threadIdx.x < rows) {
    float s = 0.f;
    for (int j = 0; j < Z; ++j) s += st[threadIdx.x * Z + j];
    row_aux[m0 + threadIdx.x] = s;
  }
}

// thread per importance-sampling row r = i*L + l
__global__ void is_sample_kernel(const float* __restrict__ mu, const float* __restrict__ ls, int n, int L, int Z,
                                 EpsSource src, float* __restrict__ z, float* __restrict__ aux) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= (int64_t)n * L) return;
  const int i = (int)(r / L), l = (int)(r % L);
  float a = 0.f;
  for (int j0 = 0; j0 < Z; j0 += 4) {
    float nrm[4];
    const uint64_t e0 = (uint64_t)((src.row_offset + i) * Z + j0);
    const bool aligned = !src.injected && (e0 & 3) == 0;
    if (aligned) philox_normal4(src.seed, src.stream, src.step, (uint32_t)l, e0 >> 2, nrm);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = j0 + q;
      if (j >= Z) break;
      float e;
      if (src.injected) e = src.injected[r * Z + j];
      else if (aligned) e = nrm[q];
      else e = philox_normal1(src.seed, src.stream, src.step, (uint32_t)l, e0 + q);
      const float lsv = ls[(size_t)i * Z + j];
      const float zv = mu[(size_t)i * Z + j] + expf(0.5f * lsv) * e;
      z[r * Z + j] = zv;
      a += -0.5f * zv * zv + 0.5f * lsv + 0.5f * e * e;
    }
  }
  aux[r] = a;
}

__global__ void recon_sample_kernel(const float* __restrict__ mu, const float* __restrict__ ls, int rows, int Z,
                                    EpsSource src, int sample, int n_rows_total, float* __restrict__ z) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * Z) return;
  const int m = (int)(i / Z), j = (int)(i % Z);
  const float e = eps_at(src, ((int64_t)sample * n_rows_total + m) * Z + j, m, j, Z, (uint32_t)sample);
  z[i] = mu[i] + expf(0.5f * ls[i]) * e;
}

// dz[L,rows,Z] -> dmu, dls.  LB: dmu = sum dz - w mu, dls = sum dz*.5*sd*eps + w*.5*(1-e^ls).
// LA: dz -= (w/L) z first, dls += w*.5 (from -log q); the (z-mu)^2/e^ls term has no net gradient.
__global__ void dprep_kernel(const float* __restrict__ dz, const float* __restrict__ z, const float* __restrict__ eps,
                             const float* __restrict__ mu, const float* __restrict__ ls, int rows, int Z, int L,
                             int la, float w, float* __restrict__ dmu, float* __restrict__ dls) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = (int64_t)rows * Z;
  if (i >= n) return;
  const float lsv = ls[i], muv = mu[i];
  const float sd = expf(0.5f * lsv);
  const float s = w / (float)L;
  float dm = 0.f, dl = 0.f;
  for (int l = 0; l < L; ++l) {
    float d = dz[(int64_t)l * n + i];
    if (la) d -= s * z[(int64_t)l * n + i];
    dm += d;
    dl += d * (0.5f * sd * eps[(int64_t)l * n + i]);
  }
  if (la) {
    dl += w * 0.5f;
  } else {
    dm -= w * muv;
    dl += w * 0.5f * (1.0f - expf(lsv));
  }
  dmu[i] = dm;
  dls[i] = dl;
}

// deterministic block sum (fixed tree), result valid in thread 0
__device__ float block_sum_1024(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float t = 0.f;
  if (wid == 0) {
    t = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
  }
  __syncthreads();
  return t;
}

__global__ void __launch_bounds__(1024)
finalize_kernel(const float* __restrict__ partial, int n_tiles, const float* __restrict__ row_aux, int rows, int L,
                float* __restrict__ per_row, float* __restrict__ base_out, float mult,
                const float* __restrict__ tprior, int n_tprior, float div, float* __restrict__ scalar_out,
                float* __restrict__ loglik, float* __restrict__ aux) {
  __shared__ float red[32];
  float acc = 0.f;
  const float invL = 1.0f / (float)L;
  for (int m = threadIdx.x; m < rows; m += blockDim.x) {
    float s = 0.f;
    for (int l = 0; l < L; ++l) {
      const float* p = partial + ((size_t)l * rows + m) * n_tiles;
      float t = 0.f;
      for (int q = 0; q < n_tiles; ++q) t += p[q];
      s += t;
    }
    const float v = s * invL + row_aux[m];
    per_row[m] = v;
    if (loglik) { loglik[m] = __fmul_rn(s, invL); aux[m] = row_aux[m]; }
    acc += v;
  }
  const float base = block_sum_1024(acc, red);
  float tp = 0.f;
  if (tprior) {
    float t = 0.f;
    for (int i = threadIdx.x; i < n_tprior; i += blockDim.x) t += tprior[i];
    tp = block_sum_1024(t, red);
  }
  if (threadIdx.x == 0) {
    *base_out = base;
    if (scalar_out) *scalar_out = (mult * base + tp) / div;
  }
}

__global__ void __launch_bounds__(256)
row_partials_sum_kernel(const float* __restrict__ part, int n_part, int rows, float* __restrict__ out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= rows) return;
  float t = 0.f;
  for (int q = 0; q < n_part; ++q) t += part[(size_t)m * n_part + q];
  out[m] = t;
}

// large row counts: per-row bounds by all SMs, then one block totals them in a fixed order -- with a ticket counter
// and a buffer for the per-block sums the LAST block to finish does it (one launch), else finalize_total_kernel
__global__ void __launch_bounds__(256)
finalize_rows_kernel(const float* __restrict__ partial, int n_tiles, const float* __restrict__ row_aux, int rows, int L,
                     float* __restrict__ per_row, unsigned int* __restrict__ counter, float* __restrict__ block_part,
                     float* __restrict__ base_out, float mult, const float* __restrict__ tprior, int n_tprior, float div,
                     float* __restrict__ scalar_out, float* __restrict__ loglik, float* __restrict__ aux) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  if (m < rows) {
    float s = 0.f;
    for (int l = 0; l < L; ++l) {
      const float* p = partial + ((size_t)l * rows + m) * n_tiles;
      float t = 0.f;
      for (int q = 0; q < n_tiles; ++q) t += p[q];
      s += t;
    }
    v = s * (1.0f / (float)L) + row_aux[m];
    per_row[m] = v;
    if (loglik) { loglik[m] = __fmul_rn(s, 1.0f / (float)L); aux[m] = row_aux[m]; }
  }
  if (!counter) return;
  __shared__ unsigned int is_last;
  __shared__ float red[32];
  const float bsum = block_sum_1024(v, red);
  if (threadIdx.x == 0) {
    block_part[blockIdx.x] = bsum;
    __threadfence();
    is_last = (atomicAdd(counter, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  float acc = 0.f;
  for (int r = threadIdx.x; r < (int)gridDim.x; r += blockDim.x) acc += __ldcg(block_part + r);
  const float base = block_sum_1024(acc, red);
  float tp = 0.f;
  if (tprior) {
    float t = 0.f;
    for (int i = threadIdx.x; i < n_tprior; i += blockDim.x) t += tprior[i];
    tp = block_sum_1024(t, red);
  }
  if (threadIdx.x == 0) {
    *base_out = base;
    if (scalar_out) *scalar_out = (mult * base + tp) / div;
    *counter = 0u;
  }
}
__global__ void __launch_bounds__(1024)
finalize_total_kernel(const float* __restrict__ per_row, int rows, float* __restrict__ base_out, float mult,
                      const float* __restrict__ tprior, int n_tprior, float div, float* __restrict__ scalar_out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int m = threadIdx.x; m < rows; m += blockDim.x) acc += per_row[m];
  const float base = block_sum_1024(acc, red);
  float tp = 0.f;
  if (tprior) {
    float t = 0.f;
    for (int i = threadIdx.x; i < n_tprior; i += blockDim.x) t += tprior[i];
    tp = block_sum_1024(t, red);
  }
  if (threadIdx.x == 0) {
    *base_out = base;
    if (scalar_out) *scalar_out = (mult * base + tp) / div;
  }
}

__global__ void is_rowsum_kernel(const float* __restrict__ partial, int n_tiles, const float* __restrict__ aux,
                                 int64_t rows, float* __restrict__ logw) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* p = partial + (size_t)r * n_tiles;
  float t = 0.f;
  for (int q = 0; q < n_tiles; ++q) t += p[q];
  logw[r] = t + aux[r];
}

// warp per point: logsumexp over L samples
__global__ void is_logsumexp_kernel(const float* __restrict__ logw, int n, int L, float* __restrict__ logp) {
  const int i = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float* w = logw + (size_t)i * L;
  float mx = -FLT_MAX;
  for (int l = lane; l < L; l += 32) mx = fmaxf(mx, w[l]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 0.f;
  for (int l = lane; l < L; l += 32) s += expf(w[l] - mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) logp[i] = mx + logf(s) - logf((float)L);
}

__global__ void add_prior_kernel(float4* __restrict__ g, const float4* __restrict__ p, int64_t n4, float prior,
                                 const float* __restrict__ base, float mult, float div,
                                 float* __restrict__ scalar_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && scalar_out) *scalar_out = (mult * *base) / div;
  if (i >= n4) return;
  float4 gv = g[i];
  const float4 pv = p[i];
  gv.x -= prior * pv.x; gv.y -= prior * pv.y; gv.z -= prior * pv.z; gv.w -= prior * pv.w;
  g[i] = gv;
}

__device__ __forceinline__ void adagrad1(float& p, float& a, float g, float lr, float eps, float prior, float p2) {
  g -= prior * p;                                  // VAEB.py:389-390
  a = a + g * g;                                   // VAEB.py:439
  float np_ = p + lr * g / (sqrtf(a) + eps);       // VAEB.py:441
  if (p2 != 0.f) np_ -= p2 * p * p;                // VAEBfullbayes.py:183-184
  p = np_;
}

// One vectorised, coalesced pass over the flat parameter buffer: 20 B/parameter (read p, acc, g; write p, acc).
// One float4 per thread; g is read once (ld.global.cs: it is dead after this kernel); p and acc are rewritten in
// place.  More loads per thread, streaming hints on p and acc, a persistent grid-stride form and a cp.async.bulk
// shared-memory pipeline all measured slower on B200 (profiles/r1_adagrad_hbm.txt).
__global__ void __launch_bounds__(256)
adagrad_kernel(float4* __restrict__ p, float4* __restrict__ acc, const float4* __restrict__ g, int64_t n4, float lr,
               float eps, float prior, float p2, const float* __restrict__ base, float mult, float div,
               float* __restrict__ scalar_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && scalar_out) *scalar_out = (mult * *base) / div;
  if (i >= n4) return;
  float4 pv = p[i], av = acc[i];
  const float4 gv = __ldcs(g + i);
  adagrad1(pv.x, av.x, gv.x, lr, eps, prior, p2);
  adagrad1(pv.y, av.y, gv.y, lr, eps, prior, p2);
  adagrad1(pv.z, av.z, gv.z, lr, eps, prior, p2);
  adagrad1(pv.w, av.w, gv.w, lr, eps, prior, p2);
  p[i] = pv; acc[i] = av;
}

// getAdaDeltaUpdates, VAEB.py:449-469 (g already carries the prior: VAEB.py:389-390), 28 B/parameter
__device__ __forceinline__ void adadelta1(float& p, float& gac, float& dxac, float g, float rho, float eps, float prior) {
  g -= prior * p;
  gac = rho * gac + (1.0f - rho) * g * g;
  const float dx = sqrtf(dxac + eps) * g / sqrtf(gac + eps);
  p += dx;
  dxac = rho * dxac + (1.0f - rho) * dx * dx;
}
__global__ void __launch_bounds__(256)
adadelta_kernel(float4* __restrict__ p, float4* __restrict__ gac, float4* __restrict__ dxac, const float4* __restrict__ g,
                int64_t n4, float rho, float eps, float prior, const float* __restrict__ base, float mult, float div,
                float* __restrict__ scalar_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && scalar_out) *scalar_out = (mult * *base) / div;
  if (i >= n4) return;
  float4 pv = p[i], av = gac[i], dv = dxac[i];
  const float4 gv = g[i];
  adadelta1(pv.x, av.x, dv.x, gv.x, rho, eps, prior);
  adadelta1(pv.y, av.y, dv.y, gv.y, rho, eps, prior);
  adadelta1(pv.z, av.z, dv.z, gv.z, rho, eps, prior);
  adadelta1(pv.w, av.w, dv.w, gv.w, rho, eps, prior);
  p[i] = pv; gac[i] = av; dxac[i] = dv;
}

// Adam (adam.cuh) over the flat buffer, 28 B/parameter (read p, m, v, g; write p, m, v)
__global__ void __launch_bounds__(256)
adam_kernel(float4* __restrict__ p, float4* __restrict__ m, float4* __restrict__ v, const float4* __restrict__ g,
            int64_t n4, float alpha_t, float s2_t, float b1, float b2, float eps, float prior,
            const float* __restrict__ base, float mult, float div, float* __restrict__ scalar_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && scalar_out) *scalar_out = (mult * *base) / div;
  if (i >= n4) return;
  float4 pv = p[i], mv = m[i], vv = v[i];
  const float4 gv = g[i];
  adam1(pv.x, mv.x, vv.x, gv.x, alpha_t, s2_t, b1, b2, eps, prior);
  adam1(pv.y, mv.y, vv.y, gv.y, alpha_t, s2_t, b1, b2, eps, prior);
  adam1(pv.z, mv.z, vv.z, gv.z, alpha_t, s2_t, b1, b2, eps, prior);
  adam1(pv.w, mv.w, vv.w, gv.w, alpha_t, s2_t, b1, b2, eps, prior);
  p[i] = pv; m[i] = mv; v[i] = vv;
}

__global__ void __launch_bounds__(256)
theta_prior_kernel(const float* __restrict__ vmu, const float* __restrict__ vsig, int64_t n,
                   float* __restrict__ partials) {
  __shared__ float red[32];
  float t = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float m = vmu[i], s = vsig[i];
    t += 0.5f * (1.0f + logf(s * s) - m * m - s * s);   // VAEB.py:363
  }
  const float b = block_sum_1024(t, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = b;
}

__global__ void sample_theta_kernel(const float* __restrict__ vmu, const float* __restrict__ vsig,
                                    const float* __restrict__ zeta_in, uint64_t seed, uint32_t step, int64_t n,
                                    float* __restrict__ theta, float* __restrict__ zeta_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float zt = zeta_in ? zeta_in[i] : philox_normal1(seed, VAEB_STREAM_ZETA, step, 0u, (uint64_t)i);
  zeta_out[i] = zt;
  theta[i] = vmu[i] + fabsf(vsig[i]) * zt;              // VAEB.py:129: normal*sqrt(sigma^2)+mu
}

__global__ void fvb_adagrad_kernel(float* __restrict__ vmu, float* __restrict__ vsig, float* __restrict__ ada_mu,
                                   float* __restrict__ ada_sig, const float* __restrict__ gtheta,
                                   const float* __restrict__ zeta, int sampled, int64_t n, float lr, float eps,
                                   float prior, float* __restrict__ gmu, float* __restrict__ gsig, int apply) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float m = vmu[i], s = vsig[i];
  // d/dmu [thetaPrior - .5*prior*mu^2] = -mu - prior*mu ; d/dsigma = 1/s - s - prior*s
  float gm = -m - prior * m;
  float gs = 1.0f / s - s - prior * s;
  if (sampled) {
    const float gt = gtheta[i];
    const float sg = (s > 0.f) ? 1.f : ((s < 0.f) ? -1.f : 0.f);
    gm += gt;
    gs += gt * zeta[i] * sg;
  }
  gmu[i] = gm;
  gsig[i] = gs;
  if (!apply) return;
  float am = ada_mu[i] + gm * gm, as = ada_sig[i] + gs * gs;
  ada_mu[i] = am;
  ada_sig[i] = as;
  vmu[i] = m + lr * gm / (sqrtf(am) + eps);
  vsig[i] = s + lr * gs / (sqrtf(as) + eps);
}

__global__ void philox_fill_kernel(uint64_t seed, uint32_t stream, uint32_t step, uint32_t sample, int64_t first,
                                   int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = philox_normal1(seed, stream, step, sample, (uint64_t)(first + i));
}

// x[i, d] ~ p(x|z) of decoder outputs mean / lv [rows, D]; noise of element (row_offset + i) * D + d of
// (VAEB_STREAM_SAMPLE, step, sample 1).  Bernoulli: x = 1 if u < mean else 0.  Gaussian: x = mean + exp(lv / 2) * eps,
// the likelihood's own variance exp(lv) (VAEB.py:302-313).
__global__ void __launch_bounds__(256)
sample_x_kernel(const float* __restrict__ mean, const float* __restrict__ lv, int64_t n, int D, uint64_t seed,
                uint32_t step, int64_t row_offset, float* __restrict__ x) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t e = (uint64_t)(row_offset * D + i);
  if (lv)
    x[i] = mean[i] + expf(0.5f * lv[i]) * philox_normal_only(seed, VAEB_STREAM_SAMPLE, step, 1u, e);
  else
    x[i] = philox_uniform1(seed, VAEB_STREAM_SAMPLE, step, 1u, e) < mean[i] ? 1.0f : 0.0f;
}

// out[i, :] = src[idx[i], :]   (ae.py:83 `givens = { X : Xtr[idx] }`: minibatches are gathered, not sliced)
__global__ void __launch_bounds__(256)
gather_rows_kernel(const float* __restrict__ src, const int* __restrict__ idx, int n, int D, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * D) return;
  const int r = (int)(i / D), c = (int)(i - (int64_t)r * D);
  out[i] = src[(size_t)idx[r] * D + c];
}
__global__ void __launch_bounds__(256)
axpy_kernel(float* __restrict__ y, const float* __restrict__ x, float a, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = fmaf(a, x[i], y[i]);
}

inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace

#define LAUNCHED() (++*launches, cudaGetLastError())

cudaError_t launch_enc2(cudaStream_t st, int64_t* launches, const float* h_e, int rows, int H, const float* W4,
                        const float* b4, const float* W5, const float* b5, int Z, int L, int la, EpsSource src,
                        float* mu, float* ls, float* eps, float* z, float* row_aux) {
  const size_t smem = (size_t)ENC2_ROWS * (H + Z) * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(enc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  enc2_kernel<<<(rows + ENC2_ROWS - 1) / ENC2_ROWS, ENC2_THREADS, smem, st>>>(h_e, rows, H, W4, b4, W5, b5, Z, L, la,
                                                                               src, mu, ls, eps, z, row_aux);
  return LAUNCHED();
}

cudaError_t launch_is_sample(cudaStream_t st, int64_t* launches, const float* mu, const float* ls, int n, int L,
                             int Z, EpsSource src, float* z, float* aux) {
  is_sample_kernel<<<blocks_for((int64_t)n * L, 256), 256, 0, st>>>(mu, ls, n, L, Z, src, z, aux);
  return LAUNCHED();
}

cudaError_t launch_recon_sample(cudaStream_t st, int64_t* launches, const float* mu, const float* ls, int rows,
                                int Z, EpsSource src, int sample, int n_rows_total, float* z) {
  recon_sample_kernel<<<blocks_for((int64_t)rows * Z, 256), 256, 0, st>>>(mu, ls, rows, Z, src, sample,
                                                                          n_rows_total, z);
  return LAUNCHED();
}

cudaError_t launch_dprep(cudaStream_t st, int64_t* launches, const float* dz, const float* z, const float* eps,
                         const float* mu, const float* ls, int rows, int Z, int L, int la, float w, float* dmu,
                         float* dls) {
  dprep_kernel<<<blocks_for((int64_t)rows * Z, 256), 256, 0, st>>>(dz, z, eps, mu, ls, rows, Z, L, la, w, dmu, dls);
  return LAUNCHED();
}

cudaError_t launch_finalize(cudaStream_t st, int64_t* launches, const float* partial, int n_tiles,
                            const float* row_aux, int rows, int L, float* per_row, float* base_out, float mult,
                            const float* tprior, int n_tprior, float div, float* scalar_out, unsigned int* counter,
                            float* block_part, float* loglik, float* aux) {
  if (rows >= 2048) {
    if (!block_part) counter = nullptr;
    finalize_rows_kernel<<<blocks_for(rows, 256), 256, 0, st>>>(partial, n_tiles, row_aux, rows, L, per_row, counter,
                                                                block_part, base_out, mult, tprior, n_tprior, div,
                                                                scalar_out, loglik, aux);
    if (counter) return LAUNCHED();
    ++*launches;
    finalize_total_kernel<<<1, 1024, 0, st>>>(per_row, rows, base_out, mult, tprior, n_tprior, div, scalar_out);
    return LAUNCHED();
  }
  finalize_kernel<<<1, 1024, 0, st>>>(partial, n_tiles, row_aux, rows, L, per_row, base_out, mult, tprior, n_tprior,
                                      div, scalar_out, loglik, aux);
  return LAUNCHED();
}

cudaError_t launch_sample_x(cudaStream_t st, int64_t* launches, const float* mean, const float* lv, int rows, int D,
                            uint64_t seed, uint32_t step, int64_t row_offset, float* x) {
  const int64_t n = (int64_t)rows * D;
  sample_x_kernel<<<blocks_for(n, 256), 256, 0, st>>>(mean, lv, n, D, seed, step, row_offset, x);
  return LAUNCHED();
}

cudaError_t launch_is_reduce(cudaStream_t st, int64_t* launches, const float* partial, int n_tiles, const float* aux,
                             int n, int L, float* logw, float* logp) {
  const int64_t rows = (int64_t)n * L;
  is_rowsum_kernel<<<blocks_for(rows, 256), 256, 0, st>>>(partial, n_tiles, aux, rows, logw);
  ++*launches;
  is_logsumexp_kernel<<<blocks_for((int64_t)n * 32, 256), 256, 0, st>>>(logw, n, L, logp);
  return LAUNCHED();
}

cudaError_t launch_add_prior(cudaStream_t st, int64_t* launches, float* g, const float* p, int64_t n4, float prior,
                             const float* base, float mult, float div, float* scalar_out) {
  add_prior_kernel<<<blocks_for(n4, 256), 256, 0, st>>>((float4*)g, (const float4*)p, n4, prior, base, mult, div,
                                                        scalar_out);
  return LAUNCHED();
}

cudaError_t launch_row_partials_sum(cudaStream_t st, int64_t* launches, const float* part, int n_part, int rows,
                                    float* out) {
  row_partials_sum_kernel<<<blocks_for(rows, 256), 256, 0, st>>>(part, n_part, rows, out);
  return LAUNCHED();
}

cudaError_t launch_gather_rows(cudaStream_t st, int64_t* launches, const float* src, const int* idx, int n, int D,
                               float* out) {
  gather_rows_kernel<<<blocks_for((int64_t)n * D, 256), 256, 0, st>>>(src, idx, n, D, out);
  return LAUNCHED();
}
cudaError_t launch_axpy(cudaStream_t st, int64_t* launches, float* y, const float* x, float a, int64_t n) {
  axpy_kernel<<<blocks_for(n, 256), 256, 0, st>>>(y, x, a, n);
  return LAUNCHED();
}

cudaError_t launch_adadelta(cudaStream_t st, int64_t* launches, float* p, float* gac, float* dxac, const float* g,
                            int64_t n4, float rho, float eps, float prior, const float* base, float mult, float div,
                            float* scalar_out) {
  adadelta_kernel<<<blocks_for(n4, 256), 256, 0, st>>>((float4*)p, (float4*)gac, (float4*)dxac, (const float4*)g, n4, rho,
                                                       eps, prior, base, mult, div, scalar_out);
  return LAUNCHED();
}

cudaError_t launch_adam(cudaStream_t st, int64_t* launches, float* p, float* m, float* v, const float* g, int64_t n4,
                        float alpha_t, float s2_t, float b1, float b2, float eps, float prior, const float* base,
                        float mult, float div, float* scalar_out) {
  adam_kernel<<<blocks_for(n4, 256), 256, 0, st>>>((float4*)p, (float4*)m, (float4*)v, (const float4*)g, n4, alpha_t,
                                                   s2_t, b1, b2, eps, prior, base, mult, div, scalar_out);
  return LAUNCHED();
}

cudaError_t launch_adagrad(cudaStream_t st, int64_t* launches, float* p, float* acc, const float* g, int64_t n4,
                           float lr, float eps, float prior, float p2, const float* base, float mult, float div,
                           float* scalar_out) {
  adagrad_kernel<<<blocks_for(n4, 256), 256, 0, st>>>((float4*)p, (float4*)acc, (const float4*)g, n4, lr, eps, prior, p2,
                                                      base, mult, div, scalar_out);
  return LAUNCHED();
}

cudaError_t launch_theta_prior(cudaStream_t st, int64_t* launches, const float* vmu, const float* vsig, int64_t n,
                               float* partials) {
  theta_prior_kernel<<<VAEB_TP_BLOCKS, 256, 0, st>>>(vmu, vsig, n, partials);
  return LAUNCHED();
}

cudaError_t launch_sample_theta(cudaStream_t st, int64_t* launches, const float* vmu, const float* vsig,
                                const float* zeta_in, uint64_t seed, uint32_t step, int64_t n, float* theta,
                                float* zeta_out) {
  sample_theta_kernel<<<blocks_for(n, 256), 256, 0, st>>>(vmu, vsig, zeta_in, seed, step, n, theta, zeta_out);
  return LAUNCHED();
}

cudaError_t launch_fvb_adagrad(cudaStream_t st, int64_t* launches, float* vmu, float* vsig, float* ada_mu,
                               float* ada_sig, const float* gtheta, const float* zeta, int sampled, int64_t n,
                               float lr, float eps, float prior, float* gmu, float* gsig, int apply) {
  fvb_adagrad_kernel<<<blocks_for(n, 256), 256, 0, st>>>(vmu, vsig, ada_mu, ada_sig, gtheta, zeta, sampled, n, lr, eps,
                                                         prior, gmu, gsig, apply);
  return LAUNCHED();
}

cudaError_t launch_philox_fill(cudaStream_t st, int64_t* launches, uint64_t seed, uint32_t stream, uint32_t step,
                               uint32_t sample, int64_t first, int64_t n, float* out) {
  philox_fill_kernel<<<blocks_for(n, 256), 256, 0, st>>>(seed, stream, step, sample, first, n, out);
  return LAUNCHED();
}

namespace {
// byte-valued inputs (MNIST / Frey pixels = k / 256): out = (float)in * scale, one IEEE product per element -- the same
// bits as np.float32(in) * np.float32(scale) on the host.  16 bytes in, 64 bytes out per thread.
__global__ void __launch_bounds__(256)
expand_u8_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, int64_t n, float scale) {
  const int64_t n16 = n >> 4;
  const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out)) & 15u) == 0;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  if (aligned) {
    for (int64_t i = tid; i < n16; i += nth) {
      const uint4 v = __ldcs(reinterpret_cast<const uint4*>(in) + i);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
      float4* o = reinterpret_cast<float4*>(out) + 4 * i;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        o[k] = make_float4(__fmul_rn((float)(w[k] & 0xffu), scale), __fmul_rn((float)((w[k] >> 8) & 0xffu), scale),
                           __fmul_rn((float)((w[k] >> 16) & 0xffu), scale), __fmul_rn((float)(w[k] >> 24), scale));
    }
    for (int64_t i = (n16 << 4) + tid; i < n; i += nth) out[i] = __fmul_rn((float)in[i], scale);
  } else {
    for (int64_t i = tid; i < n; i += nth) out[i] = __fmul_rn((float)in[i], scale);
  }
}
}  // namespace

cudaError_t launch_expand_u8(cudaStream_t st, const uint8_t* in, float* out, int64_t n, float scale) {
  const int64_t work = (n + 15) / 16;
  int64_t blocks = (work + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  expand_u8_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, out, n, scale);
  return cudaGetLastError();
}
