// The fused AEVB update: one persistent cooperative kernel for n whole steps (see fused_step.cuh).
//
// Work decomposition.  Every dense layer of the step is a "job": a grid of TM x TN output tiles
// (TM = 8*TMT, TN = 4*TNT, per-thread micro tile TMT x TNT on a fixed 8x4 lane grid).  A tile is
// owned by `ks` warps of ONE CTA, each contracting its own slice of the k index from global memory
// (L2) through a private shared-memory stage; the ks partial tiles meet in shared memory and a
// fused epilogue (tanh, reparameterisation, log-likelihood + deltas, tanh', Adagrad) writes the
// result.  At M = 100 the outputs are skinny (100 x 500 / 100 x 784), so the jobs are cut into
// ~148 CTA items of full contraction depth: no cross-CTA partial sums, results are deterministic.
//
// Dependencies between jobs are grid barriers (monotonic 64-bit counter, release/acquire at gpu
// scope).  Data produced by other CTAs is always read with ld.global.cg (L2), never through L1.
//
// Parameters are double buffered: phase k reads theta from params[cur] while the weight-gradient
// epilogues of the same step write Adagrad's theta' into params[cur^1] (the backward of a layer
// still needs the old W while its gradient is being applied).  ADA is updated in place.
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "fused_step.cuh"
#include "philox.cuh"

namespace fs {

enum { A_MK = 0, A_KM = 1 };          // A(m,k) = A[m*lda + k]  |  A[k*lda + m]
enum { B_KN = 0, B_NK = 1 };          // B(k,n) = B[k*ldb + n]  |  B[n*ldb + k]
enum { PLAIN = 0, DUALK = 1, DUALN = 2 };
// DUALK: k <  K0 -> (A0, B0), k >= K0 -> (A1, B1) at k - K0   (sum of two products)
// DUALN: tile columns [0, TN/2) come from B0, [TN/2, TN) from B1 at the same n (two heads)

struct Gemm {
  const float* A0; const float* A1; int lda;
  const float* B0; const float* B1; int ldb;
  int M, N, K0, K1;
  int ones_row;                       // A_KM: row index that reads as 1 (bias gradient), else -1
  JobCfg c;
  int avec, bvec;                     // operands may be staged with 16-byte copies
};

__device__ __forceinline__ bool al16(const float* q) { return q == nullptr || ((uintptr_t)q & 15) == 0; }
// 16-byte staging is legal when both sources are aligned, the leading dimension is a multiple of four
// floats and (for a contraction split over two sources) the split point is too
__device__ __forceinline__ Gemm make_gemm(const float* A0, const float* A1, int lda, const float* B0, const float* B1,
                                          int ldb, int M, int N, int K0, int K1, int ones_row, const JobCfg& c) {
  Gemm g{A0, A1, lda, B0, B1, ldb, M, N, K0, K1, ones_row, c, 0, 0};
  const bool ksplit_ok = K1 == 0 || (K0 & 3) == 0;
  g.avec = al16(A0) && al16(A1) && (lda & 3) == 0 && ksplit_ok;
  g.bvec = al16(B0) && al16(B1) && (ldb & 3) == 0 && ksplit_ok;
  return g;
}

__device__ __forceinline__ float softplusf_(float a) { return fmaxf(a, 0.f) + log1pf(expf(-fabsf(a))); }
__device__ __forceinline__ float sigmoidf_(float a) { return 1.0f / (1.0f + expf(-a)); }

// ---------------------------------------------------------------------------------------------
// operand staging: global (L2) -> this warp's shared-memory stage with cp.async (no staging
// registers).  Layouts keep the source's contiguous index contiguous, so 16-byte copies apply
// whenever the leading dimension and offsets are multiples of four floats (avec / bvec):
//   A_KM  sA[kk*(TM+4) + m]      A_MK  sA[m*KSTR + kk]
//   B_KN  sB[kk*TN + c]          B_NK  sB[c*KSTR + kk]
// A chunk covers k in [kc, kc+kv); everything up to kv rounded up to four is zero filled.
// ---------------------------------------------------------------------------------------------
constexpr int KSTR = KC + 4;

__device__ __forceinline__ void cp4(float* dst, const float* src, int bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)),
               "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp16(float* dst, const float* src, int bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)),
               "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int TM, int AL, int MODE>
__device__ __forceinline__ void issue_A(const Gemm& g, float* sA, int m0, int kc, int kv, int lane) {
  const int kvr = (kv + 3) & ~3;
  const int Mreal = g.ones_row >= 0 ? g.ones_row : g.M;     // the ones row is patched in after the copy lands
  if (AL == A_KM) {
    constexpr int TMS = TM + 4;
    if (g.avec) {
      constexpr int PR = TM / 4;                            // 16-byte pieces per k row
      for (int idx = lane; idx < kvr * PR; idx += 32) {
        const int kk = idx / PR, mq = idx - kk * PR;
        const int gm = m0 + 4 * mq;
        const int bytes = kk < kv ? 4 * max(0, min(4, Mreal - gm)) : 0;
        cp16(sA + kk * TMS + 4 * mq, bytes ? g.A0 + (size_t)(kc + kk) * g.lda + gm : g.A0, bytes);
      }
    } else {
      for (int idx = lane; idx < kvr * TM; idx += 32) {
        const int kk = idx / TM, m = idx - kk * TM;
        const int gm = m0 + m;
        const bool ok = kk < kv && gm < Mreal;
        cp4(sA + kk * TMS + m, ok ? g.A0 + (size_t)(kc + kk) * g.lda + gm : g.A0, ok ? 4 : 0);
      }
    }
  } else {
    if (g.avec) {
#pragma unroll
      for (int t = 0; t < TM / 8; ++t) {
        const int idx = lane + 32 * t;
        const int m = idx >> 2, kk = (idx & 3) * 4;
        if (kk < kvr) {
          const int gm = m0 + m;
          int ko = kc + kk;
          const float* src = g.A0;
          if (MODE == DUALK && ko >= g.K0) { src = g.A1; ko -= g.K0; }
          const int bytes = gm < g.M ? 4 * max(0, min(4, kv - kk)) : 0;
          cp16(sA + m * KSTR + kk, bytes ? src + (size_t)gm * g.lda + ko : g.A0, bytes);
        }
      }
    } else {
#pragma unroll
      for (int t = 0; t < TM / 2; ++t) {
        const int idx = lane + 32 * t;
        const int m = idx >> 4, kk = idx & 15;
        if (kk < kvr) {
          const int gm = m0 + m;
          int ko = kc + kk;
          const float* src = g.A0;
          if (MODE == DUALK && ko >= g.K0) { src = g.A1; ko -= g.K0; }
          const bool ok = kk < kv && gm < g.M;
          cp4(sA + m * KSTR + kk, ok ? src + (size_t)gm * g.lda + ko : g.A0, ok ? 4 : 0);
        }
      }
    }
  }
}

template <int TN, int BL, int MODE>
__device__ __forceinline__ void issue_B(const Gemm& g, float* sB, int n0, int kc, int kv, int lane) {
  static_assert(!(BL == B_KN && MODE == DUALK) && !(BL == B_NK && MODE == DUALN), "unsupported operand mode");
  const int kvr = (kv + 3) & ~3;
  if (BL == B_KN) {
    if (g.bvec) {
      constexpr int PR = TN / 4;
      for (int idx = lane; idx < kvr * PR; idx += 32) {
        const int kk = idx / PR, cq = idx - kk * PR;
        int c = 4 * cq;
        const float* src = g.B0;
        if (MODE == DUALN && c >= TN / 2) { src = g.B1; c -= TN / 2; }
        const int gn = n0 + c;
        const int bytes = kk < kv ? 4 * max(0, min(4, g.N - gn)) : 0;
        cp16(sB + kk * TN + 4 * cq, bytes ? src + (size_t)(kc + kk) * g.ldb + gn : g.B0, bytes);
      }
    } else {
      for (int idx = lane; idx < kvr * TN; idx += 32) {
        const int kk = idx / TN, cc = idx - kk * TN;
        int c = cc;
        const float* src = g.B0;
        if (MODE == DUALN && c >= TN / 2) { src = g.B1; c -= TN / 2; }
        const int gn = n0 + c;
        const bool ok = kk < kv && gn < g.N;
        cp4(sB + kk * TN + cc, ok ? src + (size_t)(kc + kk) * g.ldb + gn : g.B0, ok ? 4 : 0);
      }
    }
  } else {
    if (g.bvec) {
#pragma unroll
      for (int t = 0; t < TN / 8; ++t) {
        const int idx = lane + 32 * t;
        const int c = idx >> 2, kk = (idx & 3) * 4;
        if (kk < kvr) {
          const int gn = n0 + c;
          int ko = kc + kk;
          const float* src = g.B0;
          if (MODE == DUALK && ko >= g.K0) { src = g.B1; ko -= g.K0; }
          const int bytes = gn < g.N ? 4 * max(0, min(4, kv - kk)) : 0;
          cp16(sB + c * KSTR + kk, bytes ? src + (size_t)gn * g.ldb + ko : g.B0, bytes);
        }
      }
    } else {
#pragma unroll
      for (int t = 0; t < TN / 2; ++t) {
        const int idx = lane + 32 * t;
        const int c = idx >> 4, kk = idx & 15;
        if (kk < kvr) {
          const int gn = n0 + c;
          int ko = kc + kk;
          const float* src = g.B0;
          if (MODE == DUALK && ko >= g.K0) { src = g.B1; ko -= g.K0; }
          const bool ok = kk < kv && gn < g.N;
          cp4(sB + c * KSTR + kk, ok ? src + (size_t)gn * g.ldb + ko : g.B0, ok ? 4 : 0);
        }
      }
    }
  }
}

// micro-tile entry -> tile row / column for lane (rg, cg).  Chosen per layout so that the fragment
// loads are conflict free: k-major stages read TMT (TNT) consecutive floats, [m][k] / [n][k] stages
// read float4 along k from rows rg + 8i (columns cg + 4j).
template <int TMT, int AL>
__device__ __forceinline__ int row_of(int i, int rg) { return AL == A_KM ? rg * TMT + i : rg + 8 * i; }
template <int TNT, int BL>
__device__ __forceinline__ int col_of(int j, int cg) {
  constexpr int NA4 = TNT / 4;
  if (BL == B_NK) return cg + 4 * j;
  return j < 4 * NA4 ? (j >> 2) * 16 + cg * 4 + (j & 3) : 16 * NA4 + cg * 2 + (j - 4 * NA4);
}

// four k steps of the contraction from one stage
template <int TMT, int TNT, int AL, int BL>
__device__ __forceinline__ void fma_quad(const float* sA, const float* sB, int kk, int rg, int cg,
                                         float (&acc)[TMT][TNT]) {
  constexpr int TM = 8 * TMT, TN = 4 * TNT, TMS = TM + 4;
  constexpr int NA4 = TNT / 4, NB2 = (TNT % 4) / 2;
  float am[AL == A_MK ? TMT : 1][4], bn[BL == B_NK ? TNT : 1][4];
  if (AL == A_MK) {
#pragma unroll
    for (int i = 0; i < TMT; ++i) {
      const float4 t = *reinterpret_cast<const float4*>(sA + (rg + 8 * i) * KSTR + kk);
      am[i][0] = t.x; am[i][1] = t.y; am[i][2] = t.z; am[i][3] = t.w;
    }
  }
  if (BL == B_NK) {
#pragma unroll
    for (int j = 0; j < TNT; ++j) {
      const float4 t = *reinterpret_cast<const float4*>(sB + (cg + 4 * j) * KSTR + kk);
      bn[j][0] = t.x; bn[j][1] = t.y; bn[j][2] = t.z; bn[j][3] = t.w;
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float a[TMT], b[TNT];
    if (AL == A_MK) {
#pragma unroll
      for (int i = 0; i < TMT; ++i) a[i] = am[i][q];
    } else {
#pragma unroll
      for (int i = 0; i < TMT / 2; ++i) {
        const float2 t = *reinterpret_cast<const float2*>(sA + (kk + q) * TMS + rg * TMT + 2 * i);
        a[2 * i] = t.x; a[2 * i + 1] = t.y;
      }
    }
    if (BL == B_NK) {
#pragma unroll
      for (int j = 0; j < TNT; ++j) b[j] = bn[j][q];
    } else {
#pragma unroll
      for (int u = 0; u < NA4; ++u) {
        const float4 t = *reinterpret_cast<const float4*>(sB + (kk + q) * TN + u * 16 + cg * 4);
        b[4 * u] = t.x; b[4 * u + 1] = t.y; b[4 * u + 2] = t.z; b[4 * u + 3] = t.w;
      }
      if (NB2) {
        const float2 t = *reinterpret_cast<const float2*>(sB + (kk + q) * TN + NA4 * 16 + cg * 2);
        b[4 * NA4] = t.x; b[4 * NA4 + 1] = t.y;
      }
    }
#pragma unroll
    for (int i = 0; i < TMT; ++i)
#pragma unroll
      for (int j = 0; j < TNT; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

// elements an epilogue keeps in flight per thread (the sampled full-VB update holds 5 operands per element)
template <class Epi> struct EpiInflight { static constexpr int value = 2; };
template <bool FVB> struct EpiAdagrad;
template <bool FVB> struct EpiAdagrad2;
template <> struct EpiInflight<EpiAdagrad<true>> { static constexpr int value = 1; };
template <> struct EpiInflight<EpiAdagrad2<true>> { static constexpr int value = 1; };

// ---------------------------------------------------------------------------------------------
// one CTA item of a job.  tm_fixed >= 0: the item covers tiles (tm_fixed, item*tpi + tl) -- the
// row-block chains, where one CTA runs two dependent layers for its own rows.
// ---------------------------------------------------------------------------------------------
template <int TMT, int TNT, int AL, int BL, int MODE, class Epi>
__device__ __forceinline__ void run_item(const Gemm& g, int item, const Epi& epi, float* smem, int tm_fixed = -1) {
  static_assert(TMT % 2 == 0 && TNT % 2 == 0, "micro tile");
  constexpr int TM = 8 * TMT, TN = 4 * TNT;
  constexpr int SA = (AL == A_KM) ? KC * (TM + 4) : TM * KSTR;     // floats of one A stage
  constexpr int SB = (BL == B_KN) ? KC * TN : TN * KSTR;
  constexpr int STAGE = SA + SB;
  constexpr int TNE = (MODE == DUALN) ? TN / 2 : TN;      // distinct output columns of a tile
  static_assert(NSTAGE * STAGE <= WBUF && TM * TN <= WBUF, "shared-memory stage too small");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = g.c.ks;
  const int tl = warp / ks, ksi = warp - tl * ks;
  const int tile = item * g.c.tpi + tl;
  int tm, tn;
  bool active = tl < g.c.tpi;
  if (tm_fixed >= 0) { tm = tm_fixed; tn = tile; active = active && tn < g.c.tiles_n; }
  else { tm = tile % g.c.tiles_m; tn = tile / g.c.tiles_m; active = active && tile < g.c.tiles_m * g.c.tiles_n; }
  float* wbuf = smem + warp * WBUF;
  const int m0 = tm * TM, n0 = tn * TNE;
  if (active) {
    const int K = g.K0 + g.K1;
    // k slices start at multiples of four (16-byte copies along k stay aligned)
    const int k0 = min(K, (int)((((long long)K * ksi) / ks + 3) & ~3LL));
    const int k1 = ksi + 1 == ks ? K : min(K, (int)((((long long)K * (ksi + 1)) / ks + 3) & ~3LL));
    const int rg = lane >> 2, cg = lane & 3;
    float acc[TMT][TNT];
#pragma unroll
    for (int i = 0; i < TMT; ++i)
#pragma unroll
      for (int j = 0; j < TNT; ++j) acc[i][j] = 0.f;
    const bool ones_here = AL == A_KM && g.ones_row >= m0 && g.ones_row < m0 + TM;
    // NSTAGE-deep cp.async pipeline: chunks c+1 .. c+NSTAGE-1 are in flight while chunk c is contracted
    const int nch = (k1 - k0 + KC - 1) / KC;
#pragma unroll 1
    for (int c = 0; c < NSTAGE - 1; ++c) {
      if (c < nch) {
        const int kc = k0 + c * KC;
        float* nA = wbuf + c * STAGE;
        issue_A<TM, AL, MODE>(g, nA, m0, kc, min(KC, k1 - kc), lane);
        issue_B<TN, BL, MODE>(g, nA + SA, n0, kc, min(KC, k1 - kc), lane);
      }
      cp_commit();
    }
    int st = 0;
#pragma unroll 1
    for (int c = 0; c < nch; ++c) {
      const int kc = k0 + c * KC;
      const int kv = min(KC, k1 - kc);
      float* sA = wbuf + st * STAGE;
      float* sB = sA + SA;
      {
        const int cn = c + NSTAGE - 1;
        if (cn < nch) {
          const int kcn = k0 + cn * KC;
          int sn = st + NSTAGE - 1; if (sn >= NSTAGE) sn -= NSTAGE;
          float* nA = wbuf + sn * STAGE;
          issue_A<TM, AL, MODE>(g, nA, m0, kcn, min(KC, k1 - kcn), lane);
          issue_B<TN, BL, MODE>(g, nA + SA, n0, kcn, min(KC, k1 - kcn), lane);
        }
        cp_commit();
      }
      cp_wait<NSTAGE - 1>();
      __syncwarp();
      if (ones_here) {                     // bias-gradient row of [act | 1]^T
        if (lane < ((kv + 3) & ~3)) sA[lane * (TM + 4) + (g.ones_row - m0)] = lane < kv ? 1.f : 0.f;
        __syncwarp();
      }
#pragma unroll 1
      for (int kk = 0; kk < kv; kk += 4) fma_quad<TMT, TNT, AL, BL>(sA, sB, kk, rg, cg, acc);
      __syncwarp();
      if (++st == NSTAGE) st = 0;
    }
    cp_wait<0>();
    // this warp's partial tile, row-major [TM][TN], over its own stage
#pragma unroll
    for (int i = 0; i < TMT; ++i)
#pragma unroll
      for (int j = 0; j < TNT; ++j) wbuf[row_of<TMT, AL>(i, rg) * TN + col_of<TNT, BL>(j, cg)] = acc[i][j];
  }
  __syncthreads();
  const int gidx = ksi * 32 + lane, gsize = ks * 32;
  float* gbuf = smem + (tl * ks) * WBUF;
  if (active) {
    constexpr int U = EpiInflight<Epi>::value;   // elements in flight per thread: their global operands are
#pragma unroll 1                           // requested before the partial tiles are summed
    for (int e0 = gidx; e0 < TM * TNE; e0 += gsize * U) {
      typename Epi::Pre pre[U];
      int gm[U], gn[U], so[U];
      bool ok[U], in[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int e = e0 + u * gsize;
        in[u] = e < TM * TNE;
        const int row = e / TNE, c = e - row * TNE;
        so[u] = row * TN + c;
        gm[u] = m0 + row; gn[u] = n0 + c;
        ok[u] = in[u] && gm[u] < g.M && gn[u] < g.N;
        if (ok[u]) pre[u] = epi.pre(gm[u], gn[u]);
      }
      float v0[U], v1[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        v0[u] = 0.f; v1[u] = 0.f;
        if (in[u]) {
          for (int s = 0; s < ks; ++s) {
            v0[u] += gbuf[s * WBUF + so[u]];
            if (MODE == DUALN) v1[u] += gbuf[s * WBUF + so[u] + TN / 2];
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float term = 0.f;
        if (ok[u]) term = epi.elem(gm[u], gn[u], v0[u], v1[u], pre[u]);
        if (Epi::ROWSUM && in[u]) gbuf[so[u]] = term;
      }
    }
  }
  if (Epi::ROWSUM) {
    __syncthreads();
    if (active && gidx < TM && m0 + gidx < g.M) {
      float s = 0.f;
      const int cmax = min(TNE, g.N - n0);
      for (int c = 0; c < cmax; ++c) s += gbuf[gidx * TN + c];
      epi.rowsum(m0 + gidx, tn, s);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// epilogues: pre() requests the global operands of one output element, elem() finishes it
// ---------------------------------------------------------------------------------------------
struct EpiTanh {                      // out = tanh(acc + bias[n])               VAEB.py:246,254
  static constexpr bool ROWSUM = false;
  struct Pre { float b; };
  const float* bias; float* out; int ld;
  __device__ __forceinline__ Pre pre(int, int n) const { return Pre{__ldcg(bias + n)}; }
  __device__ __forceinline__ float elem(int m, int n, float v, float, const Pre& q) const {
    out[(size_t)m * ld + n] = tanhf(v + q.b);
    return 0.f;
  }
  __device__ __forceinline__ void rowsum(int, int, float) const {}
};

struct EpiLatent {                    // VAEB.py:248-249 heads, :41-47 reparameterisation, :343 / :322-325 row terms
  static constexpr bool ROWSUM = true;
  struct Pre { float b4, b5, e; };
  const float* b4; const float* b5; const float* eps_inj;
  uint64_t seed; uint32_t step; int64_t row_offset;
  int Z, la, n_tiles;
  float *mu, *ls, *eps, *z, *aux_part;
  __device__ __forceinline__ Pre pre(int m, int j) const {
    return Pre{__ldcg(b4 + j), __ldcg(b5 + j), eps_inj ? __ldcg(eps_inj + (size_t)m * Z + j) : 0.f};
  }
  __device__ __forceinline__ float elem(int m, int j, float v0, float v1, const Pre& q) const {
    const float am = v0 + q.b4, al = v1 + q.b5;
    const size_t o = (size_t)m * Z + j;
    const float e = eps_inj ? q.e
                            : philox_normal1(seed, VAEB_STREAM_TRAIN, step, 0u, (uint64_t)((row_offset + m) * Z + j));
    const float zv = am + expf(0.5f * al) * e;
    mu[o] = am; ls[o] = al; eps[o] = e; z[o] = zv;
    return la ? (-0.5f * zv * zv + 0.5f * al + 0.5f * e * e) : 0.5f * (1.0f + al - am * am - expf(al));
  }
  __device__ __forceinline__ void rowsum(int m, int tn, float s) const { aux_part[(size_t)m * n_tiles + tn] = s; }
};

struct EpiBernoulli {                 // VAEB.py:263,311: x*a - softplus(a); da = w*(x - sigmoid(a))
  static constexpr bool ROWSUM = true;
  struct Pre { float b, x; };
  const float* b2; const float* x; int D; float scale; float* da; float* partial; int n_tiles;
  __device__ __forceinline__ Pre pre(int m, int n) const { return Pre{__ldcg(b2 + n), __ldcg(x + (size_t)m * D + n)}; }
  __device__ __forceinline__ float elem(int m, int n, float v, float, const Pre& q) const {
    const float a = v + q.b;
    da[(size_t)m * D + n] = scale * (q.x - sigmoidf_(a));
    return q.x * a - softplusf_(a);
  }
  __device__ __forceinline__ void rowsum(int m, int tn, float s) const { partial[(size_t)m * n_tiles + tn] = s; }
};

struct EpiGaussian {                  // VAEB.py:257-258,306-307
  static constexpr bool ROWSUM = true;
  struct Pre { float b2, b6, x; };
  const float* b2; const float* b6; const float* x; int D; float scale; float* da; float* dlv; float* partial;
  int n_tiles;
  __device__ __forceinline__ Pre pre(int m, int n) const {
    return Pre{__ldcg(b2 + n), __ldcg(b6 + n), __ldcg(x + (size_t)m * D + n)};
  }
  __device__ __forceinline__ float elem(int m, int n, float v0, float v1, const Pre& q) const {
    const float a = v0 + q.b2, lv = v1 + q.b6;
    const float mx = sigmoidf_(a);
    const float d = q.x - mx;
    const float r = d * expf(-lv);
    da[(size_t)m * D + n] = scale * r * mx * (1.0f - mx);
    dlv[(size_t)m * D + n] = scale * (-0.5f + 0.5f * d * r);
    return -0.91893853320467274178f - 0.5f * lv - 0.5f * d * r;
  }
  __device__ __forceinline__ void rowsum(int m, int tn, float s) const { partial[(size_t)m * n_tiles + tn] = s; }
};

struct EpiTanhBack {                  // out = acc * (1 - h^2)
  static constexpr bool ROWSUM = false;
  struct Pre { float h; };
  const float* h; float* out; int ld;
  __device__ __forceinline__ Pre pre(int m, int n) const { return Pre{__ldcg(h + (size_t)m * ld + n)}; }
  __device__ __forceinline__ float elem(int m, int n, float v, float, const Pre& q) const {
    out[(size_t)m * ld + n] = v * (1.0f - q.h * q.h);
    return 0.f;
  }
  __device__ __forceinline__ void rowsum(int, int, float) const {}
};

struct EpiDz {                        // dz -> dmu, dls (SURVEY.md 8a backward formulas), L == 1
  static constexpr bool ROWSUM = false;
  struct Pre { float z, eps, mu, ls; };
  const float *z, *eps, *mu, *ls; int Z, la; float w; float *dmu, *dls;
  __device__ __forceinline__ Pre pre(int m, int j) const {
    const size_t o = (size_t)m * Z + j;
    return Pre{__ldcg(z + o), __ldcg(eps + o), __ldcg(mu + o), __ldcg(ls + o)};
  }
  __device__ __forceinline__ float elem(int m, int j, float v, float, const Pre& q) const {
    const size_t o = (size_t)m * Z + j;
    float d = v;
    if (la) d -= w * q.z;
    float a = d, b = d * (0.5f * expf(0.5f * q.ls) * q.eps);
    if (la) {
      b += w * 0.5f;
    } else {
      a -= w * q.mu;
      b += w * 0.5f * (1.0f - expf(q.ls));
    }
    dmu[o] = a; dls[o] = b;
    return 0.f;
  }
  __device__ __forceinline__ void rowsum(int, int, float) const {}
};

struct Hyper { float lr, eps, prior, p2; };

__device__ __forceinline__ void adagrad_apply(float p, float a0, float* Pn, float* ada, size_t o, float g, const Hyper& hy) {
  g -= hy.prior * p;                                    // VAEB.py:389-390
  const float a = a0 + g * g;                           // VAEB.py:439
  float np_ = p + hy.lr * g / (sqrtf(a) + hy.eps);      // VAEB.py:441
  if (hy.p2 != 0.f) np_ -= hy.p2 * p * p;               // VAEBfullbayes.py:183-184
  Pn[o] = np_;
  ada[o] = a;
}

// Full VB with sampled weights: theta = mu + |sigma| zeta, so dL/dmu = g and dL/dsigma = g zeta sign(sigma); the
// prior terms are d/dmu [thetaPrior - .5 prior mu^2] = -mu - prior mu and d/dsigma = 1/s - s - prior s
// (VAEB.py:359-363,391-393); Adagrad (VAEB.py:426-444) on both.
struct Fvb { float* vsig; float* ada_sig; const float* zeta; };

__device__ __forceinline__ void fvb_apply(float m, float am0, float s, float as0, float zt, float* vmu, float* ada_mu,
                                          const Fvb& f, size_t o, float g, const Hyper& hy) {
  const float sg = (s > 0.f) ? 1.f : ((s < 0.f) ? -1.f : 0.f);
  const float gm = g - m - hy.prior * m;
  const float gs = 1.0f / s - s - hy.prior * s + g * zt * sg;
  const float am = am0 + gm * gm, as = as0 + gs * gs;
  ada_mu[o] = am;
  f.ada_sig[o] = as;
  vmu[o] = m + hy.lr * gm / (sqrtf(am) + hy.eps);
  f.vsig[o] = s + hy.lr * gs / (sqrtf(as) + hy.eps);
}

template <bool FVB> struct PreAda { float p, a; };
template <> struct PreAda<true> { float p, a, s, as, zt; };
template <bool FVB> struct PreAda2 { float pa, aa, pb, ab; };
template <> struct PreAda2<true> { float pa, aa, pb, ab, sa, asa, za, sb, asb, zb; };

template <bool FVB>
struct EpiAdagrad {                   // rows < nW: weight [nW, ld]; row == nW: the bias (ones row of A)
  static constexpr bool ROWSUM = false;
  using Pre = PreAda<FVB>;
  const float* P; float* Pn; float* ada; int64_t oW, ob; int nW, ld; Hyper hy; Fvb f;
  __device__ __forceinline__ size_t off(int m, int n) const {
    return m < nW ? (size_t)oW + (size_t)m * ld + n : (size_t)ob + n;
  }
  __device__ __forceinline__ Pre pre(int m, int n) const {
    const size_t o = off(m, n);
    Pre q;
    q.p = __ldcg(P + o); q.a = __ldcg(ada + o);
    if constexpr (FVB) { q.s = __ldcg(f.vsig + o); q.as = __ldcg(f.ada_sig + o); q.zt = __ldcg(f.zeta + o); }
    return q;
  }
  __device__ __forceinline__ float elem(int m, int n, float v, float, const Pre& q) const {
    if constexpr (FVB) fvb_apply(q.p, q.a, q.s, q.as, q.zt, Pn, ada, f, off(m, n), v, hy);
    else adagrad_apply(q.p, q.a, Pn, ada, off(m, n), v, hy);
    return 0.f;
  }
  __device__ __forceinline__ void rowsum(int, int, float) const {}
};

template <bool FVB>
struct EpiAdagrad2 {                  // two heads at once (W4|W5, b4|b5)
  static constexpr bool ROWSUM = false;
  using Pre = PreAda2<FVB>;
  const float* P; float* Pn; float* ada; int64_t oWa, oba, oWb, obb; int nW, ld; Hyper hy; Fvb f;
  __device__ __forceinline__ Pre pre(int m, int n) const {
    const size_t off = m < nW ? (size_t)m * ld + n : (size_t)n;
    const size_t oa = (size_t)(m < nW ? oWa : oba) + off, ob_ = (size_t)(m < nW ? oWb : obb) + off;
    Pre q;
    q.pa = __ldcg(P + oa); q.aa = __ldcg(ada + oa); q.pb = __ldcg(P + ob_); q.ab = __ldcg(ada + ob_);
    if constexpr (FVB) {
      q.sa = __ldcg(f.vsig + oa); q.asa = __ldcg(f.ada_sig + oa); q.za = __ldcg(f.zeta + oa);
      q.sb = __ldcg(f.vsig + ob_); q.asb = __ldcg(f.ada_sig + ob_); q.zb = __ldcg(f.zeta + ob_);
    }
    return q;
  }
  __device__ __forceinline__ float elem(int m, int n, float v0, float v1, const Pre& q) const {
    const size_t off = m < nW ? (size_t)m * ld + n : (size_t)n;
    const size_t oa = (size_t)(m < nW ? oWa : oba) + off, ob_ = (size_t)(m < nW ? oWb : obb) + off;
    if constexpr (FVB) {
      fvb_apply(q.pa, q.aa, q.sa, q.asa, q.za, Pn, ada, f, oa, v0, hy);
      fvb_apply(q.pb, q.ab, q.sb, q.asb, q.zb, Pn, ada, f, ob_, v1, hy);
    } else {
      adagrad_apply(q.pa, q.aa, Pn, ada, oa, v0, hy);
      adagrad_apply(q.pb, q.ab, Pn, ada, ob_, v1, hy);
    }
    return 0.f;
  }
  __device__ __forceinline__ void rowsum(int, int, float) const {}
};

// ---------------------------------------------------------------------------------------------
// grid barrier + kernel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void grid_barrier(unsigned long long* bar, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    // release: orders every write this CTA made before the bar.sync (cumulativity) before the arrival
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(bar) : "memory");
    unsigned long long v;
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(bar) : "memory");
    } while (v < target);
    __threadfence();   // also drops this SM's L1 lines (4-byte cp.async.ca staging goes through L1)
  }
  __syncthreads();
}

__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

#define FS_JOB(J) job_tmt(J), job_tnt(J)

// the bound of step s: fixed-order sum of the row partials (VAEB.py:340-344) (+ thetaPrior, :364), / Mg -- one CTA
template <bool TPRIOR>
__device__ __forceinline__ void bound_item(const StepParams& p, float* smem, int s) {
  const int M = p.M, G = gridDim.x;
  const int tc = p.job[J_DEC2].tiles_n, ta = p.job[J_ENC2].tiles_n;
  float t = 0.f;
  for (int r = threadIdx.x; r < M; r += NT) {
    float rsum = 0.f;
    for (int q = 0; q < tc; ++q) rsum += __ldcg(p.partial + (size_t)r * tc + q);
    for (int q = 0; q < ta; ++q) rsum += __ldcg(p.aux_part + (size_t)r * ta + q);
    t += rsum;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = 0.f;
    for (int wq = 0; wq < NW; ++wq) b += smem[wq];
    float tp = 0.f;                                        // thetaPrior (full VB), fixed order
    if constexpr (TPRIOR) {
      const float* part = p.tprior_part + (size_t)(s & 1) * G;   // double buffered by step parity
      for (int c = 0; c < G; ++c) tp += __ldcg(part + c);
    }
    p.scalars[s] = (p.bmult * b + tp) / p.Mg;
  }
  __syncthreads();
}

// per-CTA partial sum of thetaPrior into the step's half of tprior_part
__device__ __forceinline__ void store_tprior(const StepParams& p, float* smem, int s, float tp) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tp += __shfl_xor_sync(0xffffffffu, tp, o);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = tp;
  __syncthreads();
  if (threadIdx.x == 0) {
    float b = 0.f;
    for (int wq = 0; wq < NW; ++wq) b += smem[wq];
    p.tprior_part[(size_t)(s & 1) * gridDim.x + blockIdx.x] = b;
  }
  __syncthreads();
}

// phases 6-8 of one update (the weight-gradient phases), templated on the update rule of their epilogues
template <bool FVB>
__device__ __forceinline__ void update_phases(const StepParams& p, float* smem, int s, const float* x, const float* P,
                                              const float* Pu, float* Pn, const Fvb& fv, const Hyper& hy,
                                              unsigned long long& target, long long* tm) {
  const int D = p.D, H = p.H, Z = p.Z, M = p.M;
  const int G = gridDim.x, cta = blockIdx.x;
    // ---- phase 6: W2 (W6) update | dz -> dmu, dls | W1 update | the bound ---------------------
    {
      const Gemm g2 = make_gemm(p.h_d, nullptr, H, p.da2, nullptr, D, H + 1, D, M, 0, H, p.job[J_WG2]);
      const EpiAdagrad<FVB> e2{Pu, Pn, p.ada, p.oW2, p.ob2, H, D, hy, fv};
      const Gemm g6 = make_gemm(p.h_d, nullptr, H, p.dlv, nullptr, D, H + 1, D, M, 0, H, p.job[J_WG6]);
      const EpiAdagrad<FVB> e6{Pu, Pn, p.ada, p.oW6, p.ob6, H, D, hy, fv};
      const Gemm gz = make_gemm(p.da1, nullptr, H, P + p.oW1, nullptr, H, M, Z, H, 0, -1, p.job[J_DZ]);
      const EpiDz ez{p.z, p.eps, p.mu, p.ls, Z, p.la, p.kl_beta ? p.w * __ldg(p.kl_beta + s) : p.w, p.dmu, p.dls};
      const Gemm g1 = make_gemm(p.z, nullptr, Z, p.da1, nullptr, H, Z + 1, H, M, 0, Z, p.job[J_WG1]);
      const EpiAdagrad<FVB> e1{Pu, Pn, p.ada, p.oW1, p.ob1, Z, H, hy, fv};
      const int n2 = g2.c.n_items, n6 = p.cont ? g6.c.n_items : 0, nz = gz.c.n_items, n1 = g1.c.n_items;
      const int total = n2 + n6 + nz + n1 + 1;
      for (int it = cta; it < total; it += G) {
        int i = it;
        if (i < n2) { run_item<FS_JOB(J_WG2), A_KM, B_KN, PLAIN>(g2, i, e2, smem); continue; }
        i -= n2;
        if (i < n6) { run_item<FS_JOB(J_WG6), A_KM, B_KN, PLAIN>(g6, i, e6, smem); continue; }
        i -= n6;
        if (i < nz) { run_item<FS_JOB(J_DZ), A_MK, B_NK, PLAIN>(gz, i, ez, smem); continue; }
        i -= nz;
        if (i < n1) { run_item<FS_JOB(J_WG1), A_KM, B_KN, PLAIN>(g1, i, e1, smem); continue; }
        bound_item<FVB>(p, smem, s);
      }
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[6] = gtime();

    // ---- phase 7: back through the latent heads | W4, W5 update ---------------------------------
    {
      const Gemm gh = make_gemm(p.dmu, p.dls, Z, P + p.oW4, P + p.oW5, Z, M, H, Z, Z, -1, p.job[J_DHE]);
      const EpiTanhBack eh{p.h_e, p.da3, H};
      const Gemm g45 = make_gemm(p.h_e, nullptr, H, p.dmu, p.dls, Z, H + 1, Z, M, 0, H, p.job[J_WG45]);
      const EpiAdagrad2<FVB> e45{Pu, Pn, p.ada, p.oW4, p.ob4, p.oW5, p.ob5, H, Z, hy, fv};
      const int nh = gh.c.n_items, total = nh + g45.c.n_items;
      for (int it = cta; it < total; it += G) {
        if (it < nh) run_item<FS_JOB(J_DHE), A_MK, B_NK, DUALK>(gh, it, eh, smem);
        else run_item<FS_JOB(J_WG45), A_KM, B_KN, DUALN>(g45, it - nh, e45, smem);
      }
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[7] = gtime();

    // ---- phase 8: W3 update -------------------------------------------------------------------
    {
      const Gemm g = make_gemm(x, nullptr, D, p.da3, nullptr, H, D + 1, H, M, 0, D, p.job[J_WG3]);
      const EpiAdagrad<FVB> epi{Pu, Pn, p.ada, p.oW3, p.ob3, D, H, hy, fv};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_WG3), A_KM, B_KN, PLAIN>(g, it, epi, smem);
    }
}

// MODE 0: L^B / L^A on plain parameters.  1: full VB with sampled weights.  2: full VB as the reference runs it
// (VAEB.py:349-367 with :127-129 dead, SURVEY F5): the layers read the frozen MAP parameters, only the bound is
// needed from them (no backward), and (mu, sigma) follow the prior terms alone -- four phases per update.
template <int MODE>
__global__ void __launch_bounds__(NT, 1) fused_step_kernel(const StepParams p) {
  constexpr bool FVB = MODE == 1;
  extern __shared__ __align__(16) float smem[];
  const int D = p.D, H = p.H, Z = p.Z, M = p.M;
  const int G = gridDim.x, cta = blockIdx.x;
  unsigned long long target = p.bar_base;
  const Hyper hy{p.lr, p.ada_eps, p.prior, p.p2};
  const bool rec = p.timing != nullptr && cta == 0 && threadIdx.x == 0;

  for (int s = 0; s < p.n_steps; ++s) {
    const int cur = (p.parity0 + s) & 1;
    const float* P = FVB ? p.theta : p.params[cur];          // what the layers read
    const float* Pu = FVB ? p.vmu : p.params[cur];           // what the update epilogues read / write
    float* Pn = FVB ? p.vmu : p.params[cur ^ 1];
    const Fvb fv{p.vsig, p.ada_sig, p.zeta};
    const float* x = p.batch_order ? p.x_base + (size_t)__ldg(p.batch_order + s) * M * D : p.x_direct;
    long long* tm = rec ? p.timing + (size_t)s * (N_PHASES + 1) : nullptr;
    if (tm) tm[0] = gtime();

    // ---- phase 0 (sampled full VB): theta = mu + |sigma| zeta, VAEB.py:127-129; thetaPrior, :359-363 -----
    if constexpr (FVB) {
      float tp = 0.f;
      // one Philox group = four consecutive flat elements (the buffers are 16-byte aligned and padded to 4)
      for (int64_t g4 = (int64_t)cta * NT + threadIdx.x; 4 * g4 < p.total; g4 += (int64_t)G * NT) {
        const float4 m4 = __ldcg(reinterpret_cast<const float4*>(p.vmu) + g4);
        const float4 s4 = __ldcg(reinterpret_cast<const float4*>(p.vsig) + g4);
        float zt[4];
        philox_normal4(p.seed, VAEB_STREAM_ZETA, p.step0 + (uint32_t)s, 0u, (uint64_t)g4, zt);
        const float mm[4] = {m4.x, m4.y, m4.z, m4.w}, ss[4] = {s4.x, s4.y, s4.z, s4.w};
        float th[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          th[j] = mm[j] + fabsf(ss[j]) * zt[j];
          if (4 * g4 + j < p.total) tp += 0.5f * (1.0f + logf(ss[j] * ss[j]) - mm[j] * mm[j] - ss[j] * ss[j]);
        }
        reinterpret_cast<float4*>(p.zeta)[g4] = make_float4(zt[0], zt[1], zt[2], zt[3]);
        reinterpret_cast<float4*>(p.theta)[g4] = make_float4(th[0], th[1], th[2], th[3]);
      }
      store_tprior(p, smem, s, tp);
      grid_barrier(p.bar, target += G);
    }
    if constexpr (MODE == 2) {
      // reference-faithful full VB: thetaPrior and the whole (mu, sigma) update in one pass -- d/dmu = -mu - prior mu,
      // d/dsigma = 1/s - s - prior s (VAEB.py:359-363,391-393), Adagrad :426-444.  Nothing downstream reads them:
      // no barrier before the layers.
      float tp = 0.f;
      for (int64_t g4 = (int64_t)cta * NT + threadIdx.x; 4 * g4 < p.total; g4 += (int64_t)G * NT) {
        float4 m4 = __ldcg(reinterpret_cast<const float4*>(p.vmu) + g4);
        float4 s4 = __ldcg(reinterpret_cast<const float4*>(p.vsig) + g4);
        float4 am4 = __ldcg(reinterpret_cast<const float4*>(p.ada) + g4);
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
        reinterpret_cast<float4*>(p.ada)[g4] = am4;
        reinterpret_cast<float4*>(p.ada_sig)[g4] = as4;
      }
      store_tprior(p, smem, s, tp);
    }

    // ---- phase 1: encoder hidden layer ------------------------------------------------------
    {
      const Gemm g = make_gemm(x, nullptr, D, P + p.oW3, nullptr, H, M, H, D, 0, -1, p.job[J_ENC1]);
      const EpiTanh epi{P + p.ob3, p.h_e, H};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_ENC1), A_MK, B_KN, PLAIN>(g, it, epi, smem);
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[1] = gtime();

    // ---- phase 2: latent heads, reparameterisation, KL / LA row terms -----------------------
    {
      const Gemm g = make_gemm(p.h_e, nullptr, H, P + p.oW4, P + p.oW5, Z, M, Z, H, 0, -1, p.job[J_ENC2]);
      const EpiLatent epi{P + p.ob4, P + p.ob5, p.eps_inj, p.seed, p.step0 + (uint32_t)s, p.row_offset, Z, p.la,
                          g.c.tiles_n, p.mu, p.ls, p.eps, p.z, p.aux_part};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_ENC2), A_MK, B_KN, DUALN>(g, it, epi, smem);
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[2] = gtime();

    // ---- phase 3: decoder hidden layer ------------------------------------------------------
    {
      const Gemm g = make_gemm(p.z, nullptr, Z, P + p.oW1, nullptr, H, M, H, Z, 0, -1, p.job[J_DEC1]);
      const EpiTanh epi{P + p.ob1, p.h_d, H};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_DEC1), A_MK, B_KN, PLAIN>(g, it, epi, smem);
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[3] = gtime();

    // ---- phase 4: decoder output layer + log-likelihood + output deltas -----------------------
    if (p.cont) {
      const Gemm g = make_gemm(p.h_d, nullptr, H, P + p.oW2, P + p.oW6, D, M, D, H, 0, -1, p.job[J_DEC2]);
      const EpiGaussian epi{P + p.ob2, P + p.ob6, x, D, p.w, p.da2, p.dlv, p.partial, g.c.tiles_n};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_DEC2), A_MK, B_KN, DUALN>(g, it, epi, smem);
    } else {
      const Gemm g = make_gemm(p.h_d, nullptr, H, P + p.oW2, nullptr, D, M, D, H, 0, -1, p.job[J_DEC2]);
      const EpiBernoulli epi{P + p.ob2, x, D, p.w, p.da2, p.partial, g.c.tiles_n};
      for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_DEC2), A_MK, B_KN, PLAIN>(g, it, epi, smem);
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[4] = gtime();

    if constexpr (MODE == 2) {
      // the bound needs every CTA's row partials and thetaPrior sums (all written before the barrier above); the next
      // update overwrites them only after its own barriers, which wait for this CTA
      if (cta == (s % G)) bound_item<true>(p, smem, s);
      continue;
    }

    // ---- phase 5: back through the decoder output layer -------------------------------------
    {
      const EpiTanhBack epi{p.h_d, p.da1, H};
      if (p.cont) {
        const Gemm g = make_gemm(p.da2, p.dlv, D, P + p.oW2, P + p.oW6, D, M, H, D, D, -1, p.job[J_DGRAD]);
        for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_DGRAD), A_MK, B_NK, DUALK>(g, it, epi, smem);
      } else {
        const Gemm g = make_gemm(p.da2, nullptr, D, P + p.oW2, nullptr, D, M, H, D, 0, -1, p.job[J_DGRAD]);
        for (int it = cta; it < g.c.n_items; it += G) run_item<FS_JOB(J_DGRAD), A_MK, B_NK, PLAIN>(g, it, epi, smem);
      }
    }
    grid_barrier(p.bar, target += G);
    if (tm) tm[5] = gtime();

    update_phases<FVB>(p, smem, s, x, P, Pu, Pn, fv, hy, target, tm);
    grid_barrier(p.bar, target += G);
    if (tm) tm[8] = gtime();
  }
}

// ---------------------------------------------------------------------------------------------
// host: decomposition of a job into CTA items
// ---------------------------------------------------------------------------------------------
static JobCfg plan_job(int job, int M, int N, int K, int n_cta, bool dual_n) {
  const int TM = 8 * job_tmt(job), TN = 4 * job_tnt(job);
  const int TNE = dual_n ? TN / 2 : TN;
  JobCfg best{};
  best.tiles_m = (M + TM - 1) / TM;
  best.tiles_n = (N + TNE - 1) / TNE;
  const int tiles = best.tiles_m * best.tiles_n;
  double best_cost = 1e30;
  const double fma = (double)job_tmt(job) * job_tnt(job) * 2.0;   // issue cycles per k per warp (one SMSP)
  for (int ks = 1; ks <= NW; ks *= 2) {
    for (int tpi = 1; tpi * ks <= NW; ++tpi) {
      const int items = (tiles + tpi - 1) / tpi;
      const int rounds = (items + n_cta - 1) / n_cta;
      const int per_smsp = (ks * tpi + 3) / 4;
      const double kper = std::ceil((double)K / ks);
      // a lone warp reaches ~40% of its scheduler's FFMA rate (issue latency, fragment loads); more
      // resident warps hide it: time ~ (warps per scheduler + 1.5) * k steps * FFMAs per k step
      const double cost = rounds * ((per_smsp + 1.5) * kper * fma + 1500.0 + 40.0 * ks);
      if (cost < best_cost) { best_cost = cost; best.ks = ks; best.tpi = tpi; best.n_items = items; }
    }
  }
  return best;
}

}  // namespace fs

int fused_step_launch(vaeb_handle* h, const int* d_order, const float* d_kl, const float* d_xrows, int rows, int n_steps,
                      const float* d_eps, int slot0, long long* d_timing) {
  using namespace fs;
  FusedState& f = h->fused;
  const Layout& l = h->lay;
  const int D = h->D, H = h->H, Z = h->Z;
  if (!f.ready) {
    int dev = h->cfg.device, coop = 0;
    VAEB_CUDA(cudaDeviceGetAttribute(&f.n_sm, cudaDevAttrMultiProcessorCount, dev));
    VAEB_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    VAEB_REQUIRE(coop != 0, "device lacks cooperative launch");
    const void* kfns[3] = {(const void*)fused_step_kernel<0>, (const void*)fused_step_kernel<1>,
                           (const void*)fused_step_kernel<2>};
    for (const void* k : kfns) {
      VAEB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
      int occ = 0;
      VAEB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, NT, SMEM_BYTES));
      VAEB_REQUIRE(occ >= 1, "fused step kernel does not fit on an SM");
    }
    VAEB_CUDA(cudaMalloc((void**)&f.bar, sizeof(unsigned long long)));
    VAEB_CUDA(cudaMemset(f.bar, 0, sizeof(unsigned long long)));
    const size_t nb = (size_t)(l.padded + 4) * sizeof(float);
    VAEB_CUDA(cudaMalloc((void**)&f.params_alt, nb));
    VAEB_CUDA(cudaMemset(f.params_alt, 0, nb));
    f.ready = true;
  }
  if (rows != f.rows) {
    VAEB_CUDA(cudaStreamSynchronize(h->stream));
    if (f.partial) VAEB_CUDA(cudaFree(f.partial));
    if (f.aux_part) VAEB_CUDA(cudaFree(f.aux_part));
    f.partial = f.aux_part = nullptr;
    const int G = f.n_sm;
    f.job[J_ENC1] = plan_job(J_ENC1, rows, H, D, G, false);
    f.job[J_ENC2] = plan_job(J_ENC2, rows, Z, H, G, true);
    f.job[J_DEC1] = plan_job(J_DEC1, rows, H, Z, G, false);
    f.job[J_DEC2] = plan_job(J_DEC2, rows, D, H, G, h->cont);
    f.job[J_DGRAD] = plan_job(J_DGRAD, rows, H, h->cont ? 2 * D : D, G, false);
    f.job[J_WG2] = plan_job(J_WG2, H + 1, D, rows, G, false);
    f.job[J_WG6] = f.job[J_WG2];
    f.job[J_DZ] = plan_job(J_DZ, rows, Z, H, G, false);
    f.job[J_WG1] = plan_job(J_WG1, Z + 1, H, rows, G, false);
    f.job[J_DHE] = plan_job(J_DHE, rows, H, 2 * Z, G, false);
    f.job[J_WG45] = plan_job(J_WG45, H + 1, Z, rows, G, true);
    f.job[J_WG3] = plan_job(J_WG3, D + 1, H, rows, G, false);
    VAEB_CUDA(cudaMalloc((void**)&f.partial, (size_t)rows * f.job[J_DEC2].tiles_n * sizeof(float)));
    VAEB_CUDA(cudaMalloc((void**)&f.aux_part, (size_t)rows * f.job[J_ENC2].tiles_n * sizeof(float)));
    f.rows = rows;
  }
  const Workspace& s = h->ws;
  StepParams p{};
  p.D = D; p.H = H; p.Z = Z; p.M = rows;
  p.cont = h->cont ? 1 : 0;
  p.la = h->cfg.estimator == VAEB_EST_LA ? 1 : 0;
  const bool fb = h->cfg.variant == VAEB_VARIANT_FULLBAYES;
  p.w = fb ? 1.0f / (float)rows : 1.0f;
  p.kl_beta = d_kl;
  p.lr = h->cfg.learning_rate; p.ada_eps = h->cfg.adagrad_eps;
  p.prior = fb ? 0.f : h->cfg.prior_scale;
  p.p2 = fb ? h->cfg.learning_rate * 1e-6f : 0.f;
  p.params[0] = h->d_params; p.params[1] = f.params_alt;
  p.ada = h->d_ada;
  p.oW3 = l.off[l.iW3]; p.oW4 = l.off[l.iW4]; p.oW5 = l.off[l.iW5]; p.oW1 = l.off[l.iW1]; p.oW2 = l.off[l.iW2];
  p.ob3 = l.off[l.ib3]; p.ob4 = l.off[l.ib4]; p.ob5 = l.off[l.ib5]; p.ob1 = l.off[l.ib1]; p.ob2 = l.off[l.ib2];
  p.oW6 = h->cont ? l.off[l.iW6] : 0; p.ob6 = h->cont ? l.off[l.ib6] : 0;
  // rows of step s: batch_order[s] * M rows into the resident data -- or into d_xrows when both are given
  // (the staging ring of the streaming host-input updates) -- else d_xrows itself for every step
  p.x_base = (d_order && d_xrows) ? d_xrows : h->d_x; p.batch_order = d_order; p.x_direct = d_xrows;
  p.eps_inj = d_eps;
  p.seed = h->cfg.seed; p.step0 = h->step; p.row_offset = 0;
  p.h_e = s.h_e; p.mu = s.mu; p.ls = s.ls; p.eps = s.eps; p.z = s.z; p.h_d = s.h_d;
  p.da2 = s.da2; p.dlv = s.dlv; p.da1 = s.da1; p.dmu = s.dmu; p.dls = s.dls; p.da3 = s.da3;
  p.partial = f.partial; p.aux_part = f.aux_part;
  p.scalars = h->d_scalars + slot0; p.Mg = (float)rows; p.bmult = 1.0f;
  const bool fvb = h->cfg.estimator == VAEB_EST_FVB_SAMPLED;
  const bool faithful = h->cfg.estimator == VAEB_EST_FVB;
  p.fvb = fvb ? 1 : (faithful ? 2 : 0);
  if (fvb || faithful) {
    // SGVB = x.shape[0]*(sum logp + sum KL) + thetaPrior, update returns SGVB/M (VAEB.py:364,412); the data term of
    // the gradient carries the same factor M; the prior terms live in the update epilogue
    if (!f.tprior_part) VAEB_CUDA(cudaMalloc((void**)&f.tprior_part, (size_t)2 * f.n_sm * sizeof(float)));
    p.w = (float)rows; p.bmult = (float)rows;
    p.prior = h->cfg.prior_scale; p.p2 = 0.f;
    p.vmu = h->d_vmu; p.vsig = h->d_vsig; p.ada = h->d_ada_mu; p.ada_sig = h->d_ada_sig;
    p.theta = h->d_theta; p.zeta = h->d_zeta; p.tprior_part = f.tprior_part; p.total = l.total;
    if (faithful) p.params[1] = p.params[0];     // the MAP parameters are frozen (VAEB.py:119,352): no ping-pong
  }
  p.n_steps = n_steps; p.parity0 = 0;
  p.bar = f.bar; p.bar_base = f.bar_count;
  p.timing = d_timing;
  for (int j = 0; j < J_COUNT; ++j) p.job[j] = f.job[j];
  void* args[] = {&p};
  const void* kfn = fvb ? (const void*)fused_step_kernel<1>
                        : (faithful ? (const void*)fused_step_kernel<2> : (const void*)fused_step_kernel<0>);
  VAEB_CUDA(cudaLaunchCooperativeKernel(kfn, dim3(f.n_sm), dim3(NT), args, SMEM_BYTES, h->stream));
  const int phases = faithful ? 4 : N_PHASES + (fvb ? 1 : 0);           // grid barriers per update
  f.bar_count += (unsigned long long)f.n_sm * (unsigned long long)phases * (unsigned long long)n_steps;
  ++h->launches;
  h->step += (uint32_t)n_steps;
  if ((n_steps & 1) && !fvb && !faithful) std::swap(h->d_params, f.params_alt);   // theta now lives in the other buffer
  h->grads_have_prior = false;
  invalidate_weight_mirrors(h);
  return VAEB_OK;
}
