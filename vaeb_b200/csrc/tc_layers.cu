// The wide layers of the AEVB step on the 5th-generation tensor cores: tcgen05.mma with bf16
// operands staged by TMA (128B swizzle), fp32 accumulation in TMEM, fused epilogues read back
// with tcgen05.ld.  NS = 1: plain bf16 operands (1e-2 tier).  NS = 2: every operand is carried as
// bf16 hi + bf16 lo and each k-step issues hi*hi + hi*lo + lo*hi into the same accumulator
// ("bf16x3": ~2^-17 relative per product, the fp32 parity tier on tensor cores).
//   enc1      h_e  = tanh(x.W3 + b3)                       VAEB.py:246     A K-major,  B MN-major
//   dec2      a    = h_d.W2 + b2 -> Bernoulli log-lik, da  VAEB.py:263,311 A K-major,  B MN-major
//   dgrad     da1  = (da.W2^T) * (1 - h_d^2)               T.grad :397     A K-major,  B K-major
//   wgrad     gW   = [act|1]^T . delta (bias row included) T.grad :397     A MN-major, B MN-major
// Warp roles (640 threads): w0 TMA producer, w1 MMA issuer, w2 TMEM allocator, w4-19 epilogue (four
// warps per TMEM lane quarter, each owning a quarter of the tile's columns: at M = 100 the whole
// layer is 8-13 CTAs, so the elementwise epilogue needs all the threads it can get).
#include <cuda_bf16.h>
#include <cstdlib>

#include "common.cuh"
#include "launchers.h"
#include "tc_common.cuh"
#include "tc_layers.h"
#include "philox.cuh"

#include "tc_epilogues.cuh"

namespace {


// contraction extent of one ring stage: the weight gradients in plain bf16 (both operands MN-major, one 3-D box each)
// take 128 rows per stage -- two 32 KB boxes per mbarrier round trip instead of two 16 KB ones: their producer is bound
// by issues (wait + expect_tx + ~120 ns per box, the TMA fill-rate probe, profiles/r1_c3_phases.txt), not by bytes
template <bool A_MN, bool B_MN, int NS>
constexpr int stage_k() { return (A_MN && B_MN && NS == 1) ? 2 * BK : BK; }

template <int BN, int NS, bool A_MN, int SK = BK>
struct LayerSmem {
  static constexpr int A_BYTES = BM * SK * 2;
  static constexpr int B_BYTES = BN * SK * 2;
  static constexpr int STAGE_BYTES = NS * (A_BYTES + B_BYTES);
  // activation layers in plain bf16 (NS = 1): 3-4 stages so that TWO CTAs share an SM and one tile's epilogue
  // overlaps the other's loads and MMAs (the kernel is one tile per CTA); bf16x3 stages are twice as large: one CTA
  // per SM.  Weight gradients (A MN-major: split-K, at most one CTA per SM, a long contraction): the whole shared
  // memory as ring -- their operand stream is bound by bytes in flight / L2 latency.
  static constexpr bool TWO_PER_SM = NS == 1 && !A_MN;
  static constexpr int BUDGET = TWO_PER_SM ? 104 * 1024 : 200 * 1024;
  static constexpr int STAGES = (BUDGET / STAGE_BYTES) > 6 ? 6 : (BUDGET / STAGE_BYTES);
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
  static_assert(STAGES >= 2, "tile too large");
};

// one output tile (bx, by) of split-K slice bz of nz; nx = column tiles of the layer
template <int BN, bool A_MN, bool B_MN, int NS, class Epi>
__device__ __forceinline__ void layer_tile(const LayerMaps& maps, Epi epi, int M, int N, int K, int a_row_off, int bx,
                                           int by, int bz, int nx, int nz) {
  constexpr int SK = stage_k<A_MN, B_MN, NS>();
  using S = LayerSmem<BN, NS, A_MN, SK>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + S::STAGES * S::STAGE_BYTES);
  uint64_t* empty = full + S::STAGES;
  uint64_t* tmem_full = empty + S::STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = by * BM, n0 = bx * BN;
  const int nkb_all = (K + SK - 1) / SK;       // ring stages over the whole contraction
  // split-K (weight gradients at large batch: few output tiles, long contraction): slice z of gridDim.z
  const int kb0 = (int)(((long long)nkb_all * bz) / nz);
  const int nkb = (int)(((long long)nkb_all * (bz + 1)) / nz) - kb0;
  epi.split(bz);
  constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&maps.a_hi);
    tc::tma_prefetch_desc(&maps.b_hi);
    if (NS == 2) { tc::tma_prefetch_desc(&maps.a_lo); tc::tma_prefetch_desc(&maps.b_lo); }
    for (int s = 0; s < S::STAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
    tc::mbar_init(tmem_full, 1);
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) may run while
  // the previous kernel of the stream drains; its results are visible only after griddepcontrol.wait.  The next
  // kernel may start its own prologue as soon as every CTA of this one got here.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S::STAGES;
      tc::mbar_wait(&empty[s], ((kb / S::STAGES) & 1) ^ 1);
      uint8_t* base = smem + s * S::STAGE_BYTES;
      tc::mbar_expect_tx(&full[s], S::STAGE_BYTES);
#pragma unroll
      for (int sp = 0; sp < NS; ++sp) {
        uint8_t* a = base + sp * S::A_BYTES;
        uint8_t* b = base + NS * S::A_BYTES + sp * S::B_BYTES;
        const CUtensorMap* ta = sp ? &maps.a_lo : &maps.a_hi;
        const CUtensorMap* tb = sp ? &maps.b_lo : &maps.b_hi;
        // MN-major operands: ONE 3-D box per tile and k block (its BM/64 resp. BN/64 column groups land as consecutive
        // 8 KB blocks) -- the producer is bound by the number of boxes it issues, not by their bytes
        if (A_MN) {   // A stored [K rows, M contiguous]: the row offset applies to the K coordinate
          tc::tma_load_3d(a, ta, &full[s], 0, a_row_off + (kb0 + kb) * SK, m0 / 64);
        } else {      // A stored [M rows, K contiguous]
          tc::tma_load_2d(a, ta, &full[s], (kb0 + kb) * SK, a_row_off + m0);
        }
        if (B_MN) {
          tc::tma_load_3d(b, tb, &full[s], 0, (kb0 + kb) * SK, n0 / 64);
        } else {
          tc::tma_load_2d(b, tb, &full[s], (kb0 + kb) * SK, n0);
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer =====
    constexpr uint32_t idesc = tc::make_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S::STAGES;
      tc::mbar_wait(&full[s], (kb / S::STAGES) & 1);
      tc::tc_fence_after();
      const uint32_t a = tc::smem_u32(smem + s * S::STAGE_BYTES);
      const uint32_t b = a + NS * S::A_BYTES;
      constexpr uint32_t GRP = 128u * SK;      // bytes of one 64-wide column group of an MN-major stage
#pragma unroll
      for (int k = 0; k < SK / 16; ++k) {
        const uint64_t dah = A_MN ? tc::desc_mnmajor(a, k, GRP) : tc::desc_kmajor(a, k);
        const uint64_t dbh = B_MN ? tc::desc_mnmajor(b, k, GRP) : tc::desc_kmajor(b, k);
        tc::umma_bf16(tmem_base, dah, dbh, idesc, (kb | k) != 0 ? 1u : 0u);
        if (NS == 2) {
          const uint64_t dal = A_MN ? tc::desc_mnmajor(a + S::A_BYTES, k, GRP) : tc::desc_kmajor(a + S::A_BYTES, k);
          const uint64_t dbl = B_MN ? tc::desc_mnmajor(b + S::B_BYTES, k, GRP) : tc::desc_kmajor(b + S::B_BYTES, k);
          tc::umma_bf16(tmem_base, dah, dbl, idesc, 1u);
          tc::umma_bf16(tmem_base, dal, dbh, idesc, 1u);
        }
      }
      tc::umma_commit(&empty[s]);
    }
    tc::umma_commit(tmem_full);
  } else if (warp >= 4) {
    // ===== epilogue: warp e = warp-4 reads lane quarter e%4, column slice e/4 of the tile =====
    const int q = warp & 3, cs = (warp - 4) >> 2;
    constexpr int SLICE = BN / (EPI_WARPS / 4);
    const int row = m0 + q * 32 + lane;
    const bool ok = row < M;
    epi.begin();
    tc::mbar_wait(tmem_full, 0);
    tc::tc_fence_after();
#pragma unroll 1
    for (int c = cs * SLICE; c < (cs + 1) * SLICE; c += 16) {
      float v[16];
      tc::tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
      tc::tmem_ld_wait();
      if (n0 + c < N) epi.chunk(row, ok, n0 + c, N, v);
    }
    epi.end(row, ok, bx * (EPI_WARPS / 4) + cs, nx * (EPI_WARPS / 4));
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int BN, bool A_MN, bool B_MN, int NS, class Epi>
__global__ void __launch_bounds__(TC_THREADS, (NS == 1 && !A_MN) ? 2 : 1)
tc_layer_kernel(const __grid_constant__ LayerMaps maps, Epi epi, int M, int N, int K, int a_row_off) {
  layer_tile<BN, A_MN, B_MN, NS, Epi>(maps, epi, M, N, K, a_row_off, blockIdx.x, blockIdx.y, blockIdx.z, gridDim.x,
                                      gridDim.z);
}

// Every weight-gradient GEMM of the step in ONE launch: gW = [act|1]^T . delta for W2, W1, [W4|W5], W3 (T.grad, VAEB.py:397).
// Block b belongs to the job whose [first_block, first_block + tiles * splits) holds it; the slices of a job go to its
// scratch region and are summed in a fixed order by the tail kernel.  The thin gradients (W1: 21 x 500, [W4|W5]: 501 x 40)
// no longer cost a launch of their own (~7.5 us each for 4 tiles), the wide ones share one wave.
struct WgradJob {
  LayerMaps maps;
  EpiWgradTc epi;
  int M, N, K, a_row_off, tiles_n, tiles_m, splits, first_block;
};
struct WgradAllArgs { WgradJob job[4]; int n_jobs; };

template <int BN, int NS>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_wgrad_all_kernel(const __grid_constant__ WgradAllArgs args) {
  int j = 0;
#pragma unroll
  for (int q = 1; q < 4; ++q)
    if (q < args.n_jobs && (int)blockIdx.x >= args.job[q].first_block) j = q;
  const WgradJob& J = args.job[j];
  const int local = blockIdx.x - J.first_block;
  const int per = J.tiles_n * J.tiles_m;
  const int bz = local / per, t = local - bz * per;
  layer_tile<BN, true, true, NS, EpiWgradTc>(J.maps, J.epi, J.M, J.N, J.K, J.a_row_off, t % J.tiles_n, t / J.tiles_n, bz,
                                             J.tiles_n, J.splits);
}

thread_local bool g_pdl = false;   // set and read within one step of one thread (tc_setup)

// ---- persistent form for large batches (A K-major: the activation layers) ---------------------------------
// One CTA per SM walks the tile list (tile = blockIdx.x + i * gridDim.x; tiles of one row block are neighbours, so
// the A rows are fetched from HBM once and shared through L2).  Two TMEM accumulators: the epilogue of tile i
// (16 warps) overlaps the loads and MMAs of tile i+1; the operand ring keeps its phase across tiles, so the TMA
// producer runs ahead into the next tile while the last k blocks of this one are still being contracted.  BN up to
// 256 (2 x 256 TMEM columns): a 128 x 256 tile re-reads A half as often as two 128 x 128 tiles -- these layers are
// bound by L2 -> shared-memory operand traffic (K <= 784: 64 flop per operand byte at 128 x 128).
template <int BN, int NS>
struct PersistSmem {
  static constexpr int A_BYTES = BM * BK * 2;               // one 128-row block of A
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = NS * (A_BYTES + B_BYTES);
  static constexpr int BUDGET = 208 * 1024;
  static constexpr int STAGES = (BUDGET / STAGE_BYTES) > 8 ? 8 : (BUDGET / STAGE_BYTES);
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
  static_assert(STAGES >= 2, "tile too large");
};

// Which tiles a CTA of the persistent kernel works on.  When the last column tile is a sliver (N = 784, BN = 256: 16 of 256
// columns) it costs about a third of a full tile (its A operand still streams in; the MMAs are N = 16 and the epilogue
// one chunk), and plain round-robin gives whole CTAs nothing but slivers (148 % 4 == 0) while the others run four full
// tiles: 66 us for dec2 at 16384 rows.  So: full tiles round-robin first; slivers go, up to three each, to the CTAs that
// got one full tile fewer, the rest round-robin.
// a last column tile at most a quarter wide
__host__ __device__ inline bool tile_sliver(int N, int bn, int tiles_n) { return tiles_n > 1 && (N - (tiles_n - 1) * bn) * 4 <= bn; }

struct TileSeq {
  int G, b, nfn, F, T, base, extra, nf, p1_ctas, p1_total, np1;
  __host__ __device__ TileSeq(int tiles_m, int tiles_n, bool sliver, int grid, int cta) {
    G = grid; b = cta;
    nfn = tiles_n - (sliver ? 1 : 0);
    F = tiles_m * nfn; T = sliver ? tiles_m : 0;
    base = F / G; extra = F % G;
    nf = base + (b < extra ? 1 : 0);
    p1_ctas = G - extra;                                   // CTAs with `base` full tiles (all of them when extra == 0)
    p1_total = T < 3 * p1_ctas ? T : 3 * p1_ctas;
    np1 = 0;
    if (b >= extra && b - extra < p1_total) np1 = (p1_total - (b - extra) + p1_ctas - 1) / p1_ctas;
  }
  __host__ __device__ bool get(int i, int& tm, int& tn) const {
    if (i < nf) { const int f = b + i * G; tm = f / nfn; tn = f - tm * nfn; return true; }
    i -= nf;
    if (i < np1) { tm = (b - extra) + i * p1_ctas; tn = nfn; return true; }
    i -= np1;
    const int j = p1_total + b + i * G;
    if (j < T) { tm = j; tn = nfn; return true; }
    return false;
  }
};

// ncu: tensor pipe 25 % active, L2 slices 25 %, 6.8 TB/s of L2 -> shared-memory fill (46 GB/s per SM, the same rate the
// IS kernel streams W2^T at): the fill rate bounds these layers.
template <int BN, bool B_MN, int NS, class Epi>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_layer_persistent_kernel(const __grid_constant__ LayerMaps maps, Epi epi, int M, int N, int K, int a_row_off) {
  using S = PersistSmem<BN, NS>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + S::STAGES * S::STAGE_BYTES);
  uint64_t* empty = full + S::STAGES;
  uint64_t* tmem_full = empty + S::STAGES;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;        // [2]
  uint32_t* tmem_slot = (uint32_t*)(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (K + BK - 1) / BK;
  const int tiles_n = (N + BN - 1) / BN, tiles_m = (M + BM - 1) / BM;
  // a last column tile at most a quarter wide is a "sliver" (see TileSeq)
  const TileSeq seq(tiles_m, tiles_n, tile_sliver(N, BN, tiles_n), (int)gridDim.x, (int)blockIdx.x);
  constexpr uint32_t ACC_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
  constexpr uint32_t NBUF = 2;                          // accumulator sets in TMEM
  constexpr uint32_t TMEM_COLS = NBUF * ACC_COLS;
  static_assert(TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM allocation");

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&maps.a_hi);
    tc::tma_prefetch_desc(&maps.b_hi);
    if (NS == 2) { tc::tma_prefetch_desc(&maps.a_lo); tc::tma_prefetch_desc(&maps.b_lo); }
    for (int s = 0; s < S::STAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { tc::mbar_init(&tmem_full[b], 1); tc::mbar_init(&tmem_empty[b], EPI_WARPS); }
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    uint32_t it = 0;                                   // k blocks issued so far (ring position across tiles)
    int tm, tn;
    for (int lt = 0; seq.get(lt, tm, tn); ++lt) {
      const int m0 = tm * BM, n0 = tn * BN;
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = it % S::STAGES;
        tc::mbar_wait(&empty[s], ((it / S::STAGES) & 1) ^ 1);
        uint8_t* base = smem + s * S::STAGE_BYTES;
        tc::mbar_expect_tx(&full[s], S::STAGE_BYTES);
#pragma unroll
        for (int sp = 0; sp < NS; ++sp) {
          uint8_t* a = base + sp * S::A_BYTES;
          uint8_t* b = base + NS * S::A_BYTES + sp * S::B_BYTES;
          const CUtensorMap* ta = sp ? &maps.a_lo : &maps.a_hi;
          const CUtensorMap* tb = sp ? &maps.b_lo : &maps.b_hi;
          tc::tma_load_2d(a, ta, &full[s], kb * BK, a_row_off + m0);
          if (B_MN) {
            tc::tma_load_3d(b, tb, &full[s], 0, kb * BK, n0 / 64);      // one box: BN/64 column groups
          } else {
            tc::tma_load_2d(b, tb, &full[s], kb * BK, n0);
          }
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer =====
    uint32_t it = 0, lt = 0;                           // ring position; tiles done by this CTA
    int tm, tn;
    for (; seq.get((int)lt, tm, tn); ++lt) {
      const uint32_t buf = lt % NBUF, use = lt / NBUF;
      // a sliver's MMAs are only as wide as its live columns (UMMA N: a multiple of 16)
      const int n_live = N - tn * BN;
      const uint32_t idesc = tc::make_idesc_bf16(BM, n_live >= BN ? BN : ((n_live + 15) & ~15), 0, B_MN ? 1 : 0);
      tc::mbar_wait(&tmem_empty[buf], (use & 1) ^ 1);           // the epilogue drained this accumulator set
      tc::tc_fence_after();
      const uint32_t acc = tmem_base + buf * ACC_COLS;
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = it % S::STAGES;
        tc::mbar_wait(&full[s], (it / S::STAGES) & 1);
        tc::tc_fence_after();
        const uint32_t a = tc::smem_u32(smem + s * S::STAGE_BYTES);
        const uint32_t b = a + NS * S::A_BYTES;
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          const uint64_t dbh = B_MN ? tc::desc_mnmajor(b, k, 8192u) : tc::desc_kmajor(b, k);
          const uint64_t dbl = NS == 2 ? (B_MN ? tc::desc_mnmajor(b + S::B_BYTES, k, 8192u) : tc::desc_kmajor(b + S::B_BYTES, k)) : 0;
          const uint64_t dah = tc::desc_kmajor(a, k);
          tc::umma_bf16(acc, dah, dbh, idesc, (kb | k) != 0 ? 1u : 0u);
          if (NS == 2) {
            const uint64_t dal = tc::desc_kmajor(a + S::A_BYTES, k);
            tc::umma_bf16(acc, dah, dbl, idesc, 1u);
            tc::umma_bf16(acc, dal, dbh, idesc, 1u);
          }
        }
        tc::umma_commit(&empty[s]);
      }
      tc::umma_commit(&tmem_full[buf]);
    }
  } else if (warp >= 4) {
    // ===== epilogue: warp e = warp-4 reads lane quarter e%4, column slice e/4 of the tile =====
    const int q = warp & 3, cs = (warp - 4) >> 2;
    constexpr int SLICE = BN / (EPI_WARPS / 4);
    uint32_t lt = 0;
    int tm, tn;
    for (; seq.get((int)lt, tm, tn); ++lt) {
      const int n0 = tn * BN;
      const uint32_t buf = lt % NBUF, use = lt / NBUF;
      const int row = tm * BM + q * 32 + lane;
      const bool ok = row < M;
      epi.begin();
      const uint32_t acc = tmem_base + buf * ACC_COLS + ((uint32_t)(q * 32) << 16);
      // the global operand of chunk i+1 (one 32-byte sector of a bf16 mirror) is requested before chunk i is finished:
      // 4 warps per scheduler, each a serial chain TMEM read -> global operand -> math -> store, cannot hide that
      // latency otherwise (ncu: 22 % of the samples on the first use of the load)
      constexpr int NCH = SLICE / 16;
      // chunks of this warp's column slice that hold live columns (a sliver tile: at most one warp group has any)
      int live = (N - n0 - cs * SLICE + 15) >> 4;
      live = live < 0 ? 0 : (live > NCH ? NCH : live);
      if (live == 0) {                                      // nothing to read: hand the accumulators straight back
        tc::mbar_wait(&tmem_full[buf], use & 1);
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&tmem_empty[buf]);
      } else if constexpr (Epi::PREFETCH) {
        uint32_t pw[2][8];
        bool ph[2];
        ph[0] = (n0 + cs * SLICE < N) && epi.preload(row, ok, n0 + cs * SLICE, N, pw[0]);
        tc::mbar_wait(&tmem_full[buf], use & 1);            // the first request overlaps the wait for the accumulator
        tc::tc_fence_after();
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          if (i >= live) break;
          const int c = cs * SLICE + 16 * i;
          if (i + 1 < NCH) ph[(i + 1) & 1] = (n0 + c + 16 < N) && epi.preload(row, ok, n0 + c + 16, N, pw[(i + 1) & 1]);
          float v[16];
          tc::tmem_ld16(acc + (uint32_t)c, v);
          tc::tmem_ld_wait();
          if (i == live - 1) {                              // last read of this warp: hand the accumulators back early
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&tmem_empty[buf]);
          }
          if (n0 + c < N) epi.chunk(row, ok, n0 + c, N, v, ph[i & 1] ? pw[i & 1] : nullptr);
        }
      } else {
        tc::mbar_wait(&tmem_full[buf], use & 1);
        tc::tc_fence_after();
#pragma unroll 1
        for (int i = 0; i < live; ++i) {
          const int c = cs * SLICE + 16 * i;
          float v[16];
          tc::tmem_ld16(acc + (uint32_t)c, v);
          tc::tmem_ld_wait();
          if (i == live - 1) {
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&tmem_empty[buf]);
          }
          epi.chunk(row, ok, n0 + c, N, v);
        }
      }
      epi.end(row, ok, tn * (EPI_WARPS / 4) + cs, tiles_n * (EPI_WARPS / 4));
    }
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int BN, bool B_MN, int NS, class Epi>
cudaError_t launch_layer_persistent(cudaStream_t st, const LayerMaps& maps, const Epi& epi, int M, int N, int K,
                                    int a_row_off) {
  using S = PersistSmem<BN, NS>;
  auto kfn = tc_layer_persistent_kernel<BN, B_MN, NS, Epi>;
  static bool attr_done = false;   // per instantiation
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    if (e != cudaSuccess) return e;
    attr_done = true;
  }
  const int tiles = ((N + BN - 1) / BN) * ((M + BM - 1) / BM);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(tiles < 148 ? tiles : 148);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  // always a programmatic dependent launch: one CTA per SM with ~200 KB of shared memory never shares an SM with the
  // kernel before it, so its prologue (barriers, TMEM, descriptors) simply hides behind that kernel's tail
  // (16384 rows, bf16: 250 -> 239 us per update)
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kfn, maps, epi, M, N, K, a_row_off);
}

// the persistent form pays off from about one 128 x 256 tile per SM (4096 rows: 145 vs 142 us, bf16x3 190 vs 169 us)
inline bool use_persistent(int M, int N, int bn) {
  return ((N + bn - 1) / bn) * ((M + BM - 1) / BM) >= 120;   // 8192 rows x 500: 128 tiles (measured: 196 -> 170 us per update)
}


template <int BN, bool A_MN, bool B_MN, int NS, class Epi>
cudaError_t launch_layer(cudaStream_t st, const LayerMaps& maps, const Epi& epi, int M, int N, int K, int a_row_off,
                         int splits = 1) {
  using S = LayerSmem<BN, NS, A_MN, stage_k<A_MN, B_MN, NS>()>;
  auto kfn = tc_layer_kernel<BN, A_MN, B_MN, NS, Epi>;
  static bool attr_done = false;   // per instantiation
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    if (e != cudaSuccess) return e;
    attr_done = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((N + BN - 1) / BN, (M + BM - 1) / BM, splits);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = S::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  // worth it when launch latency and prologue dominate, i.e. when every kernel of the step is at most about one
  // wave (tc_set_pdl): 2048 rows 195 -> 163 us per update.  With several waves the early CTAs of the dependent grid
  // only take SM slots from the tail of the previous kernel (16384 rows, bf16: 463 -> 494 us).
  cfg.numAttrs = g_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kfn, maps, epi, M, N, K, a_row_off);
}

template <bool A_MN, bool B_MN, class Epi>
cudaError_t dispatch_layer(cudaStream_t st, int ns, int bn, const LayerMaps& maps, const Epi& epi, int M, int N, int K,
                           int a_row_off, int splits = 1) {
  if constexpr (!A_MN) {
    if (bn == 256) {                   // tc_act_bn chose the persistent form
      // (32 accumulator columns per TMEM read measured slower here: the Bernoulli epilogue loses its operand prefetch,
      // dec2 57.5 -> 62.6 us, and the tanh / dgrad epilogues gain nothing)
      if (ns == 2) return launch_layer_persistent<256, B_MN, 2, Epi>(st, maps, epi, M, N, K, a_row_off);
      return launch_layer_persistent<256, B_MN, 1, Epi>(st, maps, epi, M, N, K, a_row_off);
    }
  }
  if (ns == 2) {
    if (bn == 128) return launch_layer<128, A_MN, B_MN, 2, Epi>(st, maps, epi, M, N, K, a_row_off, splits);
    return launch_layer<64, A_MN, B_MN, 2, Epi>(st, maps, epi, M, N, K, a_row_off, splits);
  }
  if (bn == 128) return launch_layer<128, A_MN, B_MN, 1, Epi>(st, maps, epi, M, N, K, a_row_off, splits);
  return launch_layer<64, A_MN, B_MN, 1, Epi>(st, maps, epi, M, N, K, a_row_off, splits);
}

// Split-K plan of a weight-gradient GEMM [Mo x No] over K: as many K slices as fill the SMs once, at least
// 8 k blocks each.  The slices go to scratch and are summed in a fixed order (deterministic, unlike atomics).
int tc_wgrad_splits(int Mo, int No, int K, int bn, int ns) {
  const int tiles = ((No + bn - 1) / bn) * ((Mo + BM - 1) / BM);
  const int sk = ns == 1 ? 2 * BK : BK;           // stage_k of the weight-gradient kernel
  const int nst = (K + sk - 1) / sk;              // ring stages over the contraction
  int s = 148 / (tiles > 0 ? tiles : 1);
  if (s > nst * sk / (8 * BK)) s = nst * sk / (8 * BK);
  if (s > nst) s = nst;
  return s < 1 ? 1 : s;
}

__global__ void __launch_bounds__(256)
wgrad_split_reduce_kernel(const float* __restrict__ scratch, int splits, size_t stride, int n_w, int n_b,
                          float* __restrict__ gW, float* __restrict__ gb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_w + n_b) return;
  float a = 0.f;
  for (int z = 0; z < splits; ++z) a += scratch[(size_t)z * stride + i];
  if (i < n_w) gW[i] = a; else gb[i - n_w] = a;
}

// One launch sums the split-K slices of every weight gradient of the step (blockIdx.y = job) in a fixed order.
// kind 0: scratch slice [n_w | n_b] -> gW, gb.  kind 1 (heads): slice [(H+1) x 2Z], column c < Z -> W4 / b4, else W5 / b5.
__global__ void __launch_bounds__(256)
wgrad_reduce_all_kernel(TcReduceJobs jobs) {
  const TcReduceJob& j = jobs.job[blockIdx.y];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n_w + j.n_b) return;
  float a = 0.f;
  for (int z = 0; z < j.splits; ++z) a += j.scratch[(size_t)z * j.stride + i];
  if (j.kind == 0) {
    if (i < j.n_w) j.gW[i] = a; else j.gb[i - j.n_w] = a;
  } else if (j.kind == 2) {            // interleaved Gaussian head [(H+1) x 2D]: column 2d -> W2 / b2, 2d + 1 -> W6 / b6
    const int D = j.Z, H = j.H;
    const int k = i / (2 * D), c = i - k * 2 * D, d = c >> 1;
    float* gW = (c & 1) ? j.gW2 : j.gW;
    float* gb = (c & 1) ? j.gb2 : j.gb;
    if (k < H) gW[(size_t)k * D + d] = a; else gb[d] = a;
  } else {
    const int Z = j.Z, H = j.H;
    const int k = i / (2 * Z), c = i - k * 2 * Z;
    float* gW = c < Z ? j.gW : j.gW2;
    float* gb = c < Z ? j.gb : j.gb2;
    const int jj = c < Z ? c : c - Z;
    if (k < H) gW[(size_t)k * Z + jj] = a; else gb[jj] = a;
  }
}

cudaError_t reduce_all_impl(cudaStream_t st, int64_t* launches, const TcReduceJobs& jobs) {
  if (jobs.n == 0) return cudaSuccess;
  int most = 0;
  for (int q = 0; q < jobs.n; ++q) most = jobs.job[q].n_w + jobs.job[q].n_b > most ? jobs.job[q].n_w + jobs.job[q].n_b : most;
  wgrad_reduce_all_kernel<<<dim3((most + 255) / 256, jobs.n), 256, 0, st>>>(jobs);
  ++*launches;
  return cudaGetLastError();
}

// a scratch region has one job (a GEMM launched again -- the per-phase profiler repeats launches -- replaces it)
bool add_reduce_job(TcReduceJobs* jobs, const TcReduceJob& j) {
  for (int q = 0; q < jobs->n; ++q)
    if (jobs->job[q].scratch == j.scratch) { jobs->job[q] = j; return true; }
  if (jobs->n >= TC_MAX_REDUCE_JOBS) return false;
  jobs->job[jobs->n++] = j;
  return true;
}

cudaError_t tc_wgrad_generic(cudaStream_t st, int64_t* launches, const LayerMaps& maps, int ns, int bn, int Kred,
                             int Hreal, int N, int a_row_off, float* gW, float* gb, float* scratch,
                             float* gW6 = nullptr, float* gb6 = nullptr) {
  int splits = scratch ? tc_wgrad_splits(Hreal + 1, N, Kred, bn, ns) : 1;
  const size_t stride = (size_t)(Hreal + 1) * N;
  if (gW6) {
    // Gaussian head: the slice holds the interleaved columns of [W2|W6]' -- always through scratch, the reduction
    // also de-interleaves (N = 2D)
    if (!scratch) return cudaErrorInvalidValue;
    while (splits > 1 && (size_t)splits * stride > tc_wgrad_scratch_elems(0, 0)) --splits;
    EpiWgradTc epi{nullptr, nullptr, Hreal, N, scratch, stride};
    ++*launches;
    cudaError_t e = dispatch_layer<true, true>(st, ns, bn, maps, epi, Hreal + 1, N, Kred, a_row_off, splits);
    if (e != cudaSuccess) return e;
    TcReduceJobs one;
    one.job[0] = TcReduceJob{scratch, splits, stride, (Hreal + 1) * N, 0, gW, gb, gW6, gb6, 2, Hreal, N / 2};
    one.n = 1;
    return reduce_all_impl(st, launches, one);
  }
  EpiWgradTc epi{gW, gb, Hreal, N, splits > 1 ? scratch : nullptr, stride};
  ++*launches;
  cudaError_t e = dispatch_layer<true, true>(st, ns, bn, maps, epi, Hreal + 1, N, Kred, a_row_off, splits);
  if (e != cudaSuccess || splits == 1) return e;
  const int tot = (int)stride;
  wgrad_split_reduce_kernel<<<(tot + 255) / 256, 256, 0, st>>>(scratch, splits, stride, Hreal * N, N, gW, gb);
  ++*launches;
  return cudaGetLastError();
}

// fp32 [rows, cols] (leading dim ld_src) -> bf16 hi (/lo) mirrors [rows, ld_dst]; column `ones_col`
// (>= cols) is set to 1 so that a weight-gradient GEMM over the mirror also yields the bias gradient.
__global__ void __launch_bounds__(256)
split_matrix_kernel(const float* __restrict__ src, int64_t rows, int cols, int ld_src, __nv_bfloat16* __restrict__ hi,
                    __nv_bfloat16* __restrict__ lo, int ld_dst, int ones_col) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * ld_dst) return;
  const int64_t r = i / ld_dst;
  const int c = (int)(i % ld_dst);
  float v = 0.f;
  if (c < cols) v = src[r * ld_src + c];
  else if (c == ones_col) v = 1.0f;
  put_split(hi, lo, (size_t)i, v);
}

// src2 != nullptr: the mirror interleaves two matrices column-wise (column 2c = src, 2c + 1 = src2: the Gaussian head)
struct MirrorSeg { const float* src; __nv_bfloat16* hi; __nv_bfloat16* lo; int rows, cols, ld; const float* src2; };
__global__ void __launch_bounds__(256)
mirror_weights_kernel(MirrorSeg s0, MirrorSeg s1) {
  const MirrorSeg& s = blockIdx.y == 0 ? s0 : s1;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s.src == nullptr || i >= (int64_t)s.rows * s.cols) return;
  const int r = (int)(i / s.cols), c = (int)(i % s.cols);
  if (s.src2) {
    put_split(s.hi, s.lo, (size_t)r * s.ld + 2 * c, s.src[i]);
    put_split(s.hi, s.lo, (size_t)r * s.ld + 2 * c + 1, s.src2[i]);
  } else {
    put_split(s.hi, s.lo, (size_t)r * s.ld + c, s.src[i]);
  }
}

// Every per-step weight preparation of the large-batch path in ONE launch (blockIdx.y = task):
//   0: W3 -> bf16 mirror   1: W2 -> mirror   2: [W4^T;W5^T] fp32 + mirror   3: interleaved heads mirror   4: W1 -> mirror
struct PrepArgs {
  const float *W3, *W2, *W4, *W5, *W1, *W6;      // W6 != nullptr (Gaussian decoder): the W2 mirror holds [W2|W6]' interleaved
  __nv_bfloat16 *w3h, *w3l, *w2h, *w2l, *w45h, *w45l, *whh, *whl, *w1h, *w1l;
  float* w45t;
  int D, H, Z, ldh, ldd, ldq;
};
// row-major fp32 [rows, cols] -> bf16 hi (/lo) mirror [rows, ld]: four elements per thread when cols % 4 == 0
// (16-byte loads, 8-byte stores), else one
__device__ __forceinline__ void mirror_quad(const float* __restrict__ src, __nv_bfloat16* hi, __nv_bfloat16* lo,
                                            int64_t q, int rows, int cols, int ld) {
  if ((cols & 3) == 0 && (ld & 3) == 0 && (((uintptr_t)src) & 15u) == 0 && ((((uintptr_t)hi) | ((uintptr_t)lo)) & 7u) == 0) {
    const int64_t i = 4 * q;
    if (i >= (int64_t)rows * cols) return;
    const float4 v = *reinterpret_cast<const float4*>(src + i);
    const size_t o = (size_t)(i / cols) * ld + (i % cols);
    const uint32_t h0 = pack_bf16x2(v.x, v.y), h1 = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(hi + o) = make_uint2(h0, h1);
    if (lo)
      *reinterpret_cast<uint2*>(lo + o) =
          make_uint2(pack_bf16x2(v.x - __uint_as_float(h0 << 16), v.y - __uint_as_float(h0 & 0xffff0000u)),
                     pack_bf16x2(v.z - __uint_as_float(h1 << 16), v.w - __uint_as_float(h1 & 0xffff0000u)));
    return;
  }
  for (int64_t i = 4 * q; i < 4 * q + 4 && i < (int64_t)rows * cols; ++i)
    put_split(hi, lo, (size_t)(i / cols) * ld + (i % cols), src[i]);
}

__global__ void __launch_bounds__(256)
prepare_weights_kernel(PrepArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int D = a.D, H = a.H, Z = a.Z;
  switch (blockIdx.y) {
    case 0:
      mirror_quad(a.W3, a.w3h, a.w3l, i, D, H, a.ldh);
      break;
    case 1:
      if (a.W6) {                        // column 2d = W2[:, d], 2d + 1 = W6[:, d]
        for (int64_t e = 4 * i; e < 4 * i + 4 && e < (int64_t)H * D; ++e) {
          const int k = (int)(e / D), d = (int)(e % D);
          put_split(a.w2h, a.w2l, (size_t)k * a.ldd + 2 * d, a.W2[e]);
          put_split(a.w2h, a.w2l, (size_t)k * a.ldd + 2 * d + 1, a.W6[e]);
        }
      } else {
        mirror_quad(a.W2, a.w2h, a.w2l, i, H, D, a.ldd);
      }
      break;
    case 2:
      if (i < (int64_t)2 * Z * H) {
        const int o = (int)(i / H), k = (int)(i % H);
        const float v = o < Z ? a.W4[(size_t)k * Z + o] : a.W5[(size_t)k * Z + (o - Z)];
        a.w45t[i] = v;
        put_split(a.w45h, a.w45l, (size_t)o * a.ldh + k, v);
      }
      break;
    case 3:
      if (i < (int64_t)H * a.ldq) {
        const int k = (int)(i / a.ldq), c = (int)(i % a.ldq), j = c >> 1;
        float v = 0.f;
        if (j < Z) v = (c & 1) ? a.W5[(size_t)k * Z + j] : a.W4[(size_t)k * Z + j];
        put_split(a.whh, a.whl, (size_t)i, v);
      }
      break;
    default:
      mirror_quad(a.W1, a.w1h, a.w1l, i, Z, H, a.ldh);
      break;
  }
}

}  // namespace

// Host arithmetic only (no device is touched): the tiles CTA `cta` of `grid` works on, in order, when the persistent layer
// kernel runs a [rows x N] layer with bn-wide tiles -- the schedule of TileSeq, exported so that a CPU test can check that
// every tile of every shape is visited exactly once (tests/test_golden_cpu.py).
extern "C" int vaeb_diag_tile_schedule(int32_t rows, int32_t N, int32_t bn, int32_t grid, int32_t cta, int32_t cap,
                                       int32_t* tm_out, int32_t* tn_out, int32_t* n_out) {
  if (rows <= 0 || N <= 0 || bn <= 0 || grid <= 0 || cta < 0 || cta >= grid || !tm_out || !tn_out || !n_out) return VAEB_EINVAL;
  const int tiles_m = (rows + BM - 1) / BM, tiles_n = (N + bn - 1) / bn;
  const TileSeq seq(tiles_m, tiles_n, tile_sliver(N, bn, tiles_n), grid, cta);
  int n = 0, tm, tn;
  for (; seq.get(n, tm, tn); ++n) {
    if (n >= cap) return VAEB_EINVAL;
    tm_out[n] = tm; tn_out[n] = tn;
  }
  *n_out = n;
  return VAEB_OK;
}

cudaError_t tc_prepare_weights(cudaStream_t st, int64_t* launches, const float* W3, const float* W2, const float* W4,
                               const float* W5, const float* W1, const TcBuffers& b, float* w45t, int D, int H, int Z,
                               const float* W6) {
  PrepArgs a{W3, W2, W4, W5, W1, W6,
             (__nv_bfloat16*)b.w3h, (__nv_bfloat16*)b.w3l, (__nv_bfloat16*)b.w2h, (__nv_bfloat16*)b.w2l,
             (__nv_bfloat16*)b.w45h, (__nv_bfloat16*)b.w45l, (__nv_bfloat16*)b.whh, (__nv_bfloat16*)b.whl,
             (__nv_bfloat16*)b.w1h, (__nv_bfloat16*)b.w1l, w45t, D, H, Z, b.ldh, b.ldd, b.ldq};
  // x-extent: a quad per thread for the three mirrors, an element per thread for the (small) transposed head copies
  int64_t n = ((int64_t)D * H + 3) / 4;
  if (n < (int64_t)2 * Z * H) n = (int64_t)2 * Z * H;
  if (n < (int64_t)H * b.ldq) n = (int64_t)H * b.ldq;
  prepare_weights_kernel<<<dim3((unsigned)((n + 255) / 256), 5), 256, 0, st>>>(a);
  ++*launches;
  return cudaGetLastError();
}

// ---- host API (tc_layers.h) -------------------------------------------------------------------
cudaError_t tc_wgrad_reduce_all(cudaStream_t st, int64_t* launches, const TcReduceJobs& jobs) {
  return reduce_all_impl(st, launches, jobs);
}
void tc_set_pdl(bool on) { g_pdl = on; }

int tc_act_bn(int rows, int n_min) {
  if (use_persistent(rows, n_min, 256)) return 256;
  return rows >= 1024 ? 128 : 64;
}

cudaError_t tc_split_matrix(cudaStream_t st, int64_t* launches, const float* src, int64_t rows, int cols, int ld_src,
                            void* hi, void* lo, int ld_dst, int ones_col) {
  const int64_t n = rows * ld_dst;
  split_matrix_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, rows, cols, ld_src, (__nv_bfloat16*)hi,
                                                                    (__nv_bfloat16*)lo, ld_dst, ones_col);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t tc_mirror_weights(cudaStream_t st, int64_t* launches, const float* w3, void* w3h, void* w3l, int D, int H,
                              int ldh, const float* w2, void* w2h, void* w2l, int ldd, const float* w6) {
  MirrorSeg s0{w3, (__nv_bfloat16*)w3h, (__nv_bfloat16*)w3l, D, H, ldh, nullptr};
  MirrorSeg s1{w2, (__nv_bfloat16*)w2h, (__nv_bfloat16*)w2l, H, D, ldd, w6};
  const int64_t n = (int64_t)D * H;
  mirror_weights_kernel<<<dim3((unsigned)((n + 255) / 256), 2), 256, 0, st>>>(s0, s1);
  ++*launches;
  return cudaGetLastError();
}

static int make_pair(CUtensorMap* hi, CUtensorMap* lo, const void* bh, const void* bl, uint64_t rows, uint64_t cols,
                     uint64_t stride, uint32_t box_rows) {
  VAEB_TRY(vaeb_make_tmap_bf16(hi, bh, rows, cols, stride, box_rows));
  if (bl) VAEB_TRY(vaeb_make_tmap_bf16(lo, bl, rows, cols, stride, box_rows));
  else *lo = *hi;
  return VAEB_OK;
}

// MN-major operand [k_rows, cols]: 3-D map with `groups` 64-wide column groups per box
static int make_pair_mn(CUtensorMap* hi, CUtensorMap* lo, const void* bh, const void* bl, uint64_t k_rows, uint64_t cols,
                        uint64_t stride, uint32_t groups, uint32_t k_box = 64) {
  VAEB_TRY(vaeb_make_tmap_bf16_mn(hi, bh, k_rows, cols, stride, groups, k_box));
  if (bl) VAEB_TRY(vaeb_make_tmap_bf16_mn(lo, bl, k_rows, cols, stride, groups, k_box));
  else *lo = *hi;
  return VAEB_OK;
}

// bn: UMMA N of the activation layers (tc_act_bn); bn_w: of the weight-gradient GEMMs
int tc_build_maps(TcMaps* m, const TcBuffers& b, int rows_data, int R, int rows, int D, int H, int bn, int Z, int bn_w,
                  int bn_d, int Dd) {
  const uint32_t gd = (uint32_t)(bn_d > 0 ? bn_d : bn) / 64;
  if (Dd <= 0) Dd = D;      // width of the decoder output layer: D, or 2 D for the interleaved Gaussian head
  const uint32_t ga = BM / 64, gb = (uint32_t)bn / 64, gw = (uint32_t)bn_w / 64;
  const uint32_t kw = b.w3l ? BK : 2 * BK;      // contraction rows per box of the weight-gradient operands (stage_k)
  // enc1: A = x mirror [rows_data, D] K-major (the ones column at D stays out of the map), B = W3 [D, H] MN-major
  LayerMaps* e1 = reinterpret_cast<LayerMaps*>(m->enc1);
  VAEB_TRY(make_pair(&e1->a_hi, &e1->a_lo, b.xh, b.xl, rows_data, D, b.ldx, BM));
  VAEB_TRY(make_pair_mn(&e1->b_hi, &e1->b_lo, b.w3h, b.w3l, D, H, b.ldh, gb));
  // dec2: A = h_d mirror [R, H] K-major, B = W2 [H, D] MN-major
  LayerMaps* d2 = reinterpret_cast<LayerMaps*>(m->dec2);
  VAEB_TRY(make_pair(&d2->a_hi, &d2->a_lo, b.hdh, b.hdl, R, H, b.ldh, BM));
  VAEB_TRY(make_pair_mn(&d2->b_hi, &d2->b_lo, b.w2h, b.w2l, H, Dd, b.ldd, gd));
  // dgrad h_d: A = da2 mirror [R, D] K-major, B = W2 [H, D] K-major (N = H rows)
  LayerMaps* dg = reinterpret_cast<LayerMaps*>(m->dgrad);
  VAEB_TRY(make_pair(&dg->a_hi, &dg->a_lo, b.da2h, b.da2l, R, Dd, b.ldd, BM));
  VAEB_TRY(make_pair(&dg->b_hi, &dg->b_lo, b.w2h, b.w2l, H, Dd, b.ldd, (uint32_t)bn));
  // wgrad W2: A = h_d mirror [R, H+1] MN-major (ones column -> bias row), B = da2 mirror [R, D] MN-major
  LayerMaps* w2 = reinterpret_cast<LayerMaps*>(m->wgrad2);
  VAEB_TRY(make_pair_mn(&w2->a_hi, &w2->a_lo, b.hdh, b.hdl, R, H + 1, b.ldh, ga, kw));
  VAEB_TRY(make_pair_mn(&w2->b_hi, &w2->b_lo, b.da2h, b.da2l, R, Dd, b.ldd, gw, kw));
  // wgrad W3: A = x mirror [rows_data, D+1] MN-major, B = da3 mirror [rows, H] MN-major
  LayerMaps* w3 = reinterpret_cast<LayerMaps*>(m->wgrad3);
  VAEB_TRY(make_pair_mn(&w3->a_hi, &w3->a_lo, b.xh, b.xl, rows_data, D + 1, b.ldx, ga, kw));
  VAEB_TRY(make_pair_mn(&w3->b_hi, &w3->b_lo, b.da3h, b.da3l, rows, H, b.ldh, gw, kw));
  if (b.heh) {
    // wgrad W1: A = z mirror [R, Z+1] MN-major (ones column -> gb1), B = da1 mirror [R, H] MN-major
    LayerMaps* w1 = reinterpret_cast<LayerMaps*>(m->wgrad1);
    VAEB_TRY(make_pair_mn(&w1->a_hi, &w1->a_lo, b.zh, b.zl, R, Z + 1, b.ldz, ga, kw));
    VAEB_TRY(make_pair_mn(&w1->b_hi, &w1->b_lo, b.d1h, b.d1l, R, H, b.ldh, gw, kw));
    // wgrad W4|W5: A = h_e mirror [rows, H+1] MN-major (ones column -> gb4|gb5), B = [dmu|dls] mirror [rows, 2Z] with
    // boxes as wide as the other weight-gradient jobs' (columns >= 2Z: zeros)
    LayerMaps* w45w = reinterpret_cast<LayerMaps*>(m->wgrad45w);
    VAEB_TRY(make_pair_mn(&w45w->a_hi, &w45w->a_lo, b.heh, b.hel, rows, H + 1, b.ldh, ga, kw));
    VAEB_TRY(make_pair_mn(&w45w->b_hi, &w45w->b_lo, b.ddh, b.ddl, rows, 2 * Z, b.ldq, gw, kw));
    // enc2: A = h_e mirror [rows, H] K-major, B = interleaved heads mirror [H, 2Z] MN-major
    LayerMaps* e2 = reinterpret_cast<LayerMaps*>(m->enc2);
    VAEB_TRY(make_pair(&e2->a_hi, &e2->a_lo, b.heh, b.hel, rows, H, b.ldh, BM));
    VAEB_TRY(make_pair_mn(&e2->b_hi, &e2->b_lo, b.whh, b.whl, H, 2 * Z, b.ldq, 1));
    // dec1: A = z mirror [R, Z] K-major (the ones column at Z stays out of the map), B = W1 mirror [Z, H] MN-major
    LayerMaps* d1 = reinterpret_cast<LayerMaps*>(m->dec1);
    VAEB_TRY(make_pair(&d1->a_hi, &d1->a_lo, b.zh, b.zl, R, Z, b.ldz, BM));
    VAEB_TRY(make_pair_mn(&d1->b_hi, &d1->b_lo, b.w1h, b.w1l, Z, H, b.ldh, gb));
    // dz: A = da1 mirror [R, H] K-major, B = W1 mirror [Z, H] K-major (N = Z rows)
    LayerMaps* dzm = reinterpret_cast<LayerMaps*>(m->dz);
    VAEB_TRY(make_pair(&dzm->a_hi, &dzm->a_lo, b.d1h, b.d1l, R, H, b.ldh, BM));
    VAEB_TRY(make_pair(&dzm->b_hi, &dzm->b_lo, b.w1h, b.w1l, Z, H, b.ldh, 64));
    // dgrad h_e: A = [dmu|dls] mirror [rows, 2Z] K-major, B = [W4^T;W5^T] mirror [2Z, H] MN-major
    LayerMaps* dh = reinterpret_cast<LayerMaps*>(m->dhe);
    VAEB_TRY(make_pair(&dh->a_hi, &dh->a_lo, b.ddh, b.ddl, rows, 2 * Z, b.ldq, BM));
    VAEB_TRY(make_pair_mn(&dh->b_hi, &dh->b_lo, b.w45h, b.w45l, 2 * Z, H, b.ldh, gb));
  }
  return VAEB_OK;
}

static_assert(sizeof(LayerMaps) == TC_LAYER_MAPS_BYTES, "TcMaps storage size");

cudaError_t tc_enc1(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int D, int H,
                    int x_row_off, const float* b3, float* h_e, void* he_hi, void* he_lo, int ldm) {
  EpiTanh epi{b3, h_e, H, (__nv_bfloat16*)he_hi, (__nv_bfloat16*)he_lo, ldm, (ns == 1 && h_e == nullptr) ? 1 : 0};
  ++*launches;
  return dispatch_layer<false, true>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.enc1), epi, rows, H, D,
                                     x_row_off);
}

cudaError_t tc_dec2_bernoulli(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                              const float* b2, const float* x, int x_div, int x_mod, float scale, void* da_hi,
                              void* da_lo, int ldda, float* partial, int* n_tiles, const void* xm_hi, const void* xm_lo,
                              int ldxm, int xm_off) {
  EpiBernoulliTc epi{b2, x, D, x_div, x_mod, scale, (__nv_bfloat16*)da_hi, (__nv_bfloat16*)da_lo, ldda, partial,
                     (const __nv_bfloat16*)xm_hi, (const __nv_bfloat16*)xm_lo, ldxm, xm_off, 0.f};
  *n_tiles = ((D + bn - 1) / bn) * (EPI_WARPS / 4);
  ++*launches;
  return dispatch_layer<false, true>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.dec2), epi, R, D, H, 0);
}

cudaError_t tc_dec2_gaussian(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                             const float* b2, const float* b6, const float* x, int x_div, int x_mod, float scale, void* da_hi,
                             void* da_lo, int ldda, float* partial, int* n_tiles, const void* xm_hi, const void* xm_lo,
                             int ldxm, int xm_off) {
  EpiGaussianTc epi{b2, b6, x, D, x_div, x_mod, scale, (__nv_bfloat16*)da_hi, (__nv_bfloat16*)da_lo, ldda, partial,
                    (const __nv_bfloat16*)xm_hi, (const __nv_bfloat16*)xm_lo, ldxm, xm_off, 0.f};
  *n_tiles = ((2 * D + bn - 1) / bn) * (EPI_WARPS / 4);
  ++*launches;
  return dispatch_layer<false, true>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.dec2), epi, R, 2 * D, H, 0);
}

cudaError_t tc_dgrad_hd(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int D, int H,
                        const float* h_d, float* da1, void* d1_hi, void* d1_lo, int ldm, const void* h_hi,
                        const void* h_lo) {
  EpiDgradTanh epi{h_d, da1, H, (__nv_bfloat16*)d1_hi, (__nv_bfloat16*)d1_lo, ldm,
                   (const __nv_bfloat16*)h_hi, (const __nv_bfloat16*)h_lo};
  ++*launches;
  return dispatch_layer<false, false>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.dgrad), epi, R, H, D, 0);
}

cudaError_t tc_enc2_heads(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int rows, int H, int Z, int la,
                          const float* b4, const float* b5, const EpsSource& src, float* mu, float* ls, float* eps,
                          float* z, void* z_hi, void* z_lo, int ldz, float* aux_part, int* n_aux) {
  EpiHeads epi{b4, b5, Z, la, src, mu, ls, eps, z, (__nv_bfloat16*)z_hi, (__nv_bfloat16*)z_lo, ldz, aux_part, 0.f};
  *n_aux = ((2 * Z + 63) / 64) * (EPI_WARPS / 4);
  ++*launches;
  return dispatch_layer<false, true>(st, ns, 64, *reinterpret_cast<const LayerMaps*>(m.enc2), epi, rows, 2 * Z, H, 0);
}

cudaError_t tc_dec1(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int Z, int H,
                    const float* b1, float* h_d, void* hd_hi, void* hd_lo, int ldm) {
  EpiTanh epi{b1, h_d, H, (__nv_bfloat16*)hd_hi, (__nv_bfloat16*)hd_lo, ldm, (ns == 1 && h_d == nullptr) ? 1 : 0};
  ++*launches;
  return dispatch_layer<false, true>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.dec1), epi, R, H, Z, 0);
}

cudaError_t tc_dz_dprep(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int R, int H, int Z, int la, float w_aux,
                        const float* z, const float* eps, const float* mu, const float* ls, float* dmu, float* dls,
                        void* dd_hi, void* dd_lo, int ldq) {
  EpiDzPrep epi{z, eps, mu, ls, Z, la, w_aux, dmu, dls, (__nv_bfloat16*)dd_hi, (__nv_bfloat16*)dd_lo, ldq};
  ++*launches;
  return dispatch_layer<false, false>(st, ns, 64, *reinterpret_cast<const LayerMaps*>(m.dz), epi, R, Z, H, 0);
}

cudaError_t tc_dgrad_he(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int Z, int H,
                        const float* h_e, float* da3, void* da3_hi, void* da3_lo, int ldm, const void* h_hi,
                        const void* h_lo) {
  EpiDgradTanh epi{h_e, da3, H, (__nv_bfloat16*)da3_hi, (__nv_bfloat16*)da3_lo, ldm,
                   (const __nv_bfloat16*)h_hi, (const __nv_bfloat16*)h_lo};
  ++*launches;
  return dispatch_layer<false, true>(st, ns, bn, *reinterpret_cast<const LayerMaps*>(m.dhe), epi, rows, H, 2 * Z, 0);
}

size_t tc_wgrad_scratch_elems(int D, int H) {
  (void)D; (void)H;
  return (size_t)148 * BM * 128;          // splits * Mo * No <= (148 / tiles) * tiles * 128 * 128
}

// gW6 != nullptr (Gaussian decoder): D is the width of the interleaved head (2 x pixels); the reduction de-interleaves
cudaError_t tc_wgrad2(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int H, int D,
                      float* gW2, float* gb2, float* scratch, float* gW6, float* gb6) {
  return tc_wgrad_generic(st, launches, *reinterpret_cast<const LayerMaps*>(m.wgrad2), ns, bn, R, H, D, 0, gW2, gb2,
                          scratch, gW6, gb6);
}

cudaError_t tc_wgrad3(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int rows, int D, int H,
                      int x_row_off, float* gW3, float* gb3, float* scratch) {
  return tc_wgrad_generic(st, launches, *reinterpret_cast<const LayerMaps*>(m.wgrad3), ns, bn, rows, D, H, x_row_off, gW3,
                          gb3, scratch);
}

// ---- every weight gradient of the step in one launch ------------------------------------------------------------
// (measured faster than four launches at every size: 16384 rows bf16x3 354.7 -> 339.6 us per update, bf16 222 -> 203)

cudaError_t tc_wgrad_all(cudaStream_t st, int64_t* launches, const TcMaps& m, int ns, int bn, int R, int rows, int D, int H,
                         int Z, int x_row_off, float* gW2, float* gb2, float* gW1, float* gb1, float* gW4, float* gb4,
                         float* gW5, float* gb5, float* gW3, float* gb3, float* scratch, size_t region, TcReduceJobs* jobs,
                         int n_sm, float* gW6, float* gb6) {
  WgradAllArgs a;
  const int Dd = gW6 ? 2 * D : D;      // Gaussian decoder: the W2 job is the interleaved head [W2|W6]'
  const int sk = ns == 1 ? 2 * BK : BK;
  auto fill = [&](int j, const unsigned char* maps, int Hreal, int N, int K, int off, float* scr, int splits) {
    WgradJob& J = a.job[j];
    J.maps = *reinterpret_cast<const LayerMaps*>(maps);
    J.M = Hreal + 1; J.N = N; J.K = K; J.a_row_off = off;
    J.tiles_n = (N + bn - 1) / bn; J.tiles_m = (Hreal + 1 + BM - 1) / BM;
    const int nst = (K + sk - 1) / sk;
    J.splits = splits < 1 ? 1 : (splits > nst ? nst : splits);
    J.epi = EpiWgradTc{nullptr, nullptr, Hreal, N, scr, (size_t)(Hreal + 1) * N};      // always through scratch
  };
  // one wave: the two wide gradients (28 tiles each at 128 x 128) share the SMs the thin ones leave
  const int thin_splits = 4;
  const int wide_tiles = ((Dd + bn - 1) / bn) * ((H + 1 + BM - 1) / BM) + ((H + bn - 1) / bn) * ((D + 1 + BM - 1) / BM);
  const int thin_tiles = ((H + bn - 1) / bn) * ((Z + 1 + BM - 1) / BM) + ((2 * Z + bn - 1) / bn) * ((H + 1 + BM - 1) / BM);
  int wide_splits = (n_sm - thin_tiles * thin_splits) / (wide_tiles > 0 ? wide_tiles : 1);
  if (wide_splits < 1) wide_splits = 1;
  fill(0, m.wgrad2, H, Dd, R, 0, scratch, wide_splits);
  fill(1, m.wgrad1, Z, H, R, 0, scratch + region, thin_splits);
  fill(2, m.wgrad45w, H, 2 * Z, rows, 0, scratch + 2 * region, thin_splits);
  fill(3, m.wgrad3, D, H, rows, x_row_off, scratch + 3 * region, wide_splits);
  a.n_jobs = 4;
  int blocks = 0;
  for (int j = 0; j < 4; ++j) { a.job[j].first_block = blocks; blocks += a.job[j].tiles_n * a.job[j].tiles_m * a.job[j].splits; }
  const size_t s2 = (size_t)(H + 1) * Dd, s1 = (size_t)(Z + 1) * H, s45 = (size_t)(H + 1) * 2 * Z, s3 = (size_t)(D + 1) * H;
  const TcReduceJob j2 = gW6 ? TcReduceJob{scratch, a.job[0].splits, s2, (H + 1) * Dd, 0, gW2, gb2, gW6, gb6, 2, H, D}
                             : TcReduceJob{scratch, a.job[0].splits, s2, H * D, D, gW2, gb2, nullptr, nullptr, 0, 0, 0};
  if (!add_reduce_job(jobs, j2) ||
      !add_reduce_job(jobs, TcReduceJob{scratch + region, a.job[1].splits, s1, Z * H, H, gW1, gb1, nullptr, nullptr, 0, 0, 0}) ||
      !add_reduce_job(jobs, TcReduceJob{scratch + 2 * region, a.job[2].splits, s45, (H + 1) * 2 * Z, 0, gW4, gb4, gW5, gb5, 1, H, Z}) ||
      !add_reduce_job(jobs, TcReduceJob{scratch + 3 * region, a.job[3].splits, s3, D * H, H, gW3, gb3, nullptr, nullptr, 0, 0, 0}))
    return cudaErrorInvalidValue;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  ++*launches;
  auto go = [&](auto kfn, int smem) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    cfg.dynamicSmemBytes = smem;
    return cudaLaunchKernelEx(&cfg, kfn, a);
  };
  if (bn == 128) {
    if (ns == 2) return go(tc_wgrad_all_kernel<128, 2>, LayerSmem<128, 2, true, stage_k<true, true, 2>()>::TOTAL);
    return go(tc_wgrad_all_kernel<128, 1>, LayerSmem<128, 1, true, stage_k<true, true, 1>()>::TOTAL);
  }
  if (ns == 2) return go(tc_wgrad_all_kernel<64, 2>, LayerSmem<64, 2, true, stage_k<true, true, 2>()>::TOTAL);
  return go(tc_wgrad_all_kernel<64, 1>, LayerSmem<64, 1, true, stage_k<true, true, 1>()>::TOTAL);
}
