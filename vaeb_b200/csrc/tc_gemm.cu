// Generic tcgen05 GEMM: C[M,N] (fp32) = A . B with bf16 operands staged by TMA (128B swizzle),
// fp32 accumulation in TMEM, tcgen05.ld epilogue.  Either operand may be K-major (contraction
// index contiguous in memory) or MN-major; the five dense contractions of an AEVB step need all
// four combinations (SURVEY.md 2b):
//   forward  x.W      : A K-major  [M,K],  B MN-major [K,N]
//   dgrad    d.W^T    : A K-major  [M,K],  B K-major  [N,K]
//   wgrad    h^T.d    : A MN-major [K,M],  B MN-major [K,N]     (contraction over the batch)
// Warp roles (256 threads): w0 TMA producer, w1 MMA issuer, w2 TMEM allocator, w4-7 epilogue.
#include <cstring>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

constexpr int BM = 128;     // UMMA M
constexpr int BK = 64;      // one 128-byte swizzle span of bf16
constexpr int STAGES = 4;

template <int BN>
struct GemmSmem {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(256, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, float* __restrict__ C,
               int M, int N, int K, int ldc) {
  using S = GemmSmem<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int nkb = (K + BK - 1) / BK;
  constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&tmA);
    tc::tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&empty[s], 1); }
    tc::mbar_init(tmem_full, 1);
    tc::fence_barrier_init();
  }
  if (warp == 2) tc::tmem_alloc(tmem_slot, TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES;
      const uint32_t ph = (kb / STAGES) & 1;
      tc::mbar_wait(&empty[s], ph ^ 1);
      uint8_t* a = smem + s * S::STAGE_BYTES;
      uint8_t* b = a + S::A_BYTES;
      tc::mbar_expect_tx(&full[s], S::STAGE_BYTES);
      if (A_MN) {
        for (int g = 0; g < BM / 64; ++g) tc::tma_load_2d(a + g * 8192, &tmA, &full[s], m0 + g * 64, kb * BK);
      } else {
        tc::tma_load_2d(a, &tmA, &full[s], kb * BK, m0);
      }
      if (B_MN) {
        for (int g = 0; g < BN / 64; ++g) tc::tma_load_2d(b + g * 8192, &tmB, &full[s], n0 + g * 64, kb * BK);
      } else {
        tc::tma_load_2d(b, &tmB, &full[s], kb * BK, n0);
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer =====
    constexpr uint32_t idesc = tc::make_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % STAGES;
      const uint32_t ph = (kb / STAGES) & 1;
      tc::mbar_wait(&full[s], ph);
      tc::tc_fence_after();
      const uint32_t a = tc::smem_u32(smem + s * S::STAGE_BYTES);
      const uint32_t b = a + S::A_BYTES;
#pragma unroll
      for (int k = 0; k < BK / 16; ++k) {
        const uint64_t da = A_MN ? tc::desc_mnmajor(a, k, 8192u) : tc::desc_kmajor(a, k);
        const uint64_t db = B_MN ? tc::desc_mnmajor(b, k, 8192u) : tc::desc_kmajor(b, k);
        tc::umma_bf16(tmem_base, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
      }
      tc::umma_commit(&empty[s]);     // frees the smem slot once these MMAs have read it
    }
    tc::umma_commit(tmem_full);       // accumulator complete
  } else if (warp >= 4) {
    // ===== epilogue: TMEM -> registers -> global =====
    tc::mbar_wait(tmem_full, 0);
    tc::tc_fence_after();
    const int q = warp & 3;                       // TMEM lane quarter of this warp
    const int row = m0 + q * 32 + lane;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      float v[32];
      tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
      tc::tmem_ld_wait();
      if (row < M) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (n0 + c + j < N) C[(size_t)row * ldc + n0 + c + j] = v[j];
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, TMEM_COLS);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return nullptr;
  fn = (EncodeTiledFn)p;
  return fn;
}

uint16_t f32_to_bf16(float f) {   // round to nearest even
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

template <int BN, bool A_MN, bool B_MN>
int launch_tc_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, float* C, int M, int N, int K, int ldc,
                   cudaStream_t st) {
  using S = GemmSmem<BN>;
  auto kfn = tc_gemm_kernel<BN, A_MN, B_MN>;
  VAEB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
  dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM);
  kfn<<<grid, 256, S::TOTAL, st>>>(tmA, tmB, C, M, N, K, ldc);
  VAEB_CUDA(cudaGetLastError());
  return VAEB_OK;
}

}  // namespace

int vaeb_make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                        uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { vaeb_set_error("cuTensorMapEncodeTiled not available from the driver"); return VAEB_ECUDA; }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {row_stride_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  if ((row_stride_elems * 2) % 16 != 0 || ((uintptr_t)base & 15) != 0) {
    vaeb_set_error("tensor map: base and row stride must be 16-byte aligned");
    return VAEB_EINVAL;
  }
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vaeb_set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return VAEB_ECUDA;
  }
  return VAEB_OK;
}

int vaeb_make_tmap_bf16_mn(CUtensorMap* out, const void* base, uint64_t k_rows, uint64_t cols, uint64_t row_stride_elems,
                           uint32_t groups, uint32_t k_box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { vaeb_set_error("cuTensorMapEncodeTiled not available from the driver"); return VAEB_ECUDA; }
  const uint64_t n_groups = (cols + 63) / 64;
  if (row_stride_elems % 64 != 0 || n_groups * 64 > row_stride_elems || ((uintptr_t)base & 127) != 0 || groups < 1 ||
      groups > 4) {
    vaeb_set_error("MN-major tensor map: the row stride must be a multiple of 64 elements covering every column group");
    return VAEB_EINVAL;
  }
  cuuint64_t gdim[3] = {64, k_rows, n_groups};
  cuuint64_t gstr[2] = {row_stride_elems * 2, 128};
  cuuint32_t box[3] = {64, k_box, groups};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vaeb_set_error("cuTensorMapEncodeTiled (3-D) failed with CUresult " + std::to_string((int)r));
    return VAEB_ECUDA;
  }
  return VAEB_OK;
}

extern "C" int vaeb_tc_gemm_test(int32_t device, int32_t M, int32_t N, int32_t K, int32_t a_mn_major,
                                 int32_t b_mn_major, int32_t block_n, const float* A, const float* B, float* C) {
  // A is the logical [M,K] matrix, B the logical [K,N] matrix (row-major fp32 on the host); they
  // are rounded to bf16 and laid out in the requested majors before upload.
  VAEB_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "null argument");
  VAEB_REQUIRE(K % 8 == 0 && M % 8 == 0 && N % 8 == 0, "M, N, K must be multiples of 8 (16-byte TMA strides)");
  VAEB_REQUIRE(block_n == 64 || block_n == 128 || block_n == 256 || (block_n == 32 && !b_mn_major),
               "block_n must be 64/128/256 (32 only with K-major B)");
  VAEB_CUDA(cudaSetDevice(device));
  std::vector<uint16_t> ha((size_t)M * K), hb((size_t)N * K);
  for (int m = 0; m < M; ++m)
    for (int k = 0; k < K; ++k) {
      const uint16_t v = f32_to_bf16(A[(size_t)m * K + k]);
      if (a_mn_major) ha[(size_t)k * M + m] = v; else ha[(size_t)m * K + k] = v;
    }
  for (int k = 0; k < K; ++k)
    for (int n = 0; n < N; ++n) {
      const uint16_t v = f32_to_bf16(B[(size_t)k * N + n]);
      if (b_mn_major) hb[(size_t)k * N + n] = v; else hb[(size_t)n * K + k] = v;
    }
  void *dA = nullptr, *dB = nullptr;
  float* dC = nullptr;
  VAEB_CUDA(cudaMalloc(&dA, ha.size() * 2));
  VAEB_CUDA(cudaMalloc(&dB, hb.size() * 2));
  VAEB_CUDA(cudaMalloc((void**)&dC, (size_t)M * N * sizeof(float)));
  VAEB_CUDA(cudaMemcpy(dA, ha.data(), ha.size() * 2, cudaMemcpyHostToDevice));
  VAEB_CUDA(cudaMemcpy(dB, hb.data(), hb.size() * 2, cudaMemcpyHostToDevice));
  VAEB_CUDA(cudaMemset(dC, 0xFF, (size_t)M * N * sizeof(float)));
  CUtensorMap tmA, tmB;
  // K-major: matrix [rows=M|N, cols=K], box [BM|BN x 64].  MN-major: matrix [rows=K, cols=M|N], box [64 x 64].
  if (a_mn_major) VAEB_TRY(vaeb_make_tmap_bf16(&tmA, dA, K, M, M, 64));
  else VAEB_TRY(vaeb_make_tmap_bf16(&tmA, dA, M, K, K, BM));
  if (b_mn_major) VAEB_TRY(vaeb_make_tmap_bf16(&tmB, dB, K, N, N, 64));
  else VAEB_TRY(vaeb_make_tmap_bf16(&tmB, dB, N, K, K, (uint32_t)block_n));
  int rc = VAEB_EINVAL;
#define DISPATCH(BN_)                                                                                          \
  if (block_n == BN_) {                                                                                        \
    if (a_mn_major && b_mn_major) rc = launch_tc_gemm<BN_, true, true>(tmA, tmB, dC, M, N, K, N, 0);            \
    else if (a_mn_major) rc = launch_tc_gemm<BN_, true, false>(tmA, tmB, dC, M, N, K, N, 0);                    \
    else if (b_mn_major) rc = launch_tc_gemm<BN_, false, true>(tmA, tmB, dC, M, N, K, N, 0);                    \
    else rc = launch_tc_gemm<BN_, false, false>(tmA, tmB, dC, M, N, K, N, 0);                                   \
  }
  DISPATCH(64) DISPATCH(128) DISPATCH(256)
  if (block_n == 32) rc = launch_tc_gemm<32, false, false>(tmA, tmB, dC, M, N, K, N, 0);
#undef DISPATCH
  if (rc == VAEB_OK) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { vaeb_set_error(std::string("tc_gemm kernel: ") + cudaGetErrorString(e)); rc = VAEB_ECUDA; }
  }
  if (rc == VAEB_OK) {
    cudaError_t e = cudaMemcpy(C, dC, (size_t)M * N * sizeof(float), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { vaeb_set_error(std::string("tc_gemm copy: ") + cudaGetErrorString(e)); rc = VAEB_ECUDA; }
  }
  cudaFree(dA); cudaFree(dB); cudaFree(dC);
  return rc;
}
