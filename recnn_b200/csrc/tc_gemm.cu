// Host side of the tcgen05 3xTF32 GEMM: tensor-map construction, launch
// configuration, and the generic C-ABI entry points recnn_gemm_tf32x3 / recnn_gemm_fp32.
#include "tc_gemm.cuh"

#include <stdlib.h>
#include <string.h>

#include <mutex>

namespace recnn {
namespace tc {

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_tmap(CUtensorMap* out, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
              int box_rows, int swizzle_bytes) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return RECNN_E_CUDA;
  }
  RECNN_REQUIRE(reinterpret_cast<uintptr_t>(base) % 16 == 0, "TMA base must be 16-byte aligned");
  RECNN_REQUIRE(ld % 4 == 0 && ld >= cols, "TMA row pitch must be a multiple of 4 floats");
  RECNN_REQUIRE(box_cols * 4 <= (swizzle_bytes == 1032 ? 128 : swizzle_bytes) && box_rows <= 256, "TMA box");
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 1032 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
                               : swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                               : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                     : CU_TENSOR_MAP_SWIZZLE_32B;
  const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld box=%dx%d", (int)r, (long long)rows,
              (long long)cols, (long long)ld, box_cols, box_rows);
    return RECNN_E_CUDA;
  }
  return RECNN_OK;
}

int split_plan(int K_total_blocks, int splits_req, int* k_chunk, int bk) {
  if (splits_req < 1) splits_req = 1;
  const int kb_per = (int)ceil_div(K_total_blocks, splits_req);
  *k_chunk = kb_per * bk;
  return (int)ceil_div(K_total_blocks, kb_per);
}

template <class C, int EPI>
static int launch_cfg(const Operand& A0, const Operand& A1, const Operand& B, const Problem& p_in, int splits,
                      const Epilogue& epi, cudaStream_t st) {
  Problem p = p_in;
  static bool attr_set = false;
  if (!attr_set) {
    RECNN_CHECK_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<C, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          C::SMEM_BYTES));
    attr_set = true;
  }
  const int nkb = (int)(ceil_div(p.K0, C::BK) + ceil_div(p.K1, C::BK));
  splits = split_plan(nkb, splits, &p.k_chunk, C::BK);
  CUtensorMap ma0, ma1, mb;
  // K-major operand: tensor [rows = M|N, cols = K], box {BK, tile rows}; MN-major: tensor [rows = K, cols = M|N], box {32, BK}
  if (!C::A_MN) {
    RECNN_PROPAGATE(make_tmap(&ma0, A0.ptr, p.M, p.K0, A0.ld, C::BK, C::BM, C::K_SWZ));
    if (p.K1 > 0) RECNN_PROPAGATE(make_tmap(&ma1, A1.ptr, p.M, p.K1, A1.ld, C::BK, C::BM, C::K_SWZ));
    else ma1 = ma0;
  } else {
    RECNN_REQUIRE(p.K1 == 0, "MN-major A cannot be a K-concat");
    RECNN_PROPAGATE(make_tmap(&ma0, A0.ptr, p.K0, p.M, A0.ld, 32, C::BK, 1032));
    ma1 = ma0;
  }
  if (!C::B_MN) RECNN_PROPAGATE(make_tmap(&mb, B.ptr, B.rows, B.cols, B.ld, C::BK, C::BN, C::K_SWZ));
  else RECNN_PROPAGATE(make_tmap(&mb, B.ptr, B.rows, B.cols, B.ld, 32, C::BK, 1032));
  dim3 grid((unsigned)ceil_div(p.N, C::BN), (unsigned)ceil_div(p.M, C::BM), (unsigned)splits);
  static const bool debug = getenv("RECNN_B200_DEBUG") != nullptr;
  if (debug)
    fprintf(stderr, "[tc_gemm] BN=%d A_MN=%d B_MN=%d EPI=%d M=%d N=%d K0=%d K1=%d k_chunk=%d bk1=%d nout=%d bn_off=%d "
            "grid=%u,%u,%u a0=%p ld=%lld a1=%p ld=%lld b=%p ld=%lld rows=%lld cols=%lld out=%p ldo=%lld\n",
            C::BN, (int)C::A_MN, (int)C::B_MN, EPI, p.M, p.N, p.K0, p.K1, p.k_chunk, p.b_k1_offset, p.n_out_offset,
            p.b_n_offset, grid.x, grid.y, grid.z, (const void*)A0.ptr, A0.ld, (const void*)A1.ptr, A1.ld,
            (const void*)B.ptr, B.ld, B.rows, B.cols, (void*)epi.out, epi.ldo);
  // programmatic stream serialization: this kernel's prologue may overlap the tail of its predecessor
  // (the kernel parks at griddepcontrol.wait before it touches global memory)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(C::THREADS, 1, 1);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  RECNN_CHECK_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<C, EPI>, ma0, ma1, mb, p, epi));
  RECNN_CHECK_LAUNCH("tc_gemm_kernel");
  if (debug) {
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      set_error("tc_gemm_kernel execution failed: %s", cudaGetErrorString(e));
      fprintf(stderr, "[tc_gemm] FAILED: %s\n", cudaGetErrorString(e));
      return RECNN_E_CUDA;
    }
  }
  return splits;
}

template <bool A_MN, bool B_MN, int EPI>
int launch(const Operand& A0, const Operand& A1, const Operand& B, const Problem& p, int splits, int bn,
           const Epilogue& epi, cudaStream_t st) {
  // stages chosen to fill ~190 KB of shared memory: stage = 16 KB (raw A) + 2 * BN/8 KB (B hi | B lo)
  if (bn >= 128) return launch_cfg<Cfg<128, 4, A_MN, B_MN>, EPI>(A0, A1, B, p, splits, epi, st);
  return launch_cfg<Cfg<64, 6, A_MN, B_MN>, EPI>(A0, A1, B, p, splits, epi, st);
}

// explicit instantiations used by step.cu / the generic entry points
#define RECNN_TC_INST(A_MN, B_MN, EPI) \
  template int launch<A_MN, B_MN, EPI>(const Operand&, const Operand&, const Operand&, const Problem&, int, int, \
                                       const Epilogue&, cudaStream_t);
RECNN_TC_INST(false, false, EPI_HIDDEN)
RECNN_TC_INST(false, false, EPI_LINEAR)
RECNN_TC_INST(false, false, EPI_STORE)
RECNN_TC_INST(false, true, EPI_STORE)
RECNN_TC_INST(false, true, EPI_GATE)
RECNN_TC_INST(true, true, EPI_STORE)
RECNN_TC_INST(true, true, EPI_PARTIAL)
RECNN_TC_INST(false, false, EPI_PARTIAL)
RECNN_TC_INST(true, false, EPI_STORE)
RECNN_TC_INST(false, false, EPI_DLOGITS)
RECNN_TC_INST(false, true, EPI_ACCUM)

}  // namespace tc
}  // namespace recnn

using namespace recnn;

// C[M,N] (row pitch ldc) = A . B^T in 3xTF32 on the tensor cores.
//   a_mn = 0: A is [M,K] row-major (pitch lda)   a_mn = 1: A is [K,M] row-major
//   b_mn = 0: B is [N,K] row-major (pitch ldb)   b_mn = 1: B is [K,N] row-major
// All pitches and base addresses must be multiples of 4 floats / 16 bytes (TMA).
extern "C" int recnn_gemm_tf32x3(int M, int N, int K, const float* A, int64_t lda, int a_mn, const float* B,
                                 int64_t ldb, int b_mn, float* C, int64_t ldc, int tile_n, void* stream) {
  RECNN_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "null pointer / sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Epilogue e;
  memset(&e, 0, sizeof(e));
  e.out = C;
  e.ldo = ldc;
  tc::Operand a0 = {A, lda, 0, 0}, a1 = {nullptr, 0, 0, 0};
  tc::Operand b = {B, ldb, b_mn ? K : N, b_mn ? N : K};
  tc::Problem p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K0 = K; p.b_k1_offset = K;
  if (tile_n <= 0) tile_n = N > 64 ? 128 : 64;
  int r;
  if (!a_mn && !b_mn) r = tc::launch<false, false, EPI_STORE>(a0, a1, b, p, 1, tile_n, e, st);
  else if (!a_mn && b_mn) r = tc::launch<false, true, EPI_STORE>(a0, a1, b, p, 1, tile_n, e, st);
  else if (a_mn && b_mn) r = tc::launch<true, true, EPI_STORE>(a0, a1, b, p, 1, tile_n, e, st);
  else r = tc::launch<true, false, EPI_STORE>(a0, a1, b, p, 1, tile_n, e, st);
  return r < 0 ? r : RECNN_OK;
}

// Same contract on the fp32 CUDA cores (exact fp32 FMA chain) -- the arbitrary-shape path.
extern "C" int recnn_gemm_fp32(int M, int N, int K, const float* A, int64_t lda, int a_mn, const float* B,
                               int64_t ldb, int b_mn, float* C, int64_t ldc, void* stream) {
  RECNN_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "null pointer / sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Epilogue e;
  memset(&e, 0, sizeof(e));
  e.out = C;
  e.ldo = ldc;
  const MatView a = mat(A, lda), b = mat(B, ldb);
  if (!a_mn && !b_mn) return launch_gemm_simt<true, true, EPI_STORE>(a, b, M, N, K, 1, e, st);
  if (!a_mn && b_mn) return launch_gemm_simt<true, false, EPI_STORE>(a, b, M, N, K, 1, e, st);
  if (a_mn && b_mn) return launch_gemm_simt<false, false, EPI_STORE>(a, b, M, N, K, 1, e, st);
  return launch_gemm_simt<false, true, EPI_STORE>(a, b, M, N, K, 1, e, st);
}
