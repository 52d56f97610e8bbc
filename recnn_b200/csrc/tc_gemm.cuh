// tcgen05 (5th-gen tensor core) GEMM with fp32-grade accuracy: error-compensated
// 3xTF32, operands staged by TMA, chunked accumulation in TMEM, sm_100a only.
//
//   C[m,n] = sum_k A(m,k) * B(n,k)            (+ fused epilogue)
//
// Why 3xTF32: the parity bar is the reference's fp32 CPU result to 1e-5
// (BASELINE.json north_star); one TF32 pass has a 10-bit mantissa (~1e-3).  Each
// fp32 operand x is split into  hi = rna_tf32(x)  and  lo = rna_tf32(x - hi)  (the
// subtraction is exact).  Three MMAs per 8-wide k-slice,  lo_a*hi_b + hi_a*lo_b + hi_a*hi_b;
// the dropped lo*lo term is < 2^-22 relative.
//
// Why chunked accumulation: the tensor core's fp32 accumulate TRUNCATES (measured: each
// tcgen05.mma accumulate loses ~3.5e-8 of the running sum; unchunked, all-positive operands
// are off by -2.8e-5 at K=1290).  So
//   * the big hi*hi products of only CH k-blocks (K = 64, 8 accumulates) are summed in a TMEM
//     chunk accumulator; after each chunk the worker warps pull it out with tcgen05.ld and add
//     it to a register-resident running sum with round-to-nearest FADDs, while the tensor
//     core fills the other chunk buffer;
//   * the two small cross terms go to a separate TMEM accumulator D_lo that lives for the whole
//     tile (its magnitude is 2^-11 of the result, so its truncation error is irrelevant) and is
//     added once at the end.
// hi is rounded to nearest (not truncated), so |lo| <= 2^-12 |x| is symmetric and the dropped
// lo*lo term is unbiased.  Measured result: ~3e-7 worst-case systematic error, independent of K.
//
// Warp roles (one 128 x BN output tile per CTA; BN = 128 with 8 worker warps, BN = 64 with 16):
//   warp 0        TMA producer: raw fp32 tiles of A and B -> smem stage s             (full[s])
//   warp 1        MMA issuer (one elected lane): per stage 3 x BK/8 tcgen05.mma, commit -> empty[s];
//                 per chunk commit -> acc_full[buf].  Running counters only (stage / phase / A slot / position
//                 in the chunk): the issue loop must not be the limiter (round 1: ~210 instructions per k-block
//                 around 12 MMAs made it so; ~95 now).
//   workers       groups of four warps taking k-blocks round robin.  (1) splitter: read the raw stage with
//                 ld.shared, A -> hi/lo into TENSOR memory (tcgen05.st), B -> `hi` back in place and the `lo`
//                 tile next to it                                                      (split[s])
//                 (2) drain: TMEM chunk -> registers, running sum += chunk             (acc_empty[buf])
//                 (3) epilogue on the register-resident row (bias/relu/dropout/...), store.
// Programmatic dependent launch: the TMA warp calls griddepcontrol.launch_dependents once its last load is issued, every
// kernel parks at griddepcontrol.wait after its prologue (barrier init, TMEM allocation, tensor-map prefetch), and is
// launched with programmatic stream serialization, so the next GEMM's prologue overlaps this one's drain / epilogue.
// Operand tiles in smem are the canonical UMMA layouts written by TMA with hardware
// swizzle, so the splitter is swizzle-agnostic (same offset in the `lo` buffer) and the
// same smem descriptors serve hi and lo.
#pragma once
#include <cuda.h>

#include <type_traits>

#include "common.cuh"
#include "gemm_simt.cuh"   // Epilogue struct + EpiKind

namespace recnn {
namespace tc {

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must not hang the GPU (a wedged box costs a whole lease), so
// after ~2 s of polling the kernel traps and the launch surfaces as a CUDA error instead.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) {
      printf("recnn_b200: mbarrier wait timed out (block %d,%d,%d thread %d bar %u)\n", blockIdx.x, blockIdx.y,
             blockIdx.z, threadIdx.x, bar);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// arrives on `bar` once every tcgen05.mma issued so far by this thread has completed
// One lane of a fully converged warp (elect.sync); the compiler then knows the guarded tcgen05/TMA
// instructions run in a single thread and emits them without a per-lane serialisation loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// acc[0..NC) += D[lane, col0 .. col0+NC) with round-to-nearest adds (NC = 16 or a multiple of 32)
template <int NC>
__device__ __forceinline__ void tmem_accumulate(uint32_t taddr, float (&acc)[NC]);
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <int NC>
__device__ __forceinline__ void tmem_accumulate(uint32_t taddr, float (&acc)[NC]) {
  if constexpr (NC == 16) {
    uint32_t r[16];
    tmem_ld16(taddr, r);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = __fadd_rn(acc[j], __uint_as_float(r[j]));
  } else {
#pragma unroll
    for (int c0 = 0; c0 < NC; c0 += 32) {
      uint32_t r[32];
      tmem_ld32(taddr + c0, r);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) acc[c0 + j] = __fadd_rn(acc[c0 + j], __uint_as_float(r[j]));
    }
  }
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
        "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// A operand read from tensor memory (128 lanes = rows, 8 fp32 columns = one k-slice), B from shared memory
__device__ __forceinline__ void mma_tf32_ta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Programmatic dependent launch: launch_dependents lets the next kernel of the stream
// be scheduled onto idle SMs while this one finishes; its threads park at griddep_wait() -- after their prologue,
// before any global-memory access -- until this grid has completed and its writes are visible.  Both are no-ops for
// a launch without the programmatic-serialization attribute.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// Round-to-nearest (ties away) to TF32 = add half a TF32 ulp to the magnitude bits, clear the low 13.
// Bit-identical to cvt.rna.tf32.f32 for finite inputs, but two full-rate integer ops instead of a
// quarter-rate conversion (the splitter was bound by the conversion pipe: 16 K cvt per k-block per SM).
__device__ __forceinline__ float tf32_rna(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}
// x = hi + lo (+ <= 2^-24 |x|): hi = rna_tf32(x), lo = rna_tf32(x - hi)
// lo is handed to the tensor core as is: the kind::tf32 datapath ignores an operand's low 13 bits, i.e. it truncates
// the (at most 13-bit) remainder to 11 bits -- an error of at most 2^-22 |x| with random sign (hi is rounded to
// nearest, so lo is symmetric), against 2^-23 |x| if lo were rounded first, for two integer instructions less per
// operand element in the split warps (measured: -4% on the layer-1 GEMM, all accuracy bars unchanged, profiles/r2c).
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = x - hi;
}
__device__ __forceinline__ void tf32_split4(const float4& x, float4& hi, float4& lo) {
  tf32_split(x.x, hi.x, lo.x);
  tf32_split(x.y, hi.y, lo.y);
  tf32_split(x.z, hi.z, lo.z);
  tf32_split(x.w, hi.w, lo.w);
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout).
__host__ __device__ constexpr uint64_t smem_desc_base(uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return (uint64_t(lbo_bytes >> 4) << 16) | (uint64_t(sbo_bytes >> 4) << 32) | (uint64_t(1) << 46) |
         (uint64_t(layout_type) << 61);
}
// Instruction descriptor for kind::tf32, fp32 accumulate (cute::UMMA::InstrDescriptor).
__host__ __device__ constexpr uint32_t instr_desc_tf32(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) |
         (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

struct Problem {
  int M, N, K0, K1;      // K = K0 (+ K1 from a second A tensor: virtual concat along K, K-major A only)
  int k_chunk;           // k extent per split (multiple of BK), split index = blockIdx.z
  int b_k1_offset;       // B's k coordinate where the K1 segment starts (== K0 for a dense weight)
  int n_out_offset;      // column offset added when storing (C window)
  int b_n_offset;        // B's n coordinate of output column 0 (window into a wider B, e.g. W1[:, S:S+A])
  int n_skip;            // the first n_skip output columns are computed but not stored (operand lead pads)
#ifdef RECNN_TC_INSTRUMENT
  unsigned long long* trace;   // per-CTA %globaltimer stamps (8 per CTA): instrumented builds only
#endif
};

#ifdef RECNN_TC_INSTRUMENT
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define RECNN_TRACE(slot)                                                                          \
  do {                                                                                             \
    if (p.trace) p.trace[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 + (slot)] = gtimer(); \
  } while (0)
#else
#define RECNN_TRACE(slot) do { } while (0)
#endif

template <int BN_, int STAGES_, bool A_MN_, bool B_MN_>
struct Cfg {
  // BK = 32 (128-byte K-major rows): TMA moves 64-byte rows at half the rate of 128-byte rows (measured:
  // 31 B/clk/SM with BK = 16), and the operand stream is one of the kernel's bottlenecks.
  static constexpr int BM = 128, BN = BN_, BK = 32, STAGES = STAGES_;
  static constexpr int CH = 64 / BK;                               // k-blocks per TMEM accumulation chunk (K = 64)
  static constexpr bool A_MN = A_MN_, B_MN = B_MN_;
  static constexpr int D_COLS = 3 * BN;                            // D_hi chunk x2 | D_lo
  // The split A tile goes to TENSOR memory (tcgen05.st) and the MMA reads it from there, so A costs shared
  // memory one TMA write + one read instead of write + read + 2 writes + 6 MMA reads.
  static constexpr int A_SLOT_COLS = 2 * BK, A_SLOTS = (512 - D_COLS) / A_SLOT_COLS;   // hi | lo per k-block: 2 slots at BN = 128, 5 at BN = 64
  static constexpr int A_BYTES = BM * BK * 4, B_BYTES = BN * BK * 4;
  static constexpr int STAGE_BYTES = A_BYTES + 2 * B_BYTES;        // raw A | raw B (split in place into hi) | lo B
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 512 /*barriers*/;
  // Worker warps come in groups of four (one warp per TMEM lane quarter); the groups take k-blocks round robin.
  // 64-wide tiles run four groups (their A ring in tensor memory has five slots), 128-wide tiles two.
  static constexpr int WORKERS = BN == 64 ? 16 : 8;
  static constexpr int COLS_PER_WORKER = BN / (WORKERS / 4);       // register-resident running sum per thread
  // MMA-issue warps: 64-wide tiles run two that take alternate k-blocks (their MMAs are short, 32 clk of pipe each, so
  // the issue loop's overhead is what the pipe waits for: -3% with two issuers), 128-wide tiles one (measured 4%
  // slower with two: the hand-over costs more than the overlap gains when every MMA keeps the pipe busy for 64 clk)
  static constexpr int ISSUERS = BN == 64 ? 2 : 1;
  static constexpr int THREADS = 96 + 32 * WORKERS;                // TMA warp, two MMA-issue warp slots, workers
  static constexpr int TMEM_COLS = 512;                            // D_hi chunk x2 | D_lo | A ring
  static constexpr int A_COL0 = D_COLS;
  static constexpr int K_SWZ = BK * 4;                             // K-major rows: 128 B (SWIZZLE_128B)
  static_assert(BN == 64 || BN == 128, "BN");
  static_assert(COLS_PER_WORKER == 16 || COLS_PER_WORKER % 32 == 0, "drain width");
  static_assert(WORKERS / 4 <= A_SLOTS, "every group in flight needs its own A slot");
  static_assert(SMEM_BYTES <= 227 * 1024, "smem");
};

// ------------------------------------------------------------------ epilogue on a register-resident row
// acc[j] is C[m, nb + j] for j < NC (NC = 16 or a multiple of 32), handled in blocks of W = min(NC, 32)
// columns.  Stores 16 bytes at a time when the destination allows it.
template <int EPI, int NC>
__device__ __forceinline__ void epilogue_row(const Epilogue& e, const Problem& p, int m, int nb, int z,
                                             float (&acc)[NC]) {
  constexpr int W = NC < 32 ? NC : 32;
  static_assert(NC % W == 0 && (W == 16 || W == 32), "epilogue block width");
  const int N = p.N;
  if (m >= p.M) return;
  float* out_row;
  if (EPI == EPI_PARTIAL) out_row = e.out + ((long long)z * p.M + m) * e.ldo + p.n_out_offset;
  else out_row = e.out + (long long)m * e.ldo + p.n_out_offset;
  float row_g = 0.f, row_max = 0.f, row_sum = 1.f;
  long long row_item = 0;                  // EPI_DLOGITS: the drawn action as a column of this output
  if (EPI == EPI_DLOGITS) {
    row_g = e.row_g[m]; row_max = e.row_max[m]; row_sum = e.row_sum[m];
    row_item = e.row_action[m] - e.col0;
  }
#pragma unroll
  for (int j0 = 0; j0 < NC; j0 += W) {
    if (nb + j0 < N) {
      uint32_t keep_bits = 0xFFFFFFFFu;
      if (EPI == EPI_HIDDEN && e.train) {
        if (e.mask) {
          keep_bits = 0;
          const uint8_t* mrow = e.mask + (long long)m * N + nb + j0;
#pragma unroll
          for (int j = 0; j < W; ++j)
            if (nb + j0 + j < N && mrow[j]) keep_bits |= 1u << j;
        } else {
          // same stream as the CUDA-core path: bit (idx & 31) of word idx >> 5, idx = m*N + n
          const unsigned long long idx = (unsigned long long)m * N + nb + j0;
          if ((idx & 31) + W <= 32) {          // the block's W bits sit in one 32-bit word
            keep_bits = philox_keep_bits32(e.seed, (unsigned long long)*e.rng_step, e.stream_id, idx >> 5) >> (idx & 31);
          } else {
            keep_bits = 0;
#pragma unroll 1
            for (int j = 0; j < W; ++j) {
              const unsigned long long ij = idx + j;
              const uint32_t w = philox_keep_bits32(e.seed, (unsigned long long)*e.rng_step, e.stream_id, ij >> 5);
              keep_bits |= ((w >> (ij & 31)) & 1u) << j;
            }
          }
        }
      }
#pragma unroll
      for (int j4 = 0; j4 < W; j4 += 4) {
        const int n = nb + j0 + j4;
        if (n < N) {
          float v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float x = acc[j0 + j4 + u];
            const int nn = n + u;
            if (nn < N) {
              if (EPI == EPI_HIDDEN) {
                x = fmaxf(x + __ldg(e.bias + nn), 0.f);
                if (e.train) x = ((keep_bits >> (j4 + u)) & 1u) ? x * 2.0f : 0.f;
              } else if (EPI == EPI_LINEAR) {
                x = x + __ldg(e.bias + nn);
                if (e.apply_tanh) x = tanhf(x);
                if (e.add_noise) {
                  float z0;
                  if (e.noise) z0 = e.noise[(long long)m * N + nn];
                  else {
                    const unsigned long long idx = (unsigned long long)m * N + nn;
                    Philox ph(e.seed);
                    const uint4 r = ph(idx, ((unsigned long long)*e.rng_step << 8) | e.stream_id);
                    const float u1 = (r.x + 1.0f) * 2.3283064365386963e-10f;
                    const float u2 = r.y * 2.3283064365386963e-10f;
                    z0 = sqrtf(-2.0f * __logf(u1)) * __cosf(6.283185307179586f * u2) * e.noise_std;
                  }
                  x += fminf(fmaxf(z0, -e.noise_clip), e.noise_clip);
                }
              } else if (EPI == EPI_GATE) {
                x = e.h[(long long)m * e.ldh + nn] > 0.f ? x * e.gate_scale : 0.f;
              } else if (EPI == EPI_DLOGITS) {
                x = dlogit(row_g, x + __ldg(e.bias + nn), row_max, row_sum, nn == row_item);
              } else if (EPI == EPI_ACCUM) {
                x = out_row[nn] + x;
                if (e.h) x = e.h[(long long)m * e.ldh + nn] > 0.f ? x * e.gate_scale : 0.f;
              }
            }
            v[u] = x;
          }
          float* dst = out_row + n;
          if (n + 3 < N && n >= p.n_skip && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
            *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
          } else {
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (n + u < N && n + u >= p.n_skip) dst[u] = v[u];
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------ the kernel
template <class C, int EPI>
__global__ void __launch_bounds__(C::THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
               const __grid_constant__ CUtensorMap map_b, Problem p, Epilogue epi) {
  constexpr int BM = C::BM, BN = C::BN, BK = C::BK, STAGES = C::STAGES, CH = C::CH;
  constexpr int NC = C::COLS_PER_WORKER, WORKERS = C::WORKERS, NG = WORKERS / 4;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;       // shared-window address, 1 KB aligned
  auto stage_addr = [&](int s, int which) -> uint32_t {              // 0 raw A, 1 raw B (-> hi B), 2 lo B
    const uint32_t base = smem + (uint32_t)s * C::STAGE_BYTES;
    return which == 0 ? base : which == 1 ? base + C::A_BYTES : base + C::A_BYTES + C::B_BYTES;
  };
  const uint32_t bars = smem + (uint32_t)STAGES * C::STAGE_BYTES;
  auto full = [&](int s) { return bars + 8u * s; };                   // TMA -> workers
  auto split = [&](int s) { return bars + 8u * (STAGES + s); };       // workers -> MMA
  auto empty = [&](int s) { return bars + 8u * (2 * STAGES + s); };   // MMA -> TMA
  auto acc_full = [&](int b) { return bars + 8u * (3 * STAGES + b); };       // MMA -> workers
  auto acc_empty = [&](int b) { return bars + 8u * (3 * STAGES + 2 + b); };  // workers -> MMA
  auto a_free = [&](int i) { return bars + 8u * (3 * STAGES + 4 + i); };    // MMA -> workers (A TMEM ring)
  auto turn = [&](int x) { return bars + 8u * (3 * STAGES + 4 + C::A_SLOTS + x); };   // MMA warp x may issue (two-issuer mode)
  const uint32_t tmem_slot = bars + 8u * (3 * STAGES + 6 + C::A_SLOTS);
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, z = blockIdx.z;
  if (threadIdx.x == 0) RECNN_TRACE(0);                       // kernel entry
  // k-blocks: segment 0 then segment 1, each padded up to a multiple of BK (TMA zero-fills the tail)
  const int nkb0 = (p.K0 + BK - 1) / BK, nkb1 = (p.K1 + BK - 1) / BK;
  const int kb_per_split = p.k_chunk / BK;
  const int kb_begin = z * kb_per_split;
  const int kb_end = min(nkb0 + nkb1, kb_begin + kb_per_split);
  const int num_kb = max(kb_end - kb_begin, 0);
  const int num_chunks = (num_kb + CH - 1) / CH;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_b);
    if (p.K1 > 0) tma_prefetch_desc(&map_a1);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full(s), 1);
      mbar_init(split(s), 4);                            // one arrive per warp of the group that split the stage
      mbar_init(empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc_full(b), C::ISSUERS);                   // one commit per MMA-issue warp
      mbar_init(acc_empty(b), WORKERS);
    }
    for (int i = 0; i < C::A_SLOTS; ++i) mbar_init(a_free(i), 1);
    mbar_init(turn(0), 1);
    mbar_init(turn(1), 1);
    fence_barrier_init();
  }
  if (warp == 1) {                       // whole warp: TMEM allocation
    tmem_alloc(tmem_slot, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  griddep_wait();                                             // everything below may touch global memory
  if (threadIdx.x == 0) RECNN_TRACE(1);                       // prologue done

  if (warp == 0) {
    // ===================================================== TMA producer (whole warp walks, one elected lane issues)
    const bool leader = elect_one();
    uint32_t s = 0, ph = 0;
    for (int i = 0; i < num_kb; ++i) {
      mbar_wait(empty(s), ph ^ 1u);
      const int kb = kb_begin + i;
      const bool seg1 = kb >= nkb0;
      const int ka = seg1 ? (kb - nkb0) * BK : kb * BK;                     // k coordinate inside A's segment
      const int kbcol = seg1 ? p.b_k1_offset + (kb - nkb0) * BK : kb * BK;  // k coordinate in B
      const CUtensorMap* ma = seg1 ? &map_a1 : &map_a0;
      const uint32_t dst_a = stage_addr(s, 0), dst_b = stage_addr(s, 1);
      if (leader) {
        mbar_expect_tx(full(s), C::A_BYTES + C::B_BYTES);
        if (!C::A_MN) {
          tma_load_2d(dst_a, ma, full(s), ka, m0);                            // box {BK, 128}
        } else {
#pragma unroll
          for (int c = 0; c < BM / 32; ++c)                                   // box {32, BK} per 32-wide M chunk
            tma_load_2d(dst_a + c * (BK * 128), ma, full(s), m0 + 32 * c, ka);
        }
        if (!C::B_MN) {
          tma_load_2d(dst_b, &map_b, full(s), kbcol, p.b_n_offset + n0);      // box {BK, BN}
        } else {
#pragma unroll
          for (int c = 0; c < BN / 32; ++c)
            tma_load_2d(dst_b + c * (BK * 128), &map_b, full(s), p.b_n_offset + n0 + 32 * c, kbcol);
        }
      }
      __syncwarp();
      if (++s == (uint32_t)STAGES) { s = 0; ph ^= 1u; }
    }
    // All loads issued, STAGES k-blocks before the last MMA: NOW the next kernel of the stream may be scheduled (one thread's
    // trigger counts for its CTA).  Its CTAs run their prologue and park at griddepcontrol.wait holding an SM each, so
    // releasing them at kernel entry (r1-r2i) let them squat on SMs that concurrent GEMMs of the step's other chains
    // could have used for a whole kernel duration; released here they wait for an epilogue's length.  r2k, DDPG step:
    // trigger at entry 2708 steps/s, never (dependents start at grid exit) 2750-2764, here 2823.
    griddep_launch_dependents();
  } else if (warp == 1 || warp == 2) {
    // ===================================================== MMA issuer(s)
    // The whole warp walks the pipeline (so every value below is warp-uniform and lives in uniform
    // registers); one elected lane issues the MMAs and commits.  Issuing under `if (lane == 0)` instead makes
    // the compiler wrap every tcgen05 instruction in an ELECT/BRA.U.ANY loop, which made the issue stream,
    // not the tensor pipe, the limiter (~130 clk per MMA against a 64 clk floor).
    // A read from tensor memory is always [M lanes, K columns] = K-major, whatever its layout in global memory.
    //
    // Two issuers: measured on the single-issuer kernel (profiles/README.md r2b/r2c), a k-block costs
    // ~(500 clk of loop overhead -- barrier polls at ~90 clk each, descriptor arithmetic in the uniform datapath) PLUS the
    // pipe time of its 12 MMAs, because the tensor core's instruction queue is too shallow to keep the pipe busy across
    // the overhead.  With two warps (1 and 2) taking alternate k-blocks, one warp's polls and arithmetic for k-block i+1 run while
    // the other issues k-block i; a `turn` barrier hands the issue slot over (tcgen05.fence::before_thread_sync ->
    // arrive -> wait -> fence::after_thread_sync orders the two threads' MMAs), and both warps commit to acc_full.
    constexpr uint32_t idesc = instr_desc_tf32(BM, BN, false, C::B_MN);
    // K-major B: rows of 128 bytes, LBO unused (1), SBO = 8 rows.  MN-major fp32/tf32 operands must
    // use the 128B_BASE32B layout (cute: "for mn-major tf32 operands, SW128_32B is the only available
    // smem layout"): 128-byte rows of 32 MN elements, swizzle period 4 k-rows => SBO = 512 B between
    // 4-row groups, LBO = pitch between 32-element MN chunks (BK rows * 128 B).
    constexpr uint64_t b_base = C::B_MN ? smem_desc_base(BK * 128, 512, 1) : smem_desc_base(16, 8 * C::K_SWZ, 2);
    constexpr uint32_t b_kstep = C::B_MN ? 1024 : 32;        // bytes to advance per 8-wide k-slice
    // Each of the two warps keeps running counters for ITS k-blocks (me, me + 2, ...): no division, no modulo --
    // every instruction in this loop sits between two tensor-core instructions (with index arithmetic instead of
    // counters the same kernel was 26% slower, profiles/r2f).  CH = 2, so issuer 0 always opens a chunk (waits for its
    // drained buffer, overwrites with its first hi*hi MMA) and issuer 1 always closes it.
    static_assert(CH == 2 && STAGES % 2 == 0, "the issue schedules assume two k-blocks per chunk and an even ring");
    constexpr int NI = C::ISSUERS;                           // k-blocks ME, ME + NI, ... belong to issuer ME
    auto issue = [&](auto me_c) {
      constexpr int ME = decltype(me_c)::value;
      const bool leader = elect_one();
      const uint32_t d_lo = tmem_base + 2u * BN;             // tile-lifetime accumulator (cross terms)
      uint32_t s = ME, ph = 0, slot = ME, kin = ME, buf = 0, par0 = 1, par1 = 1, tpar = 0;
      for (int i = ME; i < num_kb; i += NI) {
        if (kin == 0) {                                      // new chunk: its TMEM buffer must have been drained
          mbar_wait(acc_empty(buf), buf ? par1 : par0);
          if (buf) par1 ^= 1u; else par0 ^= 1u;
        }
        mbar_wait(split(s), ph);
        if (NI == 2 && i > 0) {                              // my k-block follows the other warp's k-block i - 1
          mbar_wait(turn(ME), tpar);
          tpar ^= 1u;
        }
        tc_fence_after();
        if (ME == 0 && i == 0 && lane == 0) RECNN_TRACE(2);  // first stage loaded + split
        const uint32_t d_hi = tmem_base + buf * BN;          // chunk accumulator (hi*hi)
        const uint64_t db_hi0 = b_base | uint64_t((stage_addr(s, 1) & 0x3FFFF) >> 4);
        const uint64_t db_lo0 = b_base | uint64_t((stage_addr(s, 2) & 0x3FFFF) >> 4);
        const uint32_t ta0 = tmem_base + C::A_COL0 + slot * C::A_SLOT_COLS;
        if (leader) {
#pragma unroll
          for (int k = 0; k < BK / 8; ++k) {
            const uint64_t db_hi = db_hi0 + uint64_t((k * b_kstep) >> 4);
            const uint64_t db_lo = db_lo0 + uint64_t((k * b_kstep) >> 4);
            const uint32_t ta_hi = ta0 + k * 8, ta_lo = ta_hi + BK;
            const uint32_t lo_flag = (ME == 0 && k == 0 && i == 0) ? 0u : 1u, hi_flag = (k == 0 && kin == 0) ? 0u : 1u;
            mma_tf32_ta(d_lo, ta_lo, db_hi, idesc, lo_flag);
            mma_tf32_ta(d_lo, ta_hi, db_lo, idesc, 1);
            mma_tf32_ta(d_hi, ta_hi, db_hi, idesc, hi_flag);
          }
          mma_commit(empty(s));                              // frees the stage once these MMAs have read it
          mma_commit(a_free(slot));                          // ... and the A slot in tensor memory
          if (NI == 2) {
            // acc_full collects one commit per issuer (a commit covers the issuing thread's MMAs only); the issuer of a
            // tile's last k-block also commits for a partner that has no k-block in the (short) last chunk
            mma_commit(acc_full(buf));
            if (ME == 0 && i == num_kb - 1) mma_commit(acc_full(buf));
          } else if (kin == (uint32_t)(CH - 1) || i == num_kb - 1) {
            mma_commit(acc_full(buf));
          }
        }
        __syncwarp();
        if (NI == 2 && i + 1 < num_kb) {                     // hand the issue slot to the other warp
          tc_fence_before();
          if (lane == 0) mbar_arrive(turn(ME ^ 1));
        }
        s += NI;
        if (s >= (uint32_t)STAGES) { s -= (uint32_t)STAGES; ph ^= 1u; }
        slot += NI;
        if (slot >= (uint32_t)C::A_SLOTS) slot -= (uint32_t)C::A_SLOTS;
        if (NI == 2) {
          buf ^= 1u;                                         // kin stays ME: issuer 0 opens every chunk, issuer 1 closes it
        } else if (++kin == (uint32_t)CH) {
          kin = 0;
          buf ^= 1u;
        }
      }
      if (ME == 0 && lane == 0) RECNN_TRACE(3);               // last MMA issued by issuer 0
    };
    if (warp == 1) issue(std::integral_constant<int, 0>{});
    else if (NI == 2) issue(std::integral_constant<int, 1>{});
  } else {
    // ===================================================== workers: split, drain, epilogue
    const int q = warp & 3;                  // TMEM lane quarter this warp may access
    const int g = (warp - 3) >> 2;           // worker group: k-blocks g, g + NG, ...; column slab g of the drain / epilogue
    const int tg = (threadIdx.x - 96) & 127; // index among the 128 threads of the group
    float acc[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) acc[j] = 0.f;
    const uint32_t lane_base = tmem_base + (uint32_t(32 * q) << 16) + (uint32_t)g * NC;

    auto drain = [&](int chunk) {
      const int buf = chunk & 1;
      mbar_wait(acc_full(buf), (chunk >> 1) & 1);
      tc_fence_after();
      tmem_accumulate<NC>(lane_base + (uint32_t)buf * BN, acc);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty(buf));
    };

    // The groups take k-blocks round robin, so one group's publish latency (membar + proxy fence +
    // tcgen05.wait::st) hides behind the other groups' arithmetic.
    constexpr int VB = C::B_BYTES / 16 / 128;                 // float4s of the B tile per thread of the group
    static_assert(C::B_BYTES / 16 % 128 == 0 && VB >= 1, "B tile must split evenly over a worker group");
    int next_drain = 0;
    for (int i = g; i < num_kb; i += NG) {
      const int s = i % STAGES;
      const uint32_t ph = (i / STAGES) & 1;
      mbar_wait(full(s), ph);
      const uint32_t raw = stage_addr(s, 1);                  // raw B, split in place into hi
      const uint32_t lo = stage_addr(s, 2);                   // lo B
      const int slot = i % C::A_SLOTS;
      const uint32_t ta = tmem_base + (uint32_t(32 * q) << 16) + C::A_COL0 + slot * C::A_SLOT_COLS;
      mbar_wait(a_free(slot), ((i / C::A_SLOTS) & 1) ^ 1);
      tc_fence_after();
      if (C::A_MN) {
        // MN-major A tile: 4 chunks (32 rows of M each) x BK k-rows of 128 bytes; TMA's 128B_ATOM_32B swizzle
        // XORs the 32-byte unit index with (k & 3).  My TMEM lane is row m = 32*q + lane: chunk q, element `lane`
        // of every k-row -> one conflict-free 128-byte wavefront per k for the warp.
        const uint32_t cbase = stage_addr(s, 0) + (uint32_t)q * (BK * 128u) + (((uint32_t)lane & 7u) << 2);
        const uint32_t unit = (uint32_t)lane >> 3;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float hi[16], lw[16];
#pragma unroll
          for (int kk = 0; kk < 16; ++kk) {
            const uint32_t k = 16u * half + kk;
            float x;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(x) : "r"(cbase + k * 128u + ((unit ^ (k & 3u)) << 5)));
            tf32_split(x, hi[kk], lw[kk]);
          }
          tmem_st16(ta + 16 * half, hi);
          tmem_st16(ta + BK + 16 * half, lw);
        }
      } else {
        // my row of the K-major A tile -> hi/lo in TMEM.  Rows are 128 bytes; TMA's SWIZZLE_128B XORs the
        // 16-byte chunk index with address bits [7, 10) = row & 7.
        const int row = 32 * q + lane;
        const uint32_t rbase = stage_addr(s, 0) + (uint32_t)row * 128u;
        const uint32_t sw = (uint32_t)row & 7u;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float hi[16], lw[16];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 x = lds128(rbase + (((4 * half + j) ^ sw) << 4));
            tf32_split(x.x, hi[4 * j + 0], lw[4 * j + 0]);
            tf32_split(x.y, hi[4 * j + 1], lw[4 * j + 1]);
            tf32_split(x.z, hi[4 * j + 2], lw[4 * j + 2]);
            tf32_split(x.w, hi[4 * j + 3], lw[4 * j + 3]);
          }
          tmem_st16(ta + 16 * half, hi);
          tmem_st16(ta + BK + 16 * half, lw);
        }
      }
      {
        float4 x[VB];
#pragma unroll
        for (int v = 0; v < VB; ++v) x[v] = lds128(raw + 16u * ((uint32_t)tg + v * 128u));
#pragma unroll
        for (int v = 0; v < VB; ++v) {
          float4 xh, xl;
          tf32_split4(x[v], xh, xl);
          sts128(raw + 16u * ((uint32_t)tg + v * 128u), xh);
          sts128(lo + 16u * ((uint32_t)tg + v * 128u), xl);
        }
      }
      // generic-proxy writes (B hi/lo in shared memory) -> visible to the tensor core (async proxy)
      fence_proxy_async();
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(split(s));
      // after my last k-block of chunk c, chunk c-1 has long been accumulated: drain it
      if ((i + NG) / CH != i / CH)
        while (next_drain < i / CH) drain(next_drain++);
    }
    if (threadIdx.x == 96) RECNN_TRACE(4);                    // last stage split
    while (next_drain < num_chunks) drain(next_drain++);      // the last full chunk (and a trailing partial one)
    if (threadIdx.x == 96) RECNN_TRACE(5);                    // all chunks drained (MMAs complete)
    if (num_kb > 0)   // the commit behind the last acc_full covers every MMA issued before it, D_lo's included
      tmem_accumulate<NC>(lane_base + 2u * BN, acc);
    epilogue_row<EPI, NC>(epi, p, m0 + 32 * q + lane, n0 + g * NC, z, acc);
    if (threadIdx.x == 96) RECNN_TRACE(6);                    // epilogue stored
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
  if (threadIdx.x == 0) RECNN_TRACE(7);
}

// ------------------------------------------------------------------ host side
// cuTensorMapEncodeTiled is fetched from the driver at run time (the library does not
// link libcuda, so it also loads on a box without a GPU).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn();

// 2-D fp32 tensor [rows, cols] with row pitch ld (floats, multiple of 4); box = {box_cols, box_rows}.
// swizzle_bytes: 64 / 128 = the classic 16-byte-unit swizzles; 1032 = 128B span with 32-byte units
// (CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, the partner of the UMMA 128B_BASE32B layout).
int make_tmap(CUtensorMap* out, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
              int box_rows, int swizzle_bytes);

// A global operand.  rows/cols describe the tensor as stored (only used for B; A's extents come
// from the Problem): K-major B is [N_total, K_total], MN-major B is [K_total, N_total].
struct Operand {
  const float* ptr;
  long long ld;
  long long rows, cols;
};

// k-blocks (of bk) per split and the effective split count for a requested split count.
int split_plan(int K_total_blocks, int splits_req, int* k_chunk, int bk = 16);

// Launch one GEMM.  Returns the effective number of k-splits (> 0) or a negative RECNN_E_* code.
template <bool A_MN, bool B_MN, int EPI>
int launch(const Operand& A0, const Operand& A1, const Operand& B, const Problem& p, int splits, int bn,
           const Epilogue& epi, cudaStream_t st);

}  // namespace tc
}  // namespace recnn
