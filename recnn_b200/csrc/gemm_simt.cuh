// fp32 CUDA-core GEMM with fused epilogues.
//
// Role in the design (DESIGN.md "kernels"): exact-fp32 building block for every
// contraction of the update step.  It is the arbitrary-shape path (any S/A/H,
// any row count) and the on-device reference the tcgen05 3xTF32 kernels are
// unit-tested against.  C[m,n] = sum_k A(m,k) * B(n,k) with both operands given
// as "views" so the reference's torch.cat([state, action], 1)
// (recnn/nn/models.py:207) and the bias column of a weight-gradient never have
// to be materialised.
#pragma once
#include "common.cuh"

namespace recnn {

// A matrix whose contiguous axis may be the concatenation of two buffers, plus
// an optional virtual column of ones appended at index `ones_at`.
//   elem(r, c) = c <  split ? p0[r*ld0 + c] : p1[r*ld1 + (c - split)]   (c != ones_at)
struct MatView {
  const float* p0;
  long long ld0;
  int split;        // INT_MAX => single segment
  const float* p1;
  long long ld1;
  int ones_at;      // -1 => none
};

static inline MatView mat(const float* p, long long ld) {
  MatView v; v.p0 = p; v.ld0 = ld; v.split = 0x7fffffff; v.p1 = nullptr; v.ld1 = 0; v.ones_at = -1; return v;
}
static inline MatView mat_cat(const float* p0, long long ld0, int split, const float* p1, long long ld1) {
  MatView v; v.p0 = p0; v.ld0 = ld0; v.split = split; v.p1 = p1; v.ld1 = ld1; v.ones_at = -1; return v;
}

__device__ __forceinline__ float view_at(const MatView& v, long long r, int c) {
  if (c == v.ones_at) return 1.0f;
  return c < v.split ? __ldg(v.p0 + r * v.ld0 + c) : __ldg(v.p1 + r * v.ld1 + (c - v.split));
}

enum EpiKind {
  EPI_HIDDEN = 0,   // out = relu(acc + bias[n]) * keep(m,n)*2          (models.py:66-69)
  EPI_LINEAR = 1,   // out = acc + bias[n] (+tanh) (+clamp(noise))       (models.py:70-72, td3.py:74-78)
  EPI_GATE = 2,     // out = acc * (h[m,n] > 0 ? gate_scale : 0)          (relu'/dropout backward)
  EPI_STORE = 3,    // out = acc
  EPI_PARTIAL = 4,  // split-K partial: part[z][m][n] = acc
  EPI_DLOGITS = 5,  // out = g[m] ([col0 + n == a[m]] - exp(acc + bias[n] - M[m]) / S[m])   (REINFORCE d logits)
  EPI_ACCUM = 6     // out += acc, then (h given) the EPI_GATE gate of the sum
};

struct Epilogue {
  float* out;            // [M, ldo]
  long long ldo;
  const float* bias;     // [N]
  const uint8_t* mask;   // [M, N] keep mask or null
  int train;             // dropout active (mask or philox)
  unsigned long long seed;
  const long long* rng_step;
  unsigned stream_id;
  const float* h;        // EPI_GATE: forward activation [M, ldh]
  long long ldh;
  float gate_scale;
  int apply_tanh;
  const float* noise;    // EPI_LINEAR: optional [M, N]
  float noise_clip;
  float noise_std;       // perf mode: philox normal * std (noise == null && add_noise)
  int add_noise;
  // EPI_DLOGITS: per-row softmax statistics of the full item range, the row's dL/dlp and drawn action; output column n
  // is item col0 + n
  const float* row_g;
  const float* row_max;
  const float* row_sum;
  const long long* row_action;
  long long col0;
};

// d loss / d logit of one item from its logit z (the same fp32 operations as the materialised path's
// softmax_rows_kernel + reinforce_dlogits_kernel)
__device__ __forceinline__ float dlogit(float g, float z, float M, float S, bool is_action) {
  return g * ((is_action ? 1.f : 0.f) - expf(z - M) / S);
}

template <int EPI>
__device__ __forceinline__ void epi_store(const Epilogue& e, int M, int N, int m, int n, float acc, int z) {
  if (EPI == EPI_PARTIAL) {
    e.out[((long long)z * M + m) * e.ldo + n] = acc;
    return;
  }
  float v = acc;
  if (EPI == EPI_HIDDEN) {
    v = fmaxf(v + e.bias[n], 0.f);
    if (e.train) {
      bool keep;
      if (e.mask) keep = e.mask[(long long)m * N + n] != 0;
      else {
        const unsigned long long idx = (unsigned long long)m * N + n;
        const uint32_t bits = philox_keep_bits32(e.seed, (unsigned long long)*e.rng_step, e.stream_id, idx >> 5);
        keep = (bits >> (idx & 31)) & 1u;
      }
      v = keep ? v * 2.0f : 0.f;
    }
  } else if (EPI == EPI_LINEAR) {
    v = v + e.bias[n];
    if (e.apply_tanh) v = tanhf(v);
    if (e.add_noise) {
      float z0;
      if (e.noise) z0 = e.noise[(long long)m * N + n];
      else {
        const unsigned long long idx = (unsigned long long)m * N + n;
        Philox ph(e.seed);
        const uint4 r = ph(idx, ((unsigned long long)*e.rng_step << 8) | e.stream_id);
        const float u1 = (r.x + 1.0f) * 2.3283064365386963e-10f;   // (0,1]
        const float u2 = r.y * 2.3283064365386963e-10f;
        z0 = sqrtf(-2.0f * __logf(u1)) * __cosf(6.283185307179586f * u2) * e.noise_std;
      }
      v += fminf(fmaxf(z0, -e.noise_clip), e.noise_clip);
    }
  } else if (EPI == EPI_GATE) {
    v = e.h[(long long)m * e.ldh + n] > 0.f ? v * e.gate_scale : 0.f;
  } else if (EPI == EPI_DLOGITS) {
    v = dlogit(e.row_g[m], v + e.bias[n], e.row_max[m], e.row_sum[m], e.col0 + n == e.row_action[m]);
  } else if (EPI == EPI_ACCUM) {
    v = e.out[(long long)m * e.ldo + n] + v;
    if (e.h) v = e.h[(long long)m * e.ldh + n] > 0.f ? v * e.gate_scale : 0.f;
  }
  e.out[(long long)m * e.ldo + n] = v;
}

// C[M,N] = sum_{k in split z} A(m,k) B(n,k).  A_K: A is K-contiguous (view row = m),
// else M-contiguous (view row = k).  Same for B.  Each thread owns an 8x8
// micro-tile split in 4x4 quadrants 64/BN2 apart so shared reads are conflict-free.
template <int BM, int BN, bool A_K, bool B_K, int EPI>
__global__ void __launch_bounds__((BM / 8) * (BN / 8))
gemm_simt_kernel(MatView A, MatView B, int M, int N, int K, int k_chunk, Epilogue epi) {
  constexpr int BK = 16;
  constexpr int THREADS = (BM / 8) * (BN / 8);
  constexpr int TX = BN / 8;   // threads along n
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];

  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int z = blockIdx.z;
  const int k_begin = z * k_chunk;
  const int k_end = min(K, k_begin + k_chunk);

  constexpr int A_ELEMS = BM * BK / THREADS;
  constexpr int B_ELEMS = BN * BK / THREADS;
  float ra[A_ELEMS], rb[B_ELEMS];

  auto load_tile = [&](int k0) {
#pragma unroll
    for (int i = 0; i < A_ELEMS; ++i) {
      const int e = tid + i * THREADS;
      int mm, kk;
      if (A_K) { kk = e % BK; mm = e / BK; } else { mm = e % BM; kk = e / BM; }
      const int m = m0 + mm, k = k0 + kk;
      float v = 0.f;
      if (m < M && k < k_end) v = A_K ? view_at(A, m, k) : view_at(A, k, m);
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < B_ELEMS; ++i) {
      const int e = tid + i * THREADS;
      int nn, kk;
      if (B_K) { kk = e % BK; nn = e / BK; } else { nn = e % BN; kk = e / BN; }
      const int n = n0 + nn, k = k0 + kk;
      float v = 0.f;
      if (n < N && k < k_end) v = B_K ? view_at(B, n, k) : view_at(B, k, n);
      rb[i] = v;
    }
  };
  auto stash_tile = [&](int buf) {
#pragma unroll
    for (int i = 0; i < A_ELEMS; ++i) {
      const int e = tid + i * THREADS;
      int mm, kk;
      if (A_K) { kk = e % BK; mm = e / BK; } else { mm = e % BM; kk = e / BM; }
      As[buf][kk][mm] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < B_ELEMS; ++i) {
      const int e = tid + i * THREADS;
      int nn, kk;
      if (B_K) { kk = e % BK; nn = e / BK; } else { nn = e % BN; kk = e / BN; }
      Bs[buf][kk][nn] = rb[i];
    }
  };

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  int buf = 0;
  if (k_begin < k_end) {
    load_tile(k_begin);
    stash_tile(0);
  }
  __syncthreads();
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    const bool has_next = k0 + BK < k_end;
    if (has_next) load_tile(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4 + BM / 2]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4 + BN / 2]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (has_next) {
      stash_tile(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }

#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + ty * 4 + (i & 3) + (i >> 2) * (BM / 2);
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = n0 + tx * 4 + (j & 3) + (j >> 2) * (BN / 2);
      if (n < N) epi_store<EPI>(epi, M, N, m, n, acc[i][j], z);
    }
  }
}

template <bool A_K, bool B_K, int EPI>
int launch_gemm_simt(const MatView& A, const MatView& B, int M, int N, int K, int splits,
                     const Epilogue& epi, cudaStream_t st) {
  if (M <= 0 || N <= 0) return RECNN_OK;
  if (splits < 1) splits = 1;
  int k_chunk = (int)round_up(ceil_div(K, splits), 16);
  splits = (int)ceil_div(K, k_chunk);
  // pick the largest tile that still gives ~a full wave of CTAs
  const int64_t t128 = ceil_div(M, 128) * ceil_div(N, 128) * splits;
  const int64_t t64 = ceil_div(M, 128) * ceil_div(N, 64) * splits;
  if (t128 >= 120) {
    dim3 grid((unsigned)ceil_div(N, 128), (unsigned)ceil_div(M, 128), splits);
    gemm_simt_kernel<128, 128, A_K, B_K, EPI><<<grid, 256, 0, st>>>(A, B, M, N, K, k_chunk, epi);
  } else if (t64 >= 100) {
    dim3 grid((unsigned)ceil_div(N, 64), (unsigned)ceil_div(M, 128), splits);
    gemm_simt_kernel<128, 64, A_K, B_K, EPI><<<grid, 128, 0, st>>>(A, B, M, N, K, k_chunk, epi);
  } else {
    dim3 grid((unsigned)ceil_div(N, 64), (unsigned)ceil_div(M, 64), splits);
    gemm_simt_kernel<64, 64, A_K, B_K, EPI><<<grid, 64, 0, st>>>(A, B, M, N, K, k_chunk, epi);
  }
  RECNN_CHECK_LAUNCH("gemm_simt_kernel");
  return RECNN_OK;
}

}  // namespace recnn
