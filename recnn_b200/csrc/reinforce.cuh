// REINFORCE with (Top-K) off-policy correction: the policy side (SURVEY 8f-2).
//
// Restates, for one GPU, recnn/nn/models.py:76-184 (DiscreteActor: forward, Categorical sampling, log-probs, importance
// correction, lambda_K) and recnn/nn/update/reinforce.py:10-65 (ChooseREINFORCE: the three policy losses and their
// backward).  Included at the end of step.cu: it is built from the same four contraction helpers as the DDPG / TD3 step
// (hidden_layer, linear_out, backprop_hidden, weight_grad -> tcgen05 3xTF32 GEMMs) plus three row kernels.
//
// What is different from the reference's formulation:
//   * the reference keeps one autograd graph per env step (saved_log_probs, models.py:110,156,183) and back-propagates
//     through all of them at the policy update.  The policy's weights do not change between two policy updates, so the
//     sum of those backward passes is ONE backward pass over the concatenation of the saved batches: the caller keeps
//     (state, sampled action, beta log-prob, step index) per row -- 5 KB/row instead of the [N, num_items] probability
//     matrices -- and recnn_reinforce_policy_grad recomputes the forward on the R = T*N saved rows.
//   * d loss / d logits has a closed form (softmax + log + the scalar weight of the row), so the backward starts from
//     ONE in-place row kernel that turns the probabilities into d logits; the rest is the usual three GEMMs.
//   * the normalised discounted returns (reinforce.py:44-52) are T scalars: host arithmetic in the caller.
//   * past what the [R, num_items] logits can hold (1M items), recnn_reinforce_policy_grad_streamed recomputes them one
//     item chunk at a time: a statistics pass (online softmax max / sum, the action's logit) and a backward pass whose
//     GEMM epilogue writes d logits (EPI_DLOGITS) for the chunk's dW2 and its term of dh.
//
// Per saved row n with sampled action a, p = clamp(pi[a], eps, 1-eps), lp = log p, R = return of the row's step:
//   basic   (reinforce.py:16-22)   L = -lp R                                 dL/dlp = -R
//   corr    (reinforce.py:24-33)   L = (p/b)(-lp) R     b = exp(beta lp)     dL/dlp = -R (p/b)(lp + 1)
//   top-K   (reinforce.py:35-44)   L = lam (p/b)(-lp) R, lam = K(1-p)^(K-1)  dL/dlp = -R/b [lam p (lp+1) - K(K-1)(1-p)^(K-2) p^2 lp]
// and d lp / d logits[j] = [j == a] - pi[j]   (corr and lam are NOT detached in the reference: models.py:150,168-171).
#pragma once

namespace recnn {

struct DiscreteLayout {
  int ld1, ld2;                      // row pitches of w1 [H, S] and w2 [num_items, H]
  int64_t w1, b1, w2, b2, count;
};
static inline DiscreteLayout discrete_layout(const recnn_discrete_dims& d) {
  DiscreteLayout l;
  l.ld1 = pad4(d.state_dim);
  l.ld2 = pad4(d.hidden);
  l.w1 = 0;
  l.b1 = l.w1 + (int64_t)d.hidden * l.ld1;
  l.w2 = l.b1 + pad4(d.hidden);
  l.b2 = l.w2 + (int64_t)d.num_items * l.ld2;
  l.count = l.b2 + pad4(d.num_items);
  return l;
}

constexpr int kRowThreads = 256;
constexpr float kProbEps = 1.1920928955078125e-07f;     // torch.finfo(float32).eps: Categorical clamps probs to [eps, 1-eps]

__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  float t = (threadIdx.x < nw) ? red[threadIdx.x] : -INFINITY;
  if (warp == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = fmaxf(t, __shfl_xor_sync(0xffffffffu, t, o));
  }
  if (threadIdx.x == 0) red[0] = t;
  __syncthreads();
  t = red[0];
  return t;
}

// z[r, :] <- softmax(z[r, :])      (models.py:99; F.softmax without dim on a 2-d input is dim=1)
// one CTA per row; the row is read twice (online max / sum, then the normalised write)
__global__ void __launch_bounds__(kRowThreads) softmax_rows_kernel(float* __restrict__ z, long long ld, long long n, int items) {
  __shared__ float red[32];
  for (long long r = blockIdx.x; r < n; r += gridDim.x) {
    float* row = z + r * ld;
    float m = -INFINITY, s = 0.f;
    for (int j = threadIdx.x; j < items; j += blockDim.x) {
      const float x = row[j];
      if (x > m) {
        s = s * __expf(m - x) + 1.f;      // m == -inf: s == 0, exp(-inf) == 0
        m = x;
      } else {
        s += __expf(x - m);
      }
    }
    const float M = block_max(m, red);
    s = (m == -INFINITY) ? 0.f : s * __expf(m - M);
    const float S = block_sum(s, red);
    for (int j = threadIdx.x; j < items; j += blockDim.x) row[j] = expf(row[j] - M) / S;
    __syncthreads();
  }
}

__device__ __forceinline__ float clamped_log_prob(float p) {
  return logf(fminf(fmaxf(p, kProbEps), 1.f - kProbEps));
}

// Categorical(probs).sample() and .log_prob(sample)   (models.py:107-110, 127-143).  torch normalises the probabilities
// by their row sum and clamps them to [eps, 1-eps] before the log (torch/distributions/categorical.py, utils.py).
// Sampling is by inverse CDF: the first j with cumsum(probs)[j] > u * sum(probs); u from `uniforms` (replayable) or from
// Philox keyed by (seed, draw, row).  One CTA per row.
__global__ void __launch_bounds__(kRowThreads)
categorical_sample_kernel(const float* __restrict__ probs, long long ld, long long n, int items,
                          const float* __restrict__ uniforms, unsigned long long seed, long long draw,
                          long long* __restrict__ action, float* __restrict__ logp) {
  __shared__ float red[32];
  __shared__ float warp_tot[kRowThreads / 32];
  __shared__ int found;
  __shared__ float run;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long r = blockIdx.x; r < n; r += gridDim.x) {
    const float* row = probs + r * ld;
    float t = 0.f;
    for (int j = threadIdx.x; j < items; j += blockDim.x) t += row[j];
    const float total = block_sum(t, red);
    float u;
    if (uniforms) {
      u = uniforms[r];
    } else {
      Philox ph(seed);
      const uint4 q = ph((unsigned long long)r, ((unsigned long long)draw << 8) | 0x5au);
      u = (float)(q.x >> 8) * (1.0f / 16777216.0f);          // [0, 1)
    }
    const float target = u * total;
    if (threadIdx.x == 0) {
      found = items;
      run = 0.f;
    }
    __syncthreads();
    for (int base = 0; base < items; base += blockDim.x) {
      const int j = base + threadIdx.x;
      const float p = j < items ? row[j] : 0.f;
      float incl = p;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) warp_tot[warp] = incl;
      __syncthreads();
      float before = run;
      for (int w = 0; w < warp; ++w) before += warp_tot[w];
      const float c = before + incl;
      if (j < items && p > 0.f && c > target) atomicMin(&found, j);
      __syncthreads();
      if (found < items) break;
      if (threadIdx.x == blockDim.x - 1) run = c;
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      int a = found;
      if (a >= items) {                 // u * total rounded past the last partial sum: the last possible outcome
        a = items - 1;
        while (a > 0 && !(row[a] > 0.f)) --a;
      }
      action[r] = a;
      logp[r] = clamped_log_prob(row[a] / total);
    }
    __syncthreads();
  }
}

// .log_prob(action) of given actions (models.py:142-143 with action_source {pi: beta}: the policy's log-prob of the
// behaviour policy's sample).  One warp per row.
__global__ void categorical_log_prob_kernel(const float* __restrict__ probs, long long ld, long long n, int items,
                                            const long long* __restrict__ action, float* __restrict__ logp, int* oob) {
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n) return;
  const int lane = threadIdx.x & 31;
  const float* row = probs + r * ld;
  float t = 0.f;
  for (int j = lane; j < items; j += 32) t += row[j];
  t = warp_sum(t);
  if (lane == 0) {
    const long long a = action[r];
    if (a < 0 || a >= items) {
      if (oob) *oob = 1;
      logp[r] = 0.f;
    } else {
      logp[r] = clamped_log_prob(row[a] / t);
    }
  }
}

// Row r's term L of the policy loss and g = dL / d log pi[a], from the probability pa = pi[a] of its drawn action (the
// closed forms at the top of this file).  Both the materialised and the item-streamed policy gradient call this.
__device__ __forceinline__ void reinforce_row_terms(float pa, long long r, const float* __restrict__ beta_logp,
                                                    const float* __restrict__ ret, int method, int K, float& L, float& g) {
  const float p = fminf(fmaxf(pa, kProbEps), 1.f - kProbEps);
  const bool inside = pa > kProbEps && pa < 1.f - kProbEps;       // the clamp has zero slope outside
  const float lp = logf(p), R = ret[r];
  if (method == RECNN_REINFORCE_BASIC) {
    L = -lp * R;
    g = -R;
  } else {
    const float c = p / expf(beta_logp[r]);
    if (method == RECNN_REINFORCE_CORRECTED) {
      L = c * -lp * R;
      g = -R * c * (lp + 1.f);
    } else {
      const float q = 1.f - p, Kf = (float)K;
      const float lam = Kf * powf(q, Kf - 1.f);
      const float dlam = K > 1 ? -Kf * (Kf - 1.f) * powf(q, Kf - 2.f) * p : 0.f;      // d lam / d lp
      L = lam * c * -lp * R;
      g = -R * c * (dlam * lp + lam * (lp + 1.f));
    }
  }
  if (!inside) g = 0.f;
}

// probabilities -> d loss / d logits, in place; row_loss[r] = this row's term of the policy loss.
__global__ void __launch_bounds__(kRowThreads)
reinforce_dlogits_kernel(float* __restrict__ z, long long ld, long long n, int items, const long long* __restrict__ action,
                         const float* __restrict__ beta_logp, const float* __restrict__ ret, int method, int K,
                         float* __restrict__ row_loss, int* oob) {
  __shared__ float s_g;
  for (long long r = blockIdx.x; r < n; r += gridDim.x) {
    float* row = z + r * ld;
    long long a = action[r];
    if (a < 0 || a >= items) {          // an id outside the policy's output layer: flagged, contributes nothing
      if (threadIdx.x == 0 && oob) *oob = 1;
      a = -1;
    }
    if (threadIdx.x == 0) {
      float g = 0.f, L = 0.f;
      if (a >= 0) reinforce_row_terms(row[a], r, beta_logp, ret, method, K, L, g);
      s_g = g;
      row_loss[r] = L;
    }
    __syncthreads();
    const float g = s_g;
    for (int j = threadIdx.x; j < items; j += blockDim.x) row[j] = g * ((j == a ? 1.f : 0.f) - row[j]);
    __syncthreads();
  }
}

// ---- item-streamed policy gradient: the logits of one item chunk at a time, per-row statistics in between
// Statistics pass, one chunk: z [n, cw] holds the logits of items c0 .. c0+cw.  Merges the chunk into the row's running
// max M and sum S of exp(z - M) (online softmax: M' = max(M, m_c), S' = S e^(M - M') + s_c e^(m_c - M')) and records the
// logit of the row's drawn action when it lies in the chunk.  One CTA per row; the reduction order is fixed.
__global__ void __launch_bounds__(kRowThreads)
reinforce_chunk_stats_kernel(const float* __restrict__ z, long long n, int cw, long long c0, int first,
                             const long long* __restrict__ action, float* __restrict__ row_max,
                             float* __restrict__ row_sum, float* __restrict__ za) {
  __shared__ float red[32];
  for (long long r = blockIdx.x; r < n; r += gridDim.x) {
    const float* row = z + r * cw;
    float m = -INFINITY, s = 0.f;
    for (int j = threadIdx.x; j < cw; j += blockDim.x) {      // as softmax_rows_kernel
      const float x = row[j];
      if (x > m) {
        s = s * __expf(m - x) + 1.f;
        m = x;
      } else {
        s += __expf(x - m);
      }
    }
    const float mc = block_max(m, red);
    s = (m == -INFINITY) ? 0.f : s * __expf(m - mc);
    const float sc = block_sum(s, red);
    if (threadIdx.x == 0) {
      if (first) {
        row_max[r] = mc;
        row_sum[r] = sc;
      } else {
        const float M = row_max[r], M2 = fmaxf(M, mc);
        row_sum[r] = row_sum[r] * __expf(M - M2) + sc * __expf(mc - M2);
        row_max[r] = M2;
      }
      const long long a = action[r] - c0;
      if (a >= 0 && a < cw) za[r] = row[a];
    }
    __syncthreads();
  }
}

// After the statistics pass: pi[a] = exp(z_a - M) / S, the row's loss term and g = dL / d log pi[a].  One thread per row.
__global__ void reinforce_streamed_terms_kernel(long long n, int items, const long long* __restrict__ action,
                                                const float* __restrict__ row_max, const float* __restrict__ row_sum,
                                                const float* __restrict__ za, const float* __restrict__ beta_logp,
                                                const float* __restrict__ ret, int method, int K,
                                                float* __restrict__ row_loss, float* __restrict__ row_g, int* oob) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const long long a = action[r];
  float L = 0.f, g = 0.f;
  if (a < 0 || a >= items) {            // an id outside the policy's output layer: flagged, contributes nothing
    if (oob) *oob = 1;
  } else {
    reinforce_row_terms(expf(za[r] - row_max[r]) / row_sum[r], r, beta_logp, ret, method, K, L, g);
  }
  row_loss[r] = L;
  row_g[r] = g;
}

// out[0] = sum of v[0..n) in a fixed order (one CTA)
__global__ void __launch_bounds__(1024) sum_rows_kernel(const float* __restrict__ v, long long n, float* __restrict__ out) {
  __shared__ float red[32];
  float t = 0.f;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) t += v[i];
  t = block_sum(t, red);
  if (threadIdx.x == 0) out[0] = t;
}

static int row_grid(int64_t n) { return (int)(n < (int64_t)kNumSMs * 8 ? n : (int64_t)kNumSMs * 8); }

// split-K partial space of the two weight gradients of the policy (either back end)
static int64_t reinforce_partial_floats(const recnn_discrete_dims& d, int64_t rows) {
  int64_t best = 0;
  const int shapes[2][2] = {{d.num_items, d.hidden}, {d.hidden, d.state_dim}};
  for (auto& s : shapes)
    for (int tcp = 0; tcp < 2; ++tcp) {
      const int64_t f = (int64_t)dw_splits(s[0], s[1], rows, tcp != 0) * s[0] * (s[1] + 1);
      if (f > best) best = f;
    }
  return best;
}

// Split-K partial space of the item-streamed policy gradient: dW1, and dW2 of one chunk of every width up to `chunk`
// (the last chunk may be narrower, and the split count depends on the width).  The split count is constant over
// each run of 128 widths, so the widest of each run bounds it.  Independent of num_items.
static int64_t streamed_partial_floats(const recnn_discrete_dims& d, int64_t rows, int chunk) {
  int64_t best = 0;
  for (int64_t top = 128;; top += 128) {
    const int cw = (int)(top < chunk ? top : chunk);
    for (int tcp = 0; tcp < 2; ++tcp) {
      const int64_t f = (int64_t)dw_splits(cw, d.hidden, rows, tcp != 0) * cw * (d.hidden + 1);
      if (f > best) best = f;
    }
    if (top >= chunk) break;
  }
  for (int tcp = 0; tcp < 2; ++tcp) {
    const int64_t f = (int64_t)dw_splits(d.hidden, d.state_dim, rows, tcp != 0) * d.hidden * (d.state_dim + 1);
    if (f > best) best = f;
  }
  return best;
}

struct DiscreteScratch {
  float *img, *h, *z, *dh, *row_loss, *partial;
  float *row_max, *row_sum, *za, *row_g;     // item-streamed gradient only
  int* flags;
  int64_t floats;
};
// item_chunk > 0 (backward only): the item-streamed gradient, z holds one chunk of logits [n, item_chunk]
static DiscreteScratch discrete_carve(const recnn_discrete_dims& d, int64_t n, bool backward, float* base,
                                      int item_chunk = 0) {
  DiscreteScratch s;
  int64_t off = 0;
  auto take = [&](int64_t floats) {
    float* r = base ? base + off : nullptr;
    off += round_up(floats, 64);
    return r;
  };
  s.img = take(n * pad4(d.state_dim));
  s.h = take(n * d.hidden);
  s.flags = reinterpret_cast<int*>(take(4));
  s.z = s.dh = s.row_loss = s.partial = nullptr;
  s.row_max = s.row_sum = s.za = s.row_g = nullptr;
  if (backward) {
    const int chunk = item_chunk > 0 && item_chunk < d.num_items ? item_chunk : d.num_items;
    s.z = take(n * (int64_t)chunk);
    s.dh = take(n * d.hidden);
    s.row_loss = take(n);
    if (item_chunk > 0) {
      s.row_max = take(n);
      s.row_sum = take(n);
      s.za = take(n);
      s.row_g = take(n);
      s.partial = take(streamed_partial_floats(d, n, chunk));
    } else {
      s.partial = take(reinforce_partial_floats(d, n));
    }
  }
  s.floats = off + 64;
  return s;
}
static float* align_floats(float* p) {      // 256-byte aligned start inside the caller's scratch
  return reinterpret_cast<float*>(round_up(reinterpret_cast<int64_t>(p), 256));
}

// h = relu(W1 s + b1) into s.h, kept for the backward
static int discrete_hidden(const recnn_discrete_dims& d, const float* params, const float* state, int64_t n,
                           const DiscreteScratch& s, cudaStream_t st, Seg* xs_out) {
  const DiscreteLayout l = discrete_layout(d);
  recnn_dims dd;
  memset(&dd, 0, sizeof(dd));
  dd.state_dim = d.state_dim; dd.hidden = d.hidden; dd.action_dim = d.num_items;
  Seg xs;
  RECNN_PROPAGATE(repitch_state(dd, state, n, s.img, &xs, st));
  if (xs_out) *xs_out = xs;
  Rng rng = {nullptr, 0, nullptr};
  return hidden_layer(xs, kNoSeg, params + l.w1, l.ld1, params + l.b1, d.hidden, n, false, nullptr, rng, 0, s.h, st);
}

// logits = W2 relu(W1 s + b1) + b2 into z (row pitch num_items); h kept for the backward
static int discrete_logits(const recnn_discrete_dims& d, const float* params, const float* state, int64_t n,
                           const DiscreteScratch& s, float* z, cudaStream_t st, Seg* xs_out) {
  const DiscreteLayout l = discrete_layout(d);
  const int H = d.hidden;
  RECNN_PROPAGATE(discrete_hidden(d, params, state, n, s, st, xs_out));
  const Seg sh = {s.h, H, H, 0};
  return linear_out(sh, params + l.w2, l.ld2, params + l.b2, d.num_items, n, 0, nullptr, z, d.num_items, st);
}

// The logit GEMM of items [c0, c0 + cw) into s.z [n, cw] with epilogue EPI: EPI_LINEAR (the logits, as linear_out) or
// EPI_DLOGITS (d loss / d logits).  Both passes of the streamed gradient run this one GEMM on the same operands without
// split-K, so the logits the backward recomputes are bit-identical to those the statistics were taken from.
template <int EPI>
static int item_chunk_gemm(const recnn_discrete_dims& d, const float* params, const DiscreteScratch& s, int64_t n,
                           int64_t c0, int cw, Epilogue e, cudaStream_t st) {
  const DiscreteLayout l = discrete_layout(d);
  const Seg sh = {s.h, d.hidden, d.hidden, 0};
  e.out = s.z; e.ldo = cw; e.bias = params + l.b2 + c0;
  return gemm_nt<EPI>(sh, kNoSeg, params + l.w2 + c0 * l.ld2, l.ld2, cw, n, e, st);
}

}  // namespace recnn

using namespace recnn;

static bool discrete_dims_ok(const recnn_discrete_dims* d) {
  return d && d->state_dim > 0 && d->hidden > 0 && d->num_items > 0;
}

extern "C" int recnn_discrete_layout(const recnn_discrete_dims* d, int64_t* out) {
  RECNN_REQUIRE(discrete_dims_ok(d) && out, "dims / out");
  const DiscreteLayout l = discrete_layout(*d);
  out[0] = l.w1; out[1] = l.b1; out[2] = l.w2; out[3] = l.b2; out[4] = l.ld1; out[5] = l.ld2; out[6] = l.count;
  return RECNN_OK;
}

extern "C" int64_t recnn_discrete_scratch_floats(const recnn_discrete_dims* d, int64_t n_rows, int32_t backward) {
  if (!discrete_dims_ok(d) || n_rows <= 0) return 0;
  return discrete_carve(*d, n_rows, backward != 0, nullptr).floats;
}

extern "C" int recnn_discrete_forward(const recnn_discrete_dims* d, const float* params, const float* state,
                                      int64_t n_rows, float* probs_out, float* scratch, void* stream) {
  RECNN_REQUIRE(discrete_dims_ok(d) && params && state && probs_out && scratch, "null pointer / dims");
  if (n_rows <= 0) return RECNN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const DiscreteScratch s = discrete_carve(*d, n_rows, false, align_floats(scratch));
  RECNN_PROPAGATE(discrete_logits(*d, params, state, n_rows, s, probs_out, st, nullptr));
  softmax_rows_kernel<<<row_grid(n_rows), kRowThreads, 0, st>>>(probs_out, d->num_items, n_rows, d->num_items);
  RECNN_CHECK_LAUNCH("softmax_rows_kernel");
  return RECNN_OK;
}

extern "C" int recnn_categorical_sample(const float* probs, int64_t n_rows, int32_t num_items, int64_t ld,
                                        const float* uniforms, uint64_t seed, int64_t draw, int64_t* action_out,
                                        float* log_prob_out, void* stream) {
  RECNN_REQUIRE(probs && action_out && log_prob_out, "null pointer");
  RECNN_REQUIRE(num_items > 0 && ld >= num_items, "num_items / ld");
  if (n_rows <= 0) return RECNN_OK;
  categorical_sample_kernel<<<row_grid(n_rows), kRowThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      probs, ld, n_rows, num_items, uniforms, seed, draw, reinterpret_cast<long long*>(action_out), log_prob_out);
  RECNN_CHECK_LAUNCH("categorical_sample_kernel");
  return RECNN_OK;
}

extern "C" int recnn_categorical_log_prob(const float* probs, int64_t n_rows, int32_t num_items, int64_t ld,
                                          const int64_t* action, float* log_prob_out, int32_t* oob_flag, void* stream) {
  RECNN_REQUIRE(probs && action && log_prob_out, "null pointer");
  RECNN_REQUIRE(num_items > 0 && ld >= num_items, "num_items / ld");
  if (n_rows <= 0) return RECNN_OK;
  const int warps = 8;
  categorical_log_prob_kernel<<<(unsigned)ceil_div(n_rows, warps), warps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      probs, ld, n_rows, num_items, reinterpret_cast<const long long*>(action), log_prob_out, oob_flag);
  RECNN_CHECK_LAUNCH("categorical_log_prob_kernel");
  return RECNN_OK;
}

// out[0] = policy loss, out[1] = 1.0 if an action id was outside [0, num_items) (that row contributes nothing)
static int reinforce_args_ok(const recnn_discrete_dims* d, const float* params, float* grads, const float* state,
                             const int64_t* action, const float* beta_log_prob, const float* returns, int64_t n_rows,
                             int32_t method, int32_t top_k, float* out, float* scratch) {
  RECNN_REQUIRE(discrete_dims_ok(d) && params && grads && state && action && returns && out && scratch,
                "null pointer / dims");
  RECNN_REQUIRE(method == RECNN_REINFORCE_BASIC || method == RECNN_REINFORCE_CORRECTED || method == RECNN_REINFORCE_TOPK,
                "unknown REINFORCE method");
  RECNN_REQUIRE(method == RECNN_REINFORCE_BASIC || beta_log_prob, "the corrected losses need the behaviour policy's log-probs");
  RECNN_REQUIRE(method != RECNN_REINFORCE_TOPK || top_k >= 1, "K >= 1");
  RECNN_REQUIRE(n_rows > 0, "no saved rows: select_action was never called since the last update");
  return RECNN_OK;
}

extern "C" int recnn_reinforce_policy_grad(const recnn_discrete_dims* d, const float* params, float* grads,
                                           const float* state, const int64_t* action, const float* beta_log_prob,
                                           const float* returns, int64_t n_rows, int32_t method, int32_t top_k,
                                           float* out, float* scratch, void* stream) {
  RECNN_PROPAGATE(reinforce_args_ok(d, params, grads, state, action, beta_log_prob, returns, n_rows, method, top_k, out,
                                    scratch));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const DiscreteLayout l = discrete_layout(*d);
  const int H = d->hidden, S = d->state_dim, I = d->num_items;
  const DiscreteScratch s = discrete_carve(*d, n_rows, true, align_floats(scratch));
  RECNN_CHECK_CUDA(cudaMemsetAsync(s.flags, 0, 4 * sizeof(int), st));
  Seg xs;
  RECNN_PROPAGATE(discrete_logits(*d, params, state, n_rows, s, s.z, st, &xs));
  softmax_rows_kernel<<<row_grid(n_rows), kRowThreads, 0, st>>>(s.z, I, n_rows, I);
  RECNN_CHECK_LAUNCH("softmax_rows_kernel");
  reinforce_dlogits_kernel<<<row_grid(n_rows), kRowThreads, 0, st>>>(s.z, I, n_rows, I, reinterpret_cast<const long long*>(action),
                                                                    beta_log_prob, returns, method, top_k, s.row_loss, s.flags);
  RECNN_CHECK_LAUNCH("reinforce_dlogits_kernel");
  sum_rows_kernel<<<1, 1024, 0, st>>>(s.row_loss, n_rows, out);
  RECNN_CHECK_LAUNCH("sum_rows_kernel");
  // backward: dW2 = dz^T h, db2 = colsum dz; dh = (dz W2) * [h > 0]; dW1 = dh^T s, db1 = colsum dh
  const Seg sh = {s.h, H, H, 0};
  RECNN_PROPAGATE(weight_grad(s.z, I, sh, kNoSeg, n_rows, grads + l.w2, l.ld2, grads + l.b2, s.partial, st));
  RECNN_PROPAGATE(backprop_hidden(s.z, I, params + l.w2, l.ld2, H, 0, H, n_rows, s.h, 1.f, s.dh, st));
  RECNN_PROPAGATE(weight_grad(s.dh, H, xs, kNoSeg, n_rows, grads + l.w1, l.ld1, grads + l.b1, s.partial, st));
  (void)S;
  RECNN_CHECK_CUDA(cudaMemcpyAsync(out + 1, s.flags, sizeof(int), cudaMemcpyDeviceToDevice, st));
  return RECNN_OK;
}

extern "C" int64_t recnn_reinforce_streamed_scratch_floats(const recnn_discrete_dims* d, int64_t n_rows,
                                                           int32_t item_chunk) {
  if (!discrete_dims_ok(d) || n_rows <= 0 || item_chunk < 1) return 0;
  return discrete_carve(*d, n_rows, true, nullptr, item_chunk).floats;
}

// recnn_reinforce_policy_grad without the [n_rows, num_items] logits: two passes over the item chunks [c0, c0 + C),
// each recomputing the chunk's logits with the same GEMM.  Pass 1 takes each row's softmax statistics and the logit of
// its action; pass 2 writes d logits straight from the GEMM epilogue and consumes them chunk by chunk.
extern "C" int recnn_reinforce_policy_grad_streamed(const recnn_discrete_dims* d, const float* params, float* grads,
                                                    const float* state, const int64_t* action,
                                                    const float* beta_log_prob, const float* returns, int64_t n_rows,
                                                    int32_t method, int32_t top_k, int32_t item_chunk, float* out,
                                                    float* scratch, void* stream) {
  RECNN_PROPAGATE(reinforce_args_ok(d, params, grads, state, action, beta_log_prob, returns, n_rows, method, top_k, out,
                                    scratch));
  RECNN_REQUIRE(item_chunk >= 1, "item_chunk >= 1");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const DiscreteLayout l = discrete_layout(*d);
  const int H = d->hidden, I = d->num_items;
  const int C = item_chunk < I ? item_chunk : I;
  const long long* act = reinterpret_cast<const long long*>(action);
  const DiscreteScratch s = discrete_carve(*d, n_rows, true, align_floats(scratch), item_chunk);
  RECNN_CHECK_CUDA(cudaMemsetAsync(s.flags, 0, 4 * sizeof(int), st));
  Seg xs;
  RECNN_PROPAGATE(discrete_hidden(*d, params, state, n_rows, s, st, &xs));
  // pass 1: per-row max, sum of exp and the action's logit over all items
  for (int64_t c0 = 0; c0 < I; c0 += C) {
    const int cw = (int)(I - c0 < C ? I - c0 : C);
    RECNN_PROPAGATE(item_chunk_gemm<EPI_LINEAR>(*d, params, s, n_rows, c0, cw, base_epi(), st));
    reinforce_chunk_stats_kernel<<<row_grid(n_rows), kRowThreads, 0, st>>>(s.z, n_rows, cw, c0, c0 == 0, act, s.row_max,
                                                                          s.row_sum, s.za);
    RECNN_CHECK_LAUNCH("reinforce_chunk_stats_kernel");
  }
  reinforce_streamed_terms_kernel<<<(unsigned)ceil_div(n_rows, 256), 256, 0, st>>>(
      n_rows, I, act, s.row_max, s.row_sum, s.za, beta_log_prob, returns, method, top_k, s.row_loss, s.row_g, s.flags);
  RECNN_CHECK_LAUNCH("reinforce_streamed_terms_kernel");
  sum_rows_kernel<<<1, 1024, 0, st>>>(s.row_loss, n_rows, out);
  RECNN_CHECK_LAUNCH("sum_rows_kernel");
  // pass 2, per chunk: dz = d loss / d logits from the recomputed logits; dW2, db2 of the chunk's items;
  // dh = sum over chunks of dz W2[chunk], gated by [h > 0] with the last chunk
  const Seg sh = {s.h, H, H, 0};
  Epilogue e = base_epi();
  e.row_g = s.row_g; e.row_max = s.row_max; e.row_sum = s.row_sum; e.row_action = act;
  for (int64_t c0 = 0; c0 < I; c0 += C) {
    const int cw = (int)(I - c0 < C ? I - c0 : C);
    const bool last = c0 + cw >= I;
    e.col0 = c0;
    RECNN_PROPAGATE(item_chunk_gemm<EPI_DLOGITS>(*d, params, s, n_rows, c0, cw, e, st));
    RECNN_PROPAGATE(weight_grad(s.z, cw, sh, kNoSeg, n_rows, grads + l.w2 + c0 * l.ld2, l.ld2, grads + l.b2 + c0,
                                s.partial, st));
    RECNN_PROPAGATE(backprop_hidden(s.z, cw, params + l.w2 + c0 * l.ld2, l.ld2, H, 0, H, n_rows, last ? s.h : nullptr,
                                    1.f, s.dh, st, c0 > 0));
  }
  // dW1 = dh^T s, db1 = colsum dh
  RECNN_PROPAGATE(weight_grad(s.dh, H, xs, kNoSeg, n_rows, grads + l.w1, l.ld1, grads + l.b1, s.partial, st));
  RECNN_CHECK_CUDA(cudaMemcpyAsync(out + 1, s.flags, sizeof(int), cudaMemcpyDeviceToDevice, st));
  return RECNN_OK;
}
