// Orchestration of the DDPG / TD3 update step on one GPU (one rank's shard).
// Restates recnn/nn/update/ddpg.py:8-104, misc.py:10-55 and td3.py:8-150 as a
// fixed sequence of kernel launches on the caller's stream: no allocation, no
// synchronisation, no host read-back -- so the whole call is CUDA-graph
// capturable.  Step-dependent scalars (Adam's t, the Philox step) live on the
// device for the same reason.
//
// Every contraction goes through one of four helpers (hidden_layer, linear_out,
// backprop_hidden, weight_grad).  Each has two back ends with identical
// semantics: the tcgen05 3xTF32 tensor-core kernel (tc_gemm.cuh; default) and
// the exact-fp32 CUDA-core kernel (gemm_simt.cuh; arbitrary shapes, and
// RECNN_B200_MATH=simt forces it for A/B comparisons).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "pointwise.cuh"
#include "tc_gemm.cuh"

namespace recnn {

int launch_frame_gather(const float* table, int64_t n_items, int dim, const int64_t* items, const float* ratings,
                        int64_t n_rows, int frame, int64_t s_ld, int64_t a_ld, float* state, float* next_state,
                        float* action, float* reward, int* oob_flag, cudaStream_t st);

static bool math_tc() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RECNN_B200_MATH");
    v = (e && strcmp(e, "simt") == 0) ? 0 : 1;
  }
  return v == 1;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---------------------------------------------------------------- intra-step concurrency
// The three forward chains at the head of a step are independent: (T) target policy -> target critic
// -> TD target, (V) online critic forward, (P) online policy forward.  Each GEMM fills at most 64-128
// of the 148 SMs, so they are issued on three streams (fork/join with events; capturable into the
// step's CUDA graph).  RECNN_B200_OVERLAP=0 serialises everything on the caller's stream.
struct AuxStreams {
  cudaStream_t sv, sp, sw;
  cudaEvent_t fork, v_done, p_done;
  cudaEvent_t ev[9];       // fork/join pairs: 0-3 weight-gradient GEMMs, 4 chain P, 5-8 TD3's second critic
  bool ok;
};
static AuxStreams* aux_streams() {
  static AuxStreams per_dev[64];
  static bool init[64] = {false};
  static const bool enabled = !(getenv("RECNN_B200_OVERLAP") && strcmp(getenv("RECNN_B200_OVERLAP"), "0") == 0);
  if (!enabled) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  AuxStreams& a = per_dev[dev];
  if (!init[dev]) {
    // never created while a capture is in flight: the first call of a shape is always a direct launch
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    (void)cs;
    a.ok = cudaStreamCreateWithFlags(&a.sv, cudaStreamNonBlocking) == cudaSuccess &&
           cudaStreamCreateWithFlags(&a.sp, cudaStreamNonBlocking) == cudaSuccess &&
           cudaStreamCreateWithFlags(&a.sw, cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&a.v_done, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&a.p_done, cudaEventDisableTiming) == cudaSuccess;
    for (auto& e : a.ev) a.ok = a.ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    init[dev] = true;
  }
  return a.ok ? &a : nullptr;
}

// ---------------------------------------------------------------- workspace
struct Workspace {
  float* S;        // [N, ldS] state (frame form: gathered; dense form: re-pitched copy)
  float* S2;       // [N, ldS]
  float* ACT;      // [N, ldA] batch action, stored with `lead` zero columns in front (see Seg)
  float* REW;      // [N]
  float* hb[12];   // [N,H] activation / gradient buffers (lifetimes in DESIGN.md); 8..11: TD3's second critic (target hidden, online hidden)
  float* ab[3];    // [N, ldA] next_action / gen_action (lead-padded) ; [N,A] d gen_action
  float* y;        // [N] TD target
  float* qtmp;     // [N]
  float* dq;       // [N]
  float* partial;  // split-K partials of the largest weight gradient
  float* partial2; // second partial buffer (hidden x hidden sized) so two weight gradients can be in flight
  float* block_partials;  // [1024]
  float* scalars;         // [8]: 0 = clip coef
  unsigned* tickets;      // [8]
  int64_t bytes;
};

// split count of a weight-gradient GEMM dW[C, K] = dZ^T X over n_rows (the contraction dim).
// Must be a pure function of the shapes: the workspace size depends on it.
// The tensor-core kernel holds one CTA per SM and has a fixed cost of several microseconds, so more CTAs than SMs
// means a second wave of the whole fixed cost (measured in round 1: the critic's dW1 as 22+4 tiles x 8 splits = 208
// CTAs took 48 us = two waves); aim at ONE wave of ~132 CTAs, leaving room for the GEMM that runs beside it.
static int dw_splits(int C, int K, int64_t n_rows, bool tc_path, int bn = 128) {
  if (tc_path) {
    const int64_t tiles = ceil_div(C, 128) * ceil_div(K, bn);
    int64_t s = 132 / tiles > 0 ? 132 / tiles : 1;
    const int64_t max_s = ceil_div(n_rows, 32) / 4 > 0 ? ceil_div(n_rows, 32) / 4 : 1;   // >= 4 k-blocks (128 rows) per split
    if (s > max_s) s = max_s;
    return (int)(s < 1 ? 1 : s);
  }
  const int64_t tiles = ceil_div(C, 128) * ceil_div(K + 1, 128);
  int64_t s = ceil_div(220, tiles);
  const int64_t max_s = n_rows / 256 > 0 ? n_rows / 256 : 1;
  if (s > max_s) s = max_s;
  return (int)(s < 1 ? 1 : s);
}

static int64_t partial_floats(const recnn_dims& d, int64_t n_rows) {
  const int in_c = d.state_dim + d.action_dim;
  int64_t best = 0;
  const int shapes[5][2] = {{d.hidden, in_c}, {d.hidden, d.state_dim}, {d.hidden, d.hidden},
                            {d.action_dim, d.hidden}, {1, d.hidden}};
  for (auto& s : shapes)
    for (int tcp = 0; tcp < 2; ++tcp) {
      const int64_t f = (int64_t)dw_splits(s[0], s[1], n_rows, tcp != 0) * s[0] * (s[1] + 1);
      if (f > best) best = f;
    }
  const int64_t head = (int64_t)kNumSMs * (d.hidden + 2);     // block partials of the fused value-head kernel
  return best > head ? best : head;
}

static Workspace carve(const recnn_dims& d, int64_t n, void* base) {
  Workspace w;
  char* p = static_cast<char*>(base);
  int64_t off = 0;
  auto take = [&](int64_t floats) {
    float* r = base ? reinterpret_cast<float*>(p + off) : nullptr;
    off += round_up(floats * 4, 256);
    return r;
  };
  const int ldS = pad4(d.state_dim);
  const int ldA = pad4(d.action_dim + d.state_dim % 4);
  w.S = take(n * ldS);
  w.S2 = take(n * ldS);
  w.ACT = take(n * ldA);
  w.REW = take(n);
  for (auto& b : w.hb) b = take(n * d.hidden);
  for (auto& b : w.ab) b = take(n * ldA);
  w.y = take(n);
  w.qtmp = take(n);
  w.dq = take(n);
  w.partial = take(partial_floats(d, n));
  {
    int64_t f2 = 0;
    const int shp[2][2] = {{d.hidden, d.hidden}, {d.action_dim, d.hidden}};
    for (auto& s2 : shp)
      for (int tcp = 0; tcp < 2; ++tcp) {
        const int64_t f = (int64_t)dw_splits(s2[0], s2[1], n, tcp != 0) * s2[0] * (s2[1] + 1);
        if (f > f2) f2 = f;
      }
    w.partial2 = take(f2);
  }
  w.block_partials = take(1024);
  w.scalars = take(8);
  w.tickets = reinterpret_cast<unsigned*>(take(8));
  w.bytes = off;
  return w;
}

// ---------------------------------------------------------------- building blocks
struct Rng {
  const uint8_t* const* masks;
  unsigned long long seed;
  const long long* step;
};

static Epilogue base_epi() {
  Epilogue e;
  memset(&e, 0, sizeof(e));
  e.gate_scale = 1.f;
  return e;
}

// one K-contiguous input matrix [n, cols] with row pitch ld.  `lead` of its columns are zero pads in
// front of the data: TMA needs every box to start on a 16-byte boundary in BOTH operands, and the
// critic's concat [state | action] puts the action block at weight column S = 1290 (8 mod 16 bytes).
// Storing actions with S%4 leading zeros lets the second K-segment start at weight column S - lead,
// which is aligned; the pad columns multiply state weights by zero.
struct Seg {
  const float* p;
  int cols;          // including the lead pads
  long long ld;
  int lead;
};
static const Seg kNoSeg = {nullptr, 0, 0, 0};

// GEMMs that run alone on the GPU (nothing to overlap with) prefer 64-wide tiles: twice the CTAs.
static thread_local bool t_alone = false;
struct AloneScope {
  bool prev;
  explicit AloneScope(bool on) : prev(t_alone) { t_alone = on; }
  ~AloneScope() { t_alone = prev; }
};

static int pick_bn(int64_t M, int N) {
  // 128-wide tiles when they still yield >= 64 CTAs; otherwise 64-wide (more CTAs, less reuse)
  const int64_t mt = ceil_div(M, 128);
  if (t_alone && mt * ceil_div(N, 64) <= 2 * kNumSMs) return 64;
  if (N > 64 && mt * ceil_div(N, 128) >= 64) return 128;
  return 64;
}

// out[n, N] = epi( [x0 | x1] W^T )    W is [N, K0+K1] with row pitch ldw
template <int EPI>
static int gemm_nt(const Seg& x0, const Seg& x1, const float* W, long long ldw, int N, int64_t n, const Epilogue& e,
                   cudaStream_t st) {
  const int K = x0.cols + x1.cols - x1.lead;             // logical contraction length == W's columns
  const bool tc_ok = math_tc() && aligned16(x0.p) && (x1.cols == 0 || aligned16(x1.p)) && aligned16(W) &&
                     x0.ld % 4 == 0 && (x1.cols == 0 || x1.ld % 4 == 0) && ldw % 4 == 0 && x0.lead == 0 &&
                     (x1.cols == 0 || (x0.cols - x1.lead) % 4 == 0);
  if (tc_ok) {
    tc::Operand a0 = {x0.p, x0.ld, 0, 0}, a1 = {x1.p, x1.ld, 0, 0}, b = {W, ldw, N, K};
    tc::Problem p;
    memset(&p, 0, sizeof(p));
    p.M = (int)n; p.N = N; p.K0 = x0.cols; p.K1 = x1.cols; p.b_k1_offset = x0.cols - x1.lead;
    const int r = tc::launch<false, false, EPI>(a0, a1, b, p, 1, pick_bn(n, N), e, st);
    return r < 0 ? r : RECNN_OK;
  }
  const MatView X = x1.cols ? mat_cat(x0.p + x0.lead, x0.ld, x0.cols - x0.lead, x1.p + x1.lead, x1.ld)
                            : mat(x0.p + x0.lead, x0.ld);
  return launch_gemm_simt<true, true, EPI>(X, mat(W, ldw), (int)n, N, K, 1, e, st);
}

// h = dropout(relu([x0|x1] W^T + b))
static int hidden_layer(const Seg& x0, const Seg& x1, const float* W, long long ldw, const float* b, int H,
                        int64_t n, bool train, const uint8_t* mask, const Rng& rng, unsigned stream_id, float* out,
                        cudaStream_t st) {
  Epilogue e = base_epi();
  e.out = out; e.ldo = H; e.bias = b;
  e.train = train ? 1 : 0; e.mask = mask; e.seed = rng.seed; e.rng_step = rng.step; e.stream_id = stream_id;
  return gemm_nt<EPI_HIDDEN>(x0, x1, W, ldw, H, n, e, st);
}

struct NoiseSpec {
  int add; const float* noise; float clip, std; unsigned long long seed; const long long* step; unsigned stream_id;
};

static int linear_out(const Seg& x, const float* W, long long ldw, const float* b, int out_dim, int64_t n,
                      int apply_tanh, const NoiseSpec* nz, float* out, long long ldo, cudaStream_t st) {
  Epilogue e = base_epi();
  e.out = out; e.ldo = ldo; e.bias = b; e.apply_tanh = apply_tanh;
  if (nz && nz->add) {
    e.add_noise = 1; e.noise = nz->noise; e.noise_clip = nz->clip; e.noise_std = nz->std;
    e.seed = nz->seed; e.rng_step = nz->step; e.stream_id = nz->stream_id;
  }
  return gemm_nt<EPI_LINEAR>(x, kNoSeg, W, ldw, out_dim, n, e, st);
}

// dX = (dZ W[:, col0:col0+K]) * gate(h)     dZ [n,C]; W [C, w_cols] row pitch ldw; out [n,K]
// accumulate: dX = (out + dZ W[...]) * gate(h), i.e. one more term of a sum over blocks of C (gated by the last term)
static int backprop_hidden(const float* dZ, int C, const float* W, long long ldw, int w_cols, int col0, int K,
                           int64_t n, const float* h, float gate_scale, float* out, cudaStream_t st,
                           bool accumulate = false) {
  Epilogue e = base_epi();
  e.out = out; e.ldo = K; e.h = h; e.ldh = K; e.gate_scale = gate_scale;
  const bool tc_ok = math_tc() && aligned16(dZ) && aligned16(W) && C % 4 == 0 && ldw % 4 == 0 && col0 % 4 == 0;
  if (tc_ok) {
    tc::Operand a0 = {dZ, C, 0, 0}, a1 = {nullptr, 0, 0, 0}, b = {W, ldw, C, w_cols};
    tc::Problem p;
    memset(&p, 0, sizeof(p));
    p.M = (int)n; p.N = K; p.K0 = C; p.b_k1_offset = C; p.b_n_offset = col0;
    const int bn = pick_bn(n, K);
    const int r = accumulate ? tc::launch<false, true, EPI_ACCUM>(a0, a1, b, p, 1, bn, e, st)
                  : h ? tc::launch<false, true, EPI_GATE>(a0, a1, b, p, 1, bn, e, st)
                      : tc::launch<false, true, EPI_STORE>(a0, a1, b, p, 1, bn, e, st);
    return r < 0 ? r : RECNN_OK;
  }
  if (accumulate) return launch_gemm_simt<true, false, EPI_ACCUM>(mat(dZ, C), mat(W + col0, ldw), (int)n, K, C, 1, e, st);
  if (h) return launch_gemm_simt<true, false, EPI_GATE>(mat(dZ, C), mat(W + col0, ldw), (int)n, K, C, 1, e, st);
  return launch_gemm_simt<true, false, EPI_STORE>(mat(dZ, C), mat(W + col0, ldw), (int)n, K, C, 1, e, st);
}

// dW[c,k] = sum_n dZ[n,c] [x0|x1][n,k];  db[c] = sum_n dZ[n,c].   dW has row pitch ldw.
struct SideLaunch {        // run the second K-segment's GEMM on `stream`, fork/join with these events
  cudaStream_t stream;
  cudaEvent_t fork, join;
};

// `defer` (with the gradient arena's base): do not reduce the split-K partials here; describe them instead, for the
// optimizer / all-reduce pass that consumes them directly (GradSource).
static int weight_grad(const float* dZ, int C, const Seg& x0, const Seg& x1, int64_t n, float* dW, long long ldw,
                       float* db, float* partial, cudaStream_t st, const SideLaunch* side = nullptr,
                       PartialLayer* defer = nullptr, const float* grads_base = nullptr) {
  const int K = x0.cols + x1.cols - x1.lead, K1 = K + 1;
  Epilogue e = base_epi();
  e.out = partial; e.ldo = K1;
  const bool tc_ok = math_tc() && C % 4 == 0 && C >= 32 && aligned16(dZ) && aligned16(x0.p) && x0.ld % 4 == 0 &&
                     x0.lead == 0 && (x1.cols == 0 || (aligned16(x1.p) && x1.ld % 4 == 0));
  if (tc_ok) {
    const int req = dw_splits(C, K, n, true);
    int k_chunk = 0;
    const int splits = tc::split_plan((int)ceil_div(n, 32), req, &k_chunk, 32);
    tc::Operand a0 = {dZ, C, 0, 0}, a1 = {nullptr, 0, 0, 0};
    // the padded second segment's window starts `lead` columns inside the first segment's; those pad
    // columns are computed (as zeros) but not stored (n_skip), so the two GEMMs are independent
    const Seg* segs[2] = {&x1, &x0};
    const int cols0[2] = {x0.cols - x1.lead, 0};
    const bool use_side = side && x1.cols > 0;
    if (use_side) {
      RECNN_CHECK_CUDA(cudaEventRecord(side->fork, st));
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    }
    for (int i = 0; i < 2; ++i) {
      const Seg* s = segs[i];
      if (s->cols == 0) continue;
      tc::Operand b = {s->p, s->ld, n, s->cols};
      tc::Problem p;
      memset(&p, 0, sizeof(p));
      p.M = C; p.N = s->cols; p.K0 = (int)n; p.n_out_offset = cols0[i]; p.n_skip = i == 0 ? x1.lead : 0;
      const int bn = s->cols > 64 ? 128 : 64;
      const int r = tc::launch<true, true, EPI_PARTIAL>(a0, a1, b, p, req, bn, e, (i == 0 && use_side) ? side->stream : st);
      if (r < 0) return r;
      if (r != splits) {
        set_error("internal: split plan mismatch (%d vs %d)", r, splits);
        return RECNN_E_INVALID;
      }
    }
    // the bias column of the partials (column sums of dZ) only reads dZ: with a side stream it runs there, behind the
    // short action-segment GEMM and beside the long state-segment GEMM, instead of after both
    const bool colsum_on_side = use_side;
    if (colsum_on_side) RECNN_PROPAGATE(launch_colsum_partials(dZ, n, C, k_chunk, splits, partial, K1, side->stream));
    if (use_side) {
      RECNN_CHECK_CUDA(cudaEventRecord(side->join, side->stream));
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(st, side->join, 0));
    }
    if (!colsum_on_side) RECNN_PROPAGATE(launch_colsum_partials(dZ, n, C, k_chunk, splits, partial, K1, st));
    if (defer) {
      *defer = PartialLayer{partial, splits, C, K1, (int)ldw, (long long)(dW - grads_base), (long long)(db - grads_base)};
      return RECNN_OK;
    }
    return launch_reduce_partials(partial, splits, C, K1, dW, ldw, db, st);
  }
  MatView X = x1.cols ? mat_cat(x0.p + x0.lead, x0.ld, x0.cols - x0.lead, x1.p + x1.lead, x1.ld)
                      : mat(x0.p + x0.lead, x0.ld);
  X.ones_at = K;                        // virtual bias column
  const int splits_req = dw_splits(C, K, n, false);
  // the launcher rounds the chunk; recompute the effective split count the same way
  const int k_chunk = (int)round_up(ceil_div(n, splits_req), 16);
  const int splits = (int)ceil_div(n, k_chunk);
  RECNN_PROPAGATE((launch_gemm_simt<false, false, EPI_PARTIAL>(mat(dZ, C), X, C, K1, (int)n, splits_req, e, st)));
  if (defer) {
    *defer = PartialLayer{partial, splits, C, K1, (int)ldw, (long long)(dW - grads_base), (long long)(db - grads_base)};
    return RECNN_OK;
  }
  return launch_reduce_partials(partial, splits, C, K1, dW, ldw, db, st);
}

struct Ctx {
  const recnn_step_args* a;
  recnn_dims d;
  NetLayout la, lc;
  Workspace ws;
  const float *S, *S2, *ACT, *REW, *DONE;
  long long ldS, ldA;
  int lead;          // zero columns in front of every action row (= state_dim % 4)
  int64_t n;
  cudaStream_t st;
  Rng rng;
  bool train;
  float gate;
  AuxStreams* aux;       // non-null: chains V and P run on side streams
  bool v_prefetched, p_prefetched, p_deferred, v1_prefetched;
  bool value_opt_done[2];   // critic i was already stepped inside the value-gradient phase (fused with the split-K reduction)
};
// words of Workspace::tickets: 0..3 two-level reductions / optimizer step count, 6..7 error bits of the step
// (zeroed with the tickets at the head of every call that includes RECNN_PH_GATHER or RECNN_PH_VALUE_GRAD)
enum { kTicketDpMismatch = 6, kTicketOob = 7 };

// Critic hidden layers on (s, act):  h1 -> out1, h2 -> out2
static int critic_hidden(const Ctx& c, const float* params, const float* s, const float* act, bool train,
                         int mask_base, float* out1, float* out2, cudaStream_t st) {
  const int S = c.d.state_dim, A = c.d.action_dim, H = c.d.hidden;
  const uint8_t* m1 = (train && c.rng.masks) ? c.rng.masks[mask_base] : nullptr;
  const uint8_t* m2 = (train && c.rng.masks) ? c.rng.masks[mask_base + 1] : nullptr;
  const Seg xs = {s, S, c.ldS, 0}, xa = {act, A + c.lead, c.ldA, c.lead}, h1 = {out1, H, H, 0};
  RECNN_PROPAGATE(hidden_layer(xs, xa, params + c.lc.w1, c.lc.ld1, params + c.lc.b1, H, c.n, train, m1, c.rng,
                               mask_base, out1, st));
  return hidden_layer(h1, kNoSeg, params + c.lc.w2, c.lc.ld2, params + c.lc.b2, H, c.n, train, m2, c.rng,
                      mask_base + 1, out2, st);
}

static int actor_hidden(const Ctx& c, const float* params, const float* s, bool train, int mask_base,
                        float* out1, float* out2, cudaStream_t st) {
  const int S = c.d.state_dim, H = c.d.hidden;
  const uint8_t* m1 = (train && c.rng.masks) ? c.rng.masks[mask_base] : nullptr;
  const uint8_t* m2 = (train && c.rng.masks) ? c.rng.masks[mask_base + 1] : nullptr;
  const Seg xs = {s, S, c.ldS, 0}, h1 = {out1, H, H, 0};
  RECNN_PROPAGATE(hidden_layer(xs, kNoSeg, params + c.la.w1, c.la.ld1, params + c.la.b1, H, c.n, train, m1, c.rng,
                               mask_base, out1, st));
  return hidden_layer(h1, kNoSeg, params + c.la.w2, c.la.ld2, params + c.la.b2, H, c.n, train, m2, c.rng,
                      mask_base + 1, out2, st);
}

static HeadArgs head_args(const Ctx& c, const float* params, const float* h2, int mode) {
  HeadArgs h;
  h.h2 = h2; h.w3 = params + c.lc.w3; h.b3 = params + c.lc.b3;
  h.n_rows = c.n; h.n_rows_global = c.a->n_rows_global; h.hidden = c.d.hidden; h.mode = mode;
  h.reward = c.REW; h.done = c.DONE;
  h.gamma = c.a->gamma; h.min_value = c.a->min_value; h.max_value = c.a->max_value;
  h.y = c.ws.y; h.tmp = c.ws.qtmp; h.out = nullptr; h.dq = c.ws.dq; h.loss = nullptr;
  h.block_partials = c.ws.block_partials; h.ticket = c.ws.tickets;
  return h;
}

// ---------------------------------------------------------------- phases
static int policy_actor_forward(const Ctx& c, cudaStream_t st);
static int value_opt_one(Ctx& c, int i, const GradSource* src);

static int phase_value_grad(Ctx& c) {
  const recnn_step_args& a = *c.a;
  const int S = c.d.state_dim, A = c.d.action_dim, H = c.d.hidden;
  const bool td3 = a.algo == RECNN_ALGO_TD3;
  const int n_critics = td3 ? 2 : 1;
  float *X0 = c.ws.hb[0], *X1 = c.ws.hb[1], *c1 = c.ws.hb[2], *c2 = c.ws.hb[3], *dz2 = c.ws.hb[4],
        *dz1 = c.ws.hb[5];
  float* a2 = c.ws.ab[0];
  static const bool fuse_env = [] { const char* e = getenv("RECNN_B200_FUSE_HEAD"); return !(e && e[0] == '0'); }();
  const bool fuse_head = fuse_env && value_head_fusable(H);

  // target policy on next_state, eval mode (misc.py:28 / td3.py:73) (+ clipped noise, td3.py:74-78)
  if (a.next_action_in) {       // ... unless the caller ran its own (next_action_in: any policy class)
    RECNN_CHECK_CUDA(cudaMemcpy2DAsync(a2 + c.lead, c.ldA * 4, a.next_action_in, (size_t)A * 4, (size_t)A * 4, c.n,
                                       cudaMemcpyDeviceToDevice, c.st));
  } else {
  RECNN_PROPAGATE(actor_hidden(c, a.target_policy.params, c.S2, false, 0, X0, X1, c.st));
  if (c.aux && c.p_deferred) {
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[4], c.st));
    RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.aux->sp, c.aux->ev[4], 0));
    RECNN_PROPAGATE(policy_actor_forward(c, c.aux->sp));
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->p_done, c.aux->sp));
    c.p_prefetched = true;
  }
  NoiseSpec nz = {td3 ? 1 : 0, a.noise, a.noise_clip, a.noise_std, a.seed, (const long long*)a.rng_step, 15u};
  const Seg x1s = {X1, H, H, 0};
  RECNN_PROPAGATE(linear_out(x1s, a.target_policy.params + c.la.w3, c.la.ld3, a.target_policy.params + c.la.b3, A,
                             c.n, 0, &nz, a2 + c.lead, c.ldA, c.st));
  }
  if (a.next_action_out)
    RECNN_CHECK_CUDA(cudaMemcpy2DAsync(a.next_action_out, (size_t)A * 4, a2 + c.lead, c.ldA * 4, (size_t)A * 4, c.n,
                                       cudaMemcpyDeviceToDevice, c.st));

  // target critic(s) -> TD target y (misc.py:29-35 / td3.py:80-86).  TD3: the second target critic's hidden layers run
  // on a side stream into their own buffers, beside the first's; the two heads (min of the two Q's) follow in order.
  const bool tc1_side = td3 && c.aux != nullptr;
  float *T0 = c.ws.hb[8], *T1 = c.ws.hb[9];
  if (tc1_side) {
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[6], c.st));              // next_action is ready
    RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.aux->sw, c.aux->ev[6], 0));
    RECNN_PROPAGATE(critic_hidden(c, a.target_value[1].params, c.S2, a2, false, 0, T0, T1, c.aux->sw));
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[7], c.aux->sw));
  }
  for (int i = 0; i < n_critics; ++i) {
    AloneScope alone(c.aux != nullptr && !c.p_prefetched && !tc1_side);   // alone unless another chain runs alongside
    float* th2 = X1;
    if (i == 1 && tc1_side) {
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.st, c.aux->ev[7], 0));
      th2 = T1;
    } else {
      RECNN_PROPAGATE(critic_hidden(c, a.target_value[i].params, c.S2, a2, false, 0, X0, X1, c.st));
    }
    if (fuse_head && !td3) continue;       // DDPG: the TD target is formed inside the fused value-head kernel
    HeadArgs h = head_args(c, a.target_value[i].params, th2,
                           td3 ? (i == 0 ? HEAD_TARGET_TD3_A : HEAD_TARGET_TD3_B) : HEAD_TARGET_DDPG);
    RECNN_PROPAGATE(launch_critic_head(h, c.st));
  }

  // online critic(s): value, loss, backward (misc.py:37-43 / td3.py:88-101)
  for (int i = 0; i < n_critics; ++i) {
    const float* P = a.value[i].params;
    if (i == 1 && c.v1_prefetched) {        // the second critic's forward ran on its own stream into its own buffers
      c1 = c.ws.hb[10];
      c2 = c.ws.hb[11];
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.st, c.aux->ev[5], 0));
    } else if (i == 0 && c.v_prefetched) {
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.st, c.aux->v_done, 0));      // chain V ran on the side stream
    } else {
      RECNN_PROPAGATE(critic_hidden(c, P, c.S, c.ACT, c.train, 2 * i, c1, c2, c.st));
    }
    float* G = a.value[i].grads;
    RECNN_REQUIRE(!a.learn || G != nullptr, "value net needs a grad arena when learn=1");
    if (fuse_head) {
      // loss, dq, dz2 = (dq w3) * gate(h2), dW3 = dq^T h2, db3 = sum dq (and DDPG's TD target) in one launch
      ValueHeadArgs v;
      v.h2 = c2; v.w3 = P + c.lc.w3; v.b3 = P + c.lc.b3;
      v.th2 = td3 ? nullptr : X1;
      v.tw3 = a.target_value[0].params + c.lc.w3; v.tb3 = a.target_value[0].params + c.lc.b3;
      v.reward = c.REW; v.done = c.DONE;
      v.gamma = a.gamma; v.min_value = a.min_value; v.max_value = a.max_value;
      v.y = c.ws.y; v.n_rows = c.n; v.n_rows_global = a.n_rows_global; v.hidden = H;
      v.learn = a.learn ? 1 : 0; v.gate_scale = c.gate; v.dz2 = dz2;
      v.gw3 = a.learn ? G + c.lc.w3 : nullptr; v.gb3 = a.learn ? G + c.lc.b3 : nullptr;
      v.loss = a.losses + i;
      v.block_partials = c.ws.partial;       // free here: the weight-gradient GEMMs come later
      v.ticket = c.ws.tickets + 2;
      RECNN_PROPAGATE(launch_value_head_fused(v, c.st));
      if (!a.learn) continue;
    } else {
      HeadArgs h = head_args(c, P, c2, HEAD_VALUE);
      h.loss = a.losses + i;
      RECNN_PROPAGATE(launch_critic_head(h, c.st));
      if (!a.learn) continue;
      // layer 3: dW3 = dq^T h2, db3 = sum dq ; dz2 = (dq w3) * gate(h2)
      const int64_t rows_per = 256;
      const int splits = (int)ceil_div(c.n, rows_per);       // <= dw_splits(1, H, n, false): fits ws.partial
      RECNN_PROPAGATE(launch_head_grad_partials(c.ws.dq, c2, c.n, H, rows_per, splits, c.ws.partial, c.st));
      RECNN_PROPAGATE(launch_reduce_partials(c.ws.partial, splits, 1, H + 1, G + c.lc.w3, c.lc.ld3, G + c.lc.b3, c.st));
      RECNN_PROPAGATE(launch_critic_head_bwd(c.ws.dq, 0.f, P + c.lc.w3, c2, c.gate, dz2, c.n, H, c.st));
    }
    const Seg sc1 = {c1, H, H, 0}, ss = {c.S, S, c.ldS, 0}, sa = {c.ACT, A + c.lead, c.ldA, c.lead};
    // When this call also runs the built-in optimizer, the split-K partials of layers 1-2 are not reduced by
    // kernels of their own: the optimizer (or the data-parallel all-reduce) pass sums them (GradSource).
    // (r2i A/B against separate reduce kernels: 2708 vs 2711 steps/s -- kept for the three launches it saves)
    const bool fuse_opt = (a.phases & RECNN_PH_VALUE_OPT) && a.value_optim.kind != RECNN_OPT_EXTERNAL;
    GradSource gs;
    memset(&gs, 0, sizeof(gs));
    PartialLayer* d1 = fuse_opt ? &gs.l[0] : nullptr;
    PartialLayer* d2 = fuse_opt ? &gs.l[1] : nullptr;
    if (c.aux) {
      // dW2 (needs dz2, c1) on the side stream while the main stream back-propagates to dz1;
      // dW1's action segment on a third stream next to its state segment
      RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[0], c.st));
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.aux->sv, c.aux->ev[0], 0));
      RECNN_PROPAGATE(weight_grad(dz2, H, sc1, kNoSeg, c.n, G + c.lc.w2, c.lc.ld2, G + c.lc.b2, c.ws.partial2, c.aux->sv,
                                  nullptr, d2, G));
      RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[1], c.aux->sv));
      RECNN_PROPAGATE(backprop_hidden(dz2, H, P + c.lc.w2, c.lc.ld2, H, 0, H, c.n, c1, c.gate, dz1, c.st));
      const SideLaunch side = {c.aux->sw, c.aux->ev[2], c.aux->ev[3]};
      RECNN_PROPAGATE(weight_grad(dz1, H, ss, sa, c.n, G + c.lc.w1, c.lc.ld1, G + c.lc.b1, c.ws.partial, c.st, &side, d1, G));
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.st, c.aux->ev[1], 0));
    } else {
      RECNN_PROPAGATE(weight_grad(dz2, H, sc1, kNoSeg, c.n, G + c.lc.w2, c.lc.ld2, G + c.lc.b2, c.ws.partial2, c.st,
                                  nullptr, d2, G));
      RECNN_PROPAGATE(backprop_hidden(dz2, H, P + c.lc.w2, c.lc.ld2, H, 0, H, c.n, c1, c.gate, dz1, c.st));
      RECNN_PROPAGATE(weight_grad(dz1, H, ss, sa, c.n, G + c.lc.w1, c.lc.ld1, G + c.lc.b1, c.ws.partial, c.st, nullptr, d1, G));
    }
    if (fuse_opt) {
      gs.n_layers = 2;
      RECNN_PROPAGATE(value_opt_one(c, i, &gs));
      c.value_opt_done[i] = true;
    }
  }
  return RECNN_OK;
}

// the critic's optimizer step (data parallel: all-reduce + optimizer + value-loss sum in one kernel).  `src`: the
// gradient of layers 1-2 still sits in split-K partials, summed inside this pass instead of by reduce kernels.
static int value_opt_one(Ctx& c, int i, const GradSource* src) {
  const recnn_step_args& a = *c.a;
  if (a.comm) {
    // data parallel: every rank's shard gradient -> the global-batch gradient over NVLink, the optimizer update
    // of the reduced gradient and the sum of the ranks' value-loss partial sums, all in ONE kernel
    CommReduce r;
    r.aux_in = a.losses + i; r.aux_out = a.losses + i; r.n_aux = 1;
    r.check_val = (float)a.n_rows_global; r.err_flag = reinterpret_cast<int*>(c.ws.tickets + kTicketDpMismatch);
    r.optim = &a.value_optim; r.net = &a.value[i]; r.src = src;
    return launch_comm_allreduce(a.comm, a.value[i].grads, c.lc.count, r, c.st);
  }
  return launch_optimizer(a.value_optim, a.value[i], c.lc.count, nullptr, c.st, c.ws.tickets + 3, src);
}

static int phase_value_opt(Ctx& c) {
  const recnn_step_args& a = *c.a;
  if (!a.learn || a.value_optim.kind == RECNN_OPT_EXTERNAL) return RECNN_OK;
  const int n_critics = a.algo == RECNN_ALGO_TD3 ? 2 : 1;
  for (int i = 0; i < n_critics; ++i)
    if (!c.value_opt_done[i]) RECNN_PROPAGATE(value_opt_one(c, i, nullptr));
  return RECNN_OK;
}

// pi(s): hidden activations p1,p2 (kept for the actor backward) and gen_action
static int policy_actor_forward(const Ctx& c, cudaStream_t st) {
  const recnn_step_args& a = *c.a;
  const int H = c.d.hidden, A = c.d.action_dim;
  const int pm = a.algo == RECNN_ALGO_TD3 ? 4 : 2;
  float *p1 = c.ws.hb[6], *p2 = c.ws.hb[7];
  float* gen = c.ws.ab[1];
  RECNN_PROPAGATE(actor_hidden(c, a.policy.params, c.S, c.train, pm, p1, p2, st));
  const Seg sp2 = {p2, H, H, 0};
  return linear_out(sp2, a.policy.params + c.la.w3, c.la.ld3, a.policy.params + c.la.b3, A, c.n, 0, nullptr,
                    gen + c.lead, c.ldA, st);
}

static int phase_policy_loss(Ctx& c) {
  const recnn_step_args& a = *c.a;
  const int A = c.d.action_dim;
  const bool td3 = a.algo == RECNN_ALGO_TD3;
  const int vm = td3 ? 6 : 4;                       // mask slots (header: call order)
  float *v1 = c.ws.hb[0], *v2 = c.ws.hb[1];
  float* gen = c.ws.ab[1];
  // gen_action = policy_net(state); policy_loss = -value_net(state, gen_action)  (ddpg.py:78-79, td3.py:116-118)
  if (c.p_prefetched) RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.st, c.aux->p_done, 0));
  else RECNN_PROPAGATE(policy_actor_forward(c, c.st));
  if (a.gen_action_out)
    RECNN_CHECK_CUDA(cudaMemcpy2DAsync(a.gen_action_out, (size_t)A * 4, gen + c.lead, c.ldA * 4, (size_t)A * 4, c.n,
                                       cudaMemcpyDeviceToDevice, c.st));
  {
    AloneScope alone(true);
    RECNN_PROPAGATE(critic_hidden(c, a.value[0].params, c.S, gen, c.train, vm, v1, v2, c.st));
  }
  HeadArgs h = head_args(c, a.value[0].params, v2, HEAD_POLICY);
  h.loss = a.losses + 2;
  return launch_critic_head(h, c.st);
}

static int phase_policy_grad(Ctx& c) {
  const recnn_step_args& a = *c.a;
  if (!a.do_policy_step) return RECNN_OK;
  const int S = c.d.state_dim, A = c.d.action_dim, H = c.d.hidden;
  float *p1 = c.ws.hb[6], *p2 = c.ws.hb[7], *v1 = c.ws.hb[0], *v2 = c.ws.hb[1], *dv2 = c.ws.hb[4],
        *dv1 = c.ws.hb[5];
  float* dgen = c.ws.ab[2];
  const float* Pc = a.value[0].params;
  const float* Pa = a.policy.params;
  float* G = a.policy.grads;
  RECNN_REQUIRE(G != nullptr, "policy net needs a grad arena on a policy step");
  const float dq = -1.0f / (float)a.n_rows_global;            // d(-mean q)/dq
  // through the critic, input-gradient only, and only the action slice of layer 1
  RECNN_PROPAGATE(launch_critic_head_bwd(nullptr, dq, Pc + c.lc.w3, v2, c.gate, dv2, c.n, H, c.st));
  RECNN_PROPAGATE(backprop_hidden(dv2, H, Pc + c.lc.w2, c.lc.ld2, H, 0, H, c.n, v1, c.gate, dv1, c.st));
  RECNN_PROPAGATE(backprop_hidden(dv1, H, Pc + c.lc.w1, c.lc.ld1, S + A, S, A, c.n, nullptr, 1.f, dgen, c.st));
  // actor backward
  const Seg sp2 = {p2, H, H, 0}, sp1 = {p1, H, H, 0}, ss = {c.S, S, c.ldS, 0};
  RECNN_PROPAGATE(weight_grad(dgen, A, sp2, kNoSeg, c.n, G + c.la.w3, c.la.ld3, G + c.la.b3, c.ws.partial, c.st));
  float* dp2 = dv2;   // dv2/dv1 are dead once dgen exists
  float* dp1 = dv1;
  RECNN_PROPAGATE(backprop_hidden(dgen, A, Pa + c.la.w3, c.la.ld3, H, 0, H, c.n, p2, c.gate, dp2, c.st));
  RECNN_PROPAGATE(weight_grad(dp2, H, sp1, kNoSeg, c.n, G + c.la.w2, c.la.ld2, G + c.la.b2, c.ws.partial, c.st));
  RECNN_PROPAGATE(backprop_hidden(dp2, H, Pa + c.la.w2, c.la.ld2, H, 0, H, c.n, p1, c.gate, dp1, c.st));
  RECNN_PROPAGATE(weight_grad(dp1, H, ss, kNoSeg, c.n, G + c.la.w1, c.la.ld1, G + c.la.b1, c.ws.partial, c.st));
  return RECNN_OK;
}

static int phase_policy_opt(Ctx& c) {
  const recnn_step_args& a = *c.a;
  if (!a.do_policy_step) return RECNN_OK;
  float* coef = c.ws.scalars;
  // clip_grad_norm_(policy params, max_norm=-1, norm_type=1)   (ddpg.py:92, td3.py:133)
  if (a.comm) {
    // one kernel: all-reduce of the actor gradient, L1 norm of the SUMMED gradient -> clip coefficient, scaled
    // gradient written back, the built-in optimizer's update, and the sum of the ranks' policy-loss partial sums
    CommReduce r;
    r.max_norm = -1.0f; r.coef = coef; r.l1_out = a.losses + 3;
    r.aux_in = a.losses + 2; r.aux_out = a.losses + 2; r.n_aux = 1;
    r.check_val = (float)a.n_rows_global; r.err_flag = reinterpret_cast<int*>(c.ws.tickets + kTicketDpMismatch);
    r.optim = &a.policy_optim; r.net = &a.policy;
    return launch_comm_allreduce(a.comm, a.policy.grads, c.la.count, r, c.st);
  }
  RECNN_PROPAGATE(launch_l1_clip_coef(a.policy.grads, c.la.count, -1.0f, coef, a.losses + 3,
                                      c.ws.block_partials, c.ws.tickets + 1, c.st));
  if (a.policy_optim.kind == RECNN_OPT_EXTERNAL)
    return launch_scale_inplace(a.policy.grads, c.la.count, coef, c.st);
  return launch_optimizer(a.policy_optim, a.policy, c.la.count, coef, c.st, c.ws.tickets + 3);
}

static int phase_soft_update(Ctx& c) {
  const recnn_step_args& a = *c.a;
  if (!a.do_policy_step) return RECNN_OK;
  const int n_critics = a.algo == RECNN_ALGO_TD3 ? 2 : 1;
  for (int i = 0; i < n_critics; ++i)        // ddpg.py:95-97 / td3.py:136-141
    RECNN_PROPAGATE(launch_polyak(a.target_value[i].params, a.value[i].params, c.lc.count, a.soft_tau, c.st));
  if (a.algo == RECNN_ALGO_DDPG)              // ddpg.py:98-100; TD3 never updates its target policy
    RECNN_PROPAGATE(launch_polyak(a.target_policy.params, a.policy.params, c.la.count, a.soft_tau, c.st));
  return RECNN_OK;
}

static int run_step(const recnn_step_args* a, int algo, void* stream) {
  RECNN_REQUIRE(a != nullptr, "args");
  RECNN_REQUIRE(a->algo == algo, "args->algo does not match the entry point");
  RECNN_REQUIRE(a->n_rows > 0 && a->n_rows_global >= a->n_rows, "n_rows");
  RECNN_REQUIRE(a->dims.state_dim > 0 && a->dims.action_dim > 0 && a->dims.hidden > 0, "dims");
  RECNN_REQUIRE(a->n_rows < (1ll << 31) / (a->dims.state_dim + a->dims.action_dim + 1), "n_rows too large for int32 tile indexing");
  RECNN_REQUIRE(a->losses && a->workspace, "losses/workspace");
  const bool frames = a->table != nullptr;
  if (frames) {
    RECNN_REQUIRE(a->items && a->ratings && a->n_items > 0 && a->frame > 0 && a->emb_dim > 0, "frame-form batch");
    RECNN_REQUIRE(a->dims.state_dim == a->frame * a->emb_dim + a->frame && a->dims.action_dim == a->emb_dim,
                  "state_dim/action_dim do not match frame*dim+frame / dim");
  } else {
    RECNN_REQUIRE(a->state && a->next_state && a->action && a->reward, "dense batch needs state/next_state/action/reward");
  }
  RECNN_REQUIRE(a->done != nullptr, "done");
  const int n_critics = algo == RECNN_ALGO_TD3 ? 2 : 1;
  const int policy_phases = RECNN_PH_POLICY_LOSS | RECNN_PH_POLICY_GRAD | RECNN_PH_POLICY_OPT | RECNN_PH_SOFT_UPDATE;
  RECNN_REQUIRE((a->policy.params && a->target_policy.params) || (a->next_action_in && !(a->phases & policy_phases)),
                "policy nets (or next_action_in for a call made of the value phases only)");
  RECNN_REQUIRE(!a->next_action_in || algo == RECNN_ALGO_DDPG, "next_action_in is a DDPG-critic feature");
  for (int i = 0; i < n_critics; ++i)
    RECNN_REQUIRE(a->value[i].params && a->target_value[i].params, "value nets");
  if (a->dropout && !a->masks[0]) RECNN_REQUIRE(a->rng_step != nullptr, "perf-mode dropout needs rng_step");
  if (algo == RECNN_ALGO_TD3 && !a->noise) RECNN_REQUIRE(a->rng_step != nullptr, "perf-mode noise needs rng_step");

  Ctx c;
  c.a = a;
  c.d = a->dims;
  c.la = actor_layout(c.d);
  c.lc = critic_layout(c.d);
  c.n = a->n_rows;
  c.st = static_cast<cudaStream_t>(stream);
  c.ws = carve(c.d, c.n, a->workspace);
  if (c.ws.bytes > a->workspace_bytes) {
    set_error("workspace too small: need %lld bytes, got %lld", (long long)c.ws.bytes, (long long)a->workspace_bytes);
    return RECNN_E_WORKSPACE;
  }
  c.rng.masks = a->masks[0] ? a->masks : nullptr;
  c.rng.seed = a->seed;
  c.rng.step = (const long long*)a->rng_step;
  c.train = a->dropout != 0;
  c.gate = c.train ? 2.0f : 1.0f;
  c.DONE = a->done;
  c.ldS = pad4(c.d.state_dim);
  c.lead = c.d.state_dim % 4;
  c.ldA = pad4(c.d.action_dim + c.lead);
  const int S = c.d.state_dim, A = c.d.action_dim;
  // Head of a step: the tickets of the deterministic two-level reductions (self-resetting, but an aborted launch must
  // not poison the next step) and the step's error words start at zero.  Later calls of a split step keep them.
  if (a->phases & RECNN_PH_GATHER)
    RECNN_CHECK_CUDA(cudaMemsetAsync(c.ws.tickets, 0, 8 * sizeof(unsigned), c.st));
  // The step works on state / next_state images with a 16-byte-multiple row pitch (TMA); they are
  // materialised into the workspace once per step (RECNN_PH_GATHER) from the frames or the dense batch.
  c.S = c.ws.S;
  c.S2 = c.ws.S2;
  c.ACT = c.ws.ACT;
  if (a->phases & RECNN_PH_GATHER) {
    // action buffers carry `lead` zero columns (and pitch padding) that the kernels never write
    // (only the pad columns: one small kernel touching 1/30 of the bytes of three memsets)
    if (c.ldA != A)
      RECNN_PROPAGATE(launch_zero_pad_columns(c.ws.ACT, c.ws.ab[0], c.ws.ab[1], c.n, (int)c.ldA, c.lead, A, c.st));
  }
  if (frames) {
    if (a->phases & RECNN_PH_GATHER)
      RECNN_PROPAGATE(launch_frame_gather(a->table, a->n_items, a->emb_dim, a->items, a->ratings, c.n, a->frame,
                                          c.ldS, c.ldA, c.ws.S, c.ws.S2, c.ws.ACT + c.lead, c.ws.REW,
                                          reinterpret_cast<int*>(c.ws.tickets + kTicketOob), c.st));
    c.REW = a->reward ? a->reward : c.ws.REW;
  } else {
    if (a->phases & RECNN_PH_GATHER) {
      RECNN_CHECK_CUDA(cudaMemcpy2DAsync(c.ws.S, c.ldS * 4, a->state, (size_t)S * 4, (size_t)S * 4, c.n,
                                         cudaMemcpyDeviceToDevice, c.st));
      RECNN_CHECK_CUDA(cudaMemcpy2DAsync(c.ws.S2, c.ldS * 4, a->next_state, (size_t)S * 4, (size_t)S * 4, c.n,
                                         cudaMemcpyDeviceToDevice, c.st));
      RECNN_CHECK_CUDA(cudaMemcpy2DAsync(c.ws.ACT + c.lead, c.ldA * 4, a->action, (size_t)A * 4, (size_t)A * 4, c.n,
                                         cudaMemcpyDeviceToDevice, c.st));
    }
    c.REW = a->reward;
  }
  // fork: chain V (online critic forward) and chain P (online policy forward) on side streams
  c.aux = nullptr;
  c.v_prefetched = c.p_prefetched = c.p_deferred = c.v1_prefetched = false;
  c.value_opt_done[0] = c.value_opt_done[1] = false;
  if ((a->phases & RECNN_PH_VALUE_GRAD) && (c.aux = aux_streams()) != nullptr) {
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->fork, c.st));
    RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.aux->sv, c.aux->fork, 0));
    RECNN_PROPAGATE(critic_hidden(c, a->value[0].params, c.S, c.ACT, c.train, 0, c.ws.hb[2], c.ws.hb[3], c.aux->sv));
    RECNN_CHECK_CUDA(cudaEventRecord(c.aux->v_done, c.aux->sv));
    c.v_prefetched = true;
    if (a->algo == RECNN_ALGO_TD3) {
      // TD3's second online critic: forward on a third stream into its own buffers (td3.py:88-89 for value_net2)
      RECNN_CHECK_CUDA(cudaStreamWaitEvent(c.aux->sw, c.aux->fork, 0));
      RECNN_PROPAGATE(critic_hidden(c, a->value[1].params, c.S, c.ACT, c.train, 2, c.ws.hb[10], c.ws.hb[11], c.aux->sw));
      RECNN_CHECK_CUDA(cudaEventRecord(c.aux->ev[5], c.aux->sw));
      c.v1_prefetched = true;
    }
    // chain P is forked later (after the target policy's hidden layers, see phase_value_grad): three
    // concurrent layer-1 GEMMs are 192 CTAs = two waves on 148 SMs, two are one wave
    c.p_deferred = (a->phases & RECNN_PH_POLICY_LOSS) != 0;
  }
  if (a->phases & RECNN_PH_VALUE_GRAD) RECNN_PROPAGATE(phase_value_grad(c));
  if (a->phases & RECNN_PH_VALUE_OPT) RECNN_PROPAGATE(phase_value_opt(c));
  if (a->phases & RECNN_PH_POLICY_LOSS) RECNN_PROPAGATE(phase_policy_loss(c));
  if (a->phases & RECNN_PH_POLICY_GRAD) RECNN_PROPAGATE(phase_policy_grad(c));
  if (a->phases & RECNN_PH_POLICY_OPT) RECNN_PROPAGATE(phase_policy_opt(c));
  if (a->phases & RECNN_PH_SOFT_UPDATE) RECNN_PROPAGATE(phase_soft_update(c));
  if (a->phases & RECNN_PH_FINISH) {
    // losses are shard sums / n_rows_global: the sum over ranks is the global mean.  The value losses rode on the
    // critics' all-reduces and, on a policy step, the policy loss on the actor's; only a non-policy step needs this
    // scalar-only exchange (one CTA, one NVLink flag hop).
    if (a->comm && !(a->do_policy_step && (a->phases & RECNN_PH_POLICY_OPT))) {
      CommReduce r;
      r.aux_in = a->losses + 2; r.aux_out = a->losses + 2; r.n_aux = 1;
      r.check_val = (float)a->n_rows_global; r.err_flag = reinterpret_cast<int*>(c.ws.tickets + kTicketDpMismatch);
      RECNN_PROPAGATE(launch_comm_allreduce(a->comm, nullptr, 0, r, c.st));
    }
    // ++rng_step; losses[4] <- error bits of this step (1: item id out of range in the gather, 2: the ranks disagree
    // on n_rows_global)
    RECNN_PROPAGATE(launch_finish((long long*)a->rng_step, c.ws.tickets + kTicketOob, c.ws.tickets + kTicketDpMismatch,
                                  a->losses + 4, c.st));
    if (a->losses_host)
      RECNN_CHECK_CUDA(cudaMemcpyAsync(a->losses_host, a->losses, 8 * sizeof(float), cudaMemcpyDeviceToHost, c.st));
  }
  return RECNN_OK;
}

}  // namespace recnn

using namespace recnn;

extern "C" int64_t recnn_step_workspace_bytes(const recnn_dims* d, int64_t n_rows, int32_t algo) {
  (void)algo;
  if (!d || n_rows <= 0) return 0;
  return carve(*d, n_rows, nullptr).bytes;
}

extern "C" int recnn_ddpg_step(const recnn_step_args* args, void* stream) {
  return run_step(args, RECNN_ALGO_DDPG, stream);
}

extern "C" int recnn_td3_step(const recnn_step_args* args, void* stream) {
  return run_step(args, RECNN_ALGO_TD3, stream);
}

extern "C" int64_t recnn_actor_param_count(const recnn_dims* d) { return d ? actor_layout(*d).count : 0; }
extern "C" int64_t recnn_critic_param_count(const recnn_dims* d) { return d ? critic_layout(*d).count : 0; }

extern "C" int recnn_net_layout(const recnn_dims* d, int is_critic, int64_t* out) {
  RECNN_REQUIRE(d && out, "null pointer");
  const NetLayout l = is_critic ? critic_layout(*d) : actor_layout(*d);
  const int64_t v[10] = {l.w1, l.b1, l.w2, l.b2, l.w3, l.b3, l.ld1, l.ld2, l.ld3, l.count};
  for (int i = 0; i < 10; ++i) out[i] = v[i];
  return RECNN_OK;
}

// Inference entry points take densely packed inputs ([n, S] / [n, A]).  A row pitch that is not a 16-byte
// multiple (S = 1290) cannot be a TMA tensor, so the inputs are first re-pitched into scratch images (one 2-D
// device copy each, 21 MB at 4096 rows) and every layer runs on the tcgen05 path -- the CUDA-core kernel took
// 62 us per layer-1 launch at this shape, 30x a tensor-core launch.
extern "C" int64_t recnn_forward_scratch_floats(const recnn_dims* d, int64_t n_rows, int is_critic) {
  if (!d || n_rows <= 0) return 0;
  const int64_t ldS = pad4(d->state_dim), ldA = pad4(d->action_dim + d->state_dim % 4);
  return 2 * n_rows * d->hidden + n_rows * ldS + (is_critic ? n_rows * ldA : 0) + 64;
}

// state [n, S] (pitch S) -> a pitch-ldS image when needed; returns the Seg to read
static int repitch_state(const recnn_dims& d, const float* state, int64_t n, float* img, Seg* out, cudaStream_t st) {
  const int S = d.state_dim;
  if (S % 4 == 0 && aligned16(state)) {
    *out = Seg{state, S, S, 0};
    return RECNN_OK;
  }
  const int ldS = pad4(S);
  RECNN_CHECK_CUDA(cudaMemcpy2DAsync(img, (size_t)ldS * 4, state, (size_t)S * 4, (size_t)S * 4, n,
                                     cudaMemcpyDeviceToDevice, st));
  *out = Seg{img, S, ldS, 0};
  return RECNN_OK;
}

extern "C" int recnn_actor_forward(const recnn_dims* d, const float* params, const float* state, int64_t n_rows,
                                   const uint8_t* mask1, const uint8_t* mask2, int apply_tanh, float* action_out,
                                   float* scratch, void* stream) {
  RECNN_REQUIRE(d && params && state && action_out && scratch, "null pointer");
  RECNN_REQUIRE((mask1 == nullptr) == (mask2 == nullptr), "give both masks or neither");
  if (n_rows <= 0) return RECNN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const NetLayout l = actor_layout(*d);
  const int H = d->hidden;
  float* h1 = scratch;
  float* h2 = scratch + n_rows * H;
  float* img = reinterpret_cast<float*>(round_up(reinterpret_cast<int64_t>(h2 + n_rows * H), 16));
  Rng rng = {nullptr, 0, nullptr};
  const bool train = mask1 != nullptr;
  Seg xs;
  RECNN_PROPAGATE(repitch_state(*d, state, n_rows, img, &xs, st));
  const Seg s1 = {h1, H, H, 0}, s2 = {h2, H, H, 0};
  RECNN_PROPAGATE(hidden_layer(xs, kNoSeg, params + l.w1, l.ld1, params + l.b1, H, n_rows, train, mask1, rng, 0, h1, st));
  RECNN_PROPAGATE(hidden_layer(s1, kNoSeg, params + l.w2, l.ld2, params + l.b2, H, n_rows, train, mask2, rng, 1, h2, st));
  return linear_out(s2, params + l.w3, l.ld3, params + l.b3, d->action_dim, n_rows, apply_tanh, nullptr, action_out,
                    d->action_dim, st);
}

extern "C" int recnn_critic_forward(const recnn_dims* d, const float* params, const float* state,
                                    const float* action, int64_t n_rows, const uint8_t* mask1,
                                    const uint8_t* mask2, float* value_out, float* scratch, void* stream) {
  RECNN_REQUIRE(d && params && state && action && value_out && scratch, "null pointer");
  RECNN_REQUIRE((mask1 == nullptr) == (mask2 == nullptr), "give both masks or neither");
  if (n_rows <= 0) return RECNN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const NetLayout l = critic_layout(*d);
  const int H = d->hidden, S = d->state_dim, A = d->action_dim;
  float* h1 = scratch;
  float* h2 = scratch + n_rows * H;
  float* img = reinterpret_cast<float*>(round_up(reinterpret_cast<int64_t>(h2 + n_rows * H), 16));
  Rng rng = {nullptr, 0, nullptr};
  const bool train = mask1 != nullptr;
  Seg xs;
  RECNN_PROPAGATE(repitch_state(*d, state, n_rows, img, &xs, st));
  // the action block starts at weight column S: with S % 4 != 0 it needs `lead` zero columns in front (see Seg)
  const int lead = S % 4, ldA = pad4(A + lead);
  Seg xa = {action, A, A, 0};
  if (lead != 0 || A % 4 != 0 || !aligned16(action)) {
    float* aimg = img + n_rows * (int64_t)pad4(S);
    RECNN_CHECK_CUDA(cudaMemsetAsync(aimg, 0, sizeof(float) * n_rows * ldA, st));
    RECNN_CHECK_CUDA(cudaMemcpy2DAsync(aimg + lead, (size_t)ldA * 4, action, (size_t)A * 4, (size_t)A * 4, n_rows,
                                       cudaMemcpyDeviceToDevice, st));
    xa = Seg{aimg, A + lead, ldA, lead};
  }
  const Seg s1 = {h1, H, H, 0};
  RECNN_PROPAGATE(hidden_layer(xs, xa, params + l.w1, l.ld1, params + l.b1, H, n_rows, train, mask1, rng, 0, h1, st));
  RECNN_PROPAGATE(hidden_layer(s1, kNoSeg, params + l.w2, l.ld2, params + l.b2, H, n_rows, train, mask2, rng, 1, h2, st));
  HeadArgs h;
  h.h2 = h2; h.w3 = params + l.w3; h.b3 = params + l.b3; h.n_rows = n_rows; h.n_rows_global = n_rows;
  h.hidden = H; h.mode = HEAD_PLAIN; h.reward = nullptr; h.done = nullptr; h.gamma = 0; h.min_value = 0;
  h.max_value = 0; h.y = nullptr; h.tmp = nullptr; h.out = value_out; h.dq = nullptr; h.loss = nullptr;
  h.block_partials = nullptr; h.ticket = nullptr;
  return launch_critic_head(h, st);
}

extern "C" int recnn_linear_forward(const float* x, int64_t n_rows, int in_dim, const float* weight,
                                    const float* bias, int out_dim, int relu, float* out, void* stream) {
  RECNN_REQUIRE(x && weight && bias && out, "null pointer");
  RECNN_REQUIRE(in_dim > 0 && out_dim > 0 && n_rows >= 0, "sizes");
  if (n_rows == 0) return RECNN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Seg xs = {x, in_dim, in_dim, 0};
  if (relu) {
    Rng rng = {nullptr, 0, nullptr};
    return hidden_layer(xs, kNoSeg, weight, in_dim, bias, out_dim, n_rows, false, nullptr, rng, 0, out, st);
  }
  return linear_out(xs, weight, in_dim, bias, out_dim, n_rows, 0, nullptr, out, out_dim, st);
}

// ---------------------------------------------------------------- REINFORCE (policy side)
#include "reinforce.cuh"
