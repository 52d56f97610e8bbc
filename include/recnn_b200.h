/*
 * recnn_b200 -- C ABI of the B200-native RecNN DDPG/TD3 update hot path.
 *
 * The reference (awarebayes/RecNN) is pure Python on PyTorch and has NO FFI:
 * its seams for this path are Python call sites (SURVEY.md 8b).  Each entry
 * point below names the reference function (file:line under /root/reference)
 * whose work it replaces; the Python host layer in recnn_b200/ binds them with
 * ctypes and keeps the reference's own signatures on top (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless it says host;
 *   - every call takes the CUDA stream to launch on (cudaStream_t as void*);
 *     nothing synchronises, nothing allocates: scratch comes from the caller
 *     (recnn_step_workspace_bytes);
 *   - return 0 on success, a negative RECNN_E_* code otherwise;
 *     recnn_b200_last_error() returns a thread-local message;
 *   - all floating point data is fp32, item indices are int64 (as the
 *     reference's LongTensor), dropout masks are uint8 {0,1}.
 *   - a "net" is one 3-layer MLP stored as ONE flat fp32 arena in
 *     nn.Module.parameters() order: linear1.weight [H,in], linear1.bias [H],
 *     linear2.weight [H,H], linear2.bias [H], linear3.weight [out,H],
 *     linear3.bias [out]  (nn.Linear layout, y = x W^T + b;
 *     recnn/nn/models.py:41-57 Actor, :187-203 Critic).  Every matrix row and every
 *     segment is padded to a multiple of 4 floats (16 bytes, the TMA granule):
 *     recnn_net_layout() returns the offsets and row pitches; pad elements are 0.
 */
#ifndef RECNN_B200_H
#define RECNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RECNN_B200_ABI_VERSION 3

#if defined(__GNUC__)
#define RECNN_API __attribute__((visibility("default")))
#else
#define RECNN_API
#endif

enum {
  RECNN_OK = 0,
  RECNN_E_INVALID = -1,   /* bad argument (null pointer, non-positive size ...) */
  RECNN_E_CUDA = -2,      /* a CUDA runtime call / launch failed */
  RECNN_E_WORKSPACE = -3, /* workspace too small */
  RECNN_E_UNSUPPORTED = -4
};

RECNN_API int recnn_b200_abi_version(void);
RECNN_API const char* recnn_b200_last_error(void);
/* number of kernels this library has launched in this process (bench accounting) */
RECNN_API int64_t recnn_b200_launch_count(void);
/* struct-layout probes so a foreign binding can verify its mirror of recnn_step_args */
RECNN_API int64_t recnn_sizeof_step_args(void);
RECNN_API int64_t recnn_offsetof_step_args(int field);

/* ------------------------------------------------------------------ data path */

/* recnn/data/utils.py:51-68 batch_tensor_embeddings: gather table rows for the
 * F+1 items of every sample and assemble state / next_state / action / reward.
 *   table  fp32[n_items, dim] row-major      items   int64[n_rows, frame+1]
 *   ratings fp32[n_rows, frame+1]
 *   state, next_state fp32[n_rows, frame*dim+frame]; action fp32[n_rows, dim];
 *   reward fp32[n_rows].  Any output pointer may be NULL (skipped).
 * Bit-exact copy semantics.  Indices are checked on device; an out-of-range
 * index sets *oob_flag (device int32, may be NULL) and the row reads item 0. */
RECNN_API int recnn_frame_gather(const float* table, int64_t n_items, int dim,
                       const int64_t* items, const float* ratings,
                       int64_t n_rows, int frame,
                       float* state, float* next_state, float* action, float* reward,
                       int* oob_flag, void* stream);

/* recnn/data/utils.py:70-71: done = zeros(n_rows); done[cumsum(sizes-frame)-1] = 1.
 * sizes int64[n_users] (device). */
RECNN_API int recnn_done_from_sizes(const int64_t* sizes, int64_t n_users, int frame,
                          float* done, int64_t n_rows, void* stream);

/* Device-resident FrameEnv feed.  The reference builds every minibatch on the host, inside a
 * DataLoader worker: UserDataset.__getitem__ (recnn/data/env.py:47-64) hands out one user's
 * time-ordered items / ratings, and the collate function cuts ALL length-(frame+1) sliding
 * windows of every user of the batch and concatenates them (rolling_window, recnn/data/utils.py:7-10;
 * prepare_batch_static_size, :161-181; ratings cast with .float(), :178).  Here the histories stay in
 * HBM as a CSR over users
 *     hist_items int64[total]   hist_ratings fp32[total] (the .float() cast, done once)
 *     hist_offsets int64[n_users+1]
 * and the windows are cut on the device: the only per-minibatch input is the list of users.
 * Outputs are exactly what the collate hands to embed_batch: items int64[n_rows, frame+1],
 * ratings fp32[n_rows, frame+1] (feed them to recnn_frame_gather or to the frame form of
 * recnn_ddpg_step / recnn_td3_step), plus done fp32[n_rows] (recnn/data/utils.py:70-71:
 * 1 on the last window of every user) and sizes int64[n_batch] (history lengths, :171).
 * Any output pointer may be NULL.  Bit-exact (copies only).
 *   batch_users int64[n_batch]    positions of the minibatch's users in the CSR, in batch order
 *   row_offsets int64[n_batch+1]  exclusive prefix sum of (length - frame) over batch_users;
 *                                 n_rows == row_offsets[n_batch] (host-side plan: lengths are
 *                                 known to the caller, so no device->host sync is needed)
 * A user index out of range, or a plan that disagrees with the resident lengths, sets *err_flag
 * (device int32, may be NULL) and zero-fills the affected rows. */
RECNN_API int recnn_window_gather_users(const int64_t* hist_items, const float* hist_ratings,
                              const int64_t* hist_offsets, int64_t n_users,
                              const int64_t* batch_users, const int64_t* row_offsets, int64_t n_batch,
                              int frame, int64_t n_rows,
                              int64_t* items, float* ratings, float* done, int64_t* sizes,
                              int* err_flag, void* stream);

/* Fixed-size minibatch over the same CSR: row n is the window with GLOBAL id window_ids[n], windows
 * being numbered user by user in storage order (win_offsets int64[n_users+1] = exclusive prefix sum
 * of max(length - frame, 0)).  Equals rows window_ids of the reference collate over ALL users
 * (prepare_batch_static_size over the whole UserDataset, recnn/data/utils.py:161-181), so a
 * replay-style sampler can draw a constant number of rows per step (constant shapes keep the update
 * step one CUDA graph).  users_out int64[n_rows] (optional) = CSR position of each row's user;
 * done = 1 where the window is its user's last.  Out-of-range ids set *err_flag and zero-fill. */
RECNN_API int recnn_window_gather_ids(const int64_t* hist_items, const float* hist_ratings,
                            const int64_t* hist_offsets, const int64_t* win_offsets, int64_t n_users,
                            const int64_t* window_ids, int frame, int64_t n_rows,
                            int64_t* items, float* ratings, float* done, int64_t* users_out,
                            int* err_flag, void* stream);

/* ------------------------------------------------------------------ networks */

typedef struct recnn_dims {
  int32_t state_dim;   /* S = frame*dim + frame (1290) */
  int32_t action_dim;  /* A (128) */
  int32_t hidden;      /* H (256) */
  int32_t reserved;
} recnn_dims;

/* number of fp32 in an Actor / Critic arena for these dims (padding included) */
RECNN_API int64_t recnn_actor_param_count(const recnn_dims* d);
RECNN_API int64_t recnn_critic_param_count(const recnn_dims* d);

/* arena geometry: offsets (in floats) of w1,b1,w2,b2,w3,b3 then the row pitches of w1,w2,w3,
 * then the total count -> out[10].  is_critic selects in = S+A / out = 1. */
RECNN_API int recnn_net_layout(const recnn_dims* d, int is_critic, int64_t* out);

/* recnn/nn/models.py:59-73 Actor.forward.  masks: two uint8[n_rows,H] arrays
 * (train mode: h = relu(z) * mask * 2) or NULL,NULL for eval().  apply_tanh as
 * the reference's `tanh` argument.  scratch: fp32[recnn_forward_scratch_floats(d, n_rows, 0)]
 * (two hidden activations + a 16-byte-pitch image of `state` when its row pitch is not a 16-byte multiple,
 * so that every layer runs on the tensor cores). */
RECNN_API int64_t recnn_forward_scratch_floats(const recnn_dims* d, int64_t n_rows, int is_critic);
RECNN_API int recnn_actor_forward(const recnn_dims* d, const float* params, const float* state,
                        int64_t n_rows, const uint8_t* mask1, const uint8_t* mask2,
                        int apply_tanh, float* action_out, float* scratch, void* stream);

/* recnn/nn/models.py:205-213 Critic.forward (concat is virtual).  value_out fp32[n_rows];
 * scratch: fp32[recnn_forward_scratch_floats(d, n_rows, 1)]. */
RECNN_API int recnn_critic_forward(const recnn_dims* d, const float* params, const float* state,
                         const float* action, int64_t n_rows,
                         const uint8_t* mask1, const uint8_t* mask2,
                         float* value_out, float* scratch, void* stream);

/* One nn.Linear (+ optional ReLU) on its own: out[n_rows,out_dim] = act(x W^T + b)
 * (recnn/nn/models.py:52-54 layers; exposed so a single layer can be timed / reused). */
RECNN_API int recnn_linear_forward(const float* x, int64_t n_rows, int in_dim, const float* weight,
                         const float* bias, int out_dim, int relu, float* out, void* stream);

/* Generic contraction C[M,N] (pitch ldc) = A . B^T, the building block of every Linear
 * forward/backward in this path (torch addmm sites: recnn/nn/models.py:66-70, :207-212 and
 * their autograd backward).  a_mn=0: A is [M,K] row-major, a_mn=1: A is stored [K,M];
 * same for B with N.  recnn_gemm_tf32x3 runs on the tcgen05 tensor cores with
 * error-compensated 3xTF32 (fp32-grade accuracy; pitches and bases must be 16-byte
 * multiples; tile_n in {0 (auto), 64, 128}); recnn_gemm_fp32 is the exact-fp32
 * CUDA-core path for arbitrary shapes. */
RECNN_API int recnn_gemm_tf32x3(int M, int N, int K, const float* A, int64_t lda, int a_mn, const float* B,
                      int64_t ldb, int b_mn, float* C, int64_t ldc, int tile_n, void* stream);
RECNN_API int recnn_gemm_fp32(int M, int N, int K, const float* A, int64_t lda, int a_mn, const float* B,
                    int64_t ldb, int b_mn, float* C, int64_t ldc, void* stream);

/* recnn/utils/misc.py:1-5 soft_update over one flat arena:
 * target = target*(1-tau) + net*tau   (tau==1 is an exact copy, as in the reference) */
RECNN_API int recnn_polyak_update(float* target, const float* net, int64_t count, double tau, void* stream);

/* ------------------------------------------------------------------ update step */

typedef struct recnn_net {
  float* params;      /* arena */
  float* grads;       /* arena, same layout; NULL for target nets */
  float* opt_m;       /* Adam exp_avg / SGD momentum buffer (built-in optimizers), else NULL */
  float* opt_v;       /* Adam exp_avg_sq, else NULL */
  int32_t* opt_t;     /* device int32: number of optimizer steps taken so far */
  float* opt_slow;    /* Ranger: Lookahead slow weights (arena), else NULL */
} recnn_net;

/* RANGER = RAdam + Lookahead as in torch_optimizer.Ranger, the optimizer recnn.nn.DDPG/TD3 construct by default
 * (recnn/nn/algo.py:84-89, :139-147).  torch_optimizer is an un-vendored third-party dependency of the reference
 * (requirements.txt:7, unpinned) and absent from this environment: the restatement follows the published algorithm
 * (Liu et al. 2019 rectified Adam with the N_sma_threshhold switch; Zhang et al. 2019 Lookahead every k steps) and
 * its parity with the package is UNPINNED (DESIGN.md section 2). */
enum { RECNN_OPT_EXTERNAL = 0, RECNN_OPT_SGD = 1, RECNN_OPT_ADAM = 2, RECNN_OPT_RANGER = 3 };

typedef struct recnn_optim {   /* torch.optim.SGD / torch.optim.Adam / torch_optimizer.Ranger semantics */
  int32_t kind;
  int32_t k;          /* Ranger: Lookahead period (6) */
  /* doubles: torch keeps these as python floats and rounds to fp32 only where the
   * tensor op consumes them (e.g. step_size = lr / (1 - beta1**t) is formed in double) */
  double lr, beta1, beta2, eps, weight_decay, momentum;
  double alpha;            /* Ranger: Lookahead interpolation (0.5) */
  double n_sma_threshold;  /* Ranger: rectification switch (5) */
} recnn_optim;

/* what one call executes; OR them.  A drop-in single-GPU step passes RECNN_PH_ALL.
 * Multi-GPU data parallel and external torch optimizers split the step at the
 * two points where gradients are complete. */
enum {
  RECNN_PH_VALUE_GRAD = 1,   /* targets, TD target, value loss, critic backward        */
  RECNN_PH_VALUE_OPT = 2,    /* built-in critic optimizer step(s)                      */
  RECNN_PH_POLICY_LOSS = 4,  /* pi(s), Q(s,pi(s)) with the *updated* critic, loss      */
  RECNN_PH_POLICY_GRAD = 8,  /* actor backward through the critic (policy steps only)  */
  RECNN_PH_POLICY_OPT = 16,  /* L1 "clip" quirk (+ built-in actor optimizer step)      */
  RECNN_PH_SOFT_UPDATE = 32, /* Polyak target updates (policy steps only)              */
  RECNN_PH_GATHER = 64,      /* frame form: materialise state/next_state/action into the
                              * workspace (split-phase callers pass it once per step)  */
  RECNN_PH_FINISH = 128,     /* end of step: error bits -> losses[4], copy losses to losses_host (if set), ++*rng_step */
  RECNN_PH_ALL = 255
};

enum { RECNN_ALGO_DDPG = 0, RECNN_ALGO_TD3 = 1 };

/* Peer-memory communicator of the data-parallel step (see "data parallel" below); opaque. */
typedef struct recnn_comm recnn_comm;

typedef struct recnn_step_args {
  int32_t algo;            /* RECNN_ALGO_* */
  int32_t phases;          /* RECNN_PH_* mask */
  int32_t learn;           /* reference `learn` flag */
  int32_t do_policy_step;  /* learn && step % policy_step == 0 (ddpg.py:89 / td3.py:130) */
  recnn_dims dims;

  /* batch: EITHER dense (state,next_state,action) OR frames (table,items,ratings).
   * reward/done fp32[n_rows] may be NULL in frame form for reward (= ratings[:,F]). */
  int64_t n_rows;          /* rows in this call (this rank's shard)          */
  int64_t n_rows_global;   /* denominator of the batch means (all ranks)     */
  const float* state;
  const float* next_state;
  const float* action;
  const float* table;
  int64_t n_items;
  int32_t frame;
  int32_t emb_dim;
  const int64_t* items;
  const float* ratings;
  const float* reward;
  const float* done;

  /* nets.  DDPG: value[0], target_value[0].  TD3: [0] and [1]. */
  recnn_net policy, target_policy;
  recnn_net value[2], target_value[2];
  recnn_optim policy_optim, value_optim;

  /* hyper-parameters (recnn/nn/algo.py:103-109, :164-174) */
  float gamma, min_value, max_value, noise_std, noise_clip;
  int32_t dropout;         /* 1: online nets are in train() mode (Dropout p=.5 active) */
  double soft_tau;

  /* randomness.  Parity mode: explicit masks (uint8[n_rows,H]) in the reference's
   * drop_layer call order -- DDPG: value(2) policy(2) value(2); TD3: value1(2)
   * value2(2) policy(2) value1(2) -- and the raw N(0,noise_std) draw fp32[n_rows,A].
   * Perf mode: all NULL; Philox4x32-10 keyed by (seed, *rng_step) on device. */
  const uint8_t* masks[8];
  const float* noise;
  uint64_t seed;
  int64_t* rng_step;         /* device int64 counter; read by every phase, incremented by RECNN_PH_FINISH */

  /* outputs */
  float* losses;           /* device, 8 words: fp32 value(1), value2, policy, ||actor grad||_1; then one int32 of
                            * error bits written by RECNN_PH_FINISH (1: an item id of the frame-form batch was outside
                            * [0, n_items) -- such rows read table row 0; 2: the ranks of a data-parallel step
                            * disagree on n_rows_global); 3 spare words */
  float* losses_host;      /* optional PINNED host buffer of 8 words: RECNN_PH_FINISH copies `losses` here (async) */
  float* next_action_out;  /* optional fp32[n_rows,A] (debug["next_action"]) */
  float* gen_action_out;   /* optional fp32[n_rows,A] (debug["gen_action"])  */
  /* optional fp32[n_rows,A]: the target policy's action on next_state, computed by the caller.  When given the
   * step does not run a target policy of its own (policy / target_policy may then be all-NULL for a call made only of
   * the VALUE phases): this is how misc.py:28 is served when the policy is not an Actor -- the REINFORCE critic is
   * updated against DiscreteActor probabilities (recnn/nn/update/reinforce.py:92-102). */
  const float* next_action_in;

  void* workspace;
  int64_t workspace_bytes;

  /* data parallel (optional, NULL on one GPU): when set, the step all-reduces (sums) the gradient
   * arenas over the communicator's ranks before each optimizer update, and the three loss scalars
   * before RECNN_PH_FINISH, with kernels on `stream` -- no host-side collective between phases.
   * Each rank passes its shard (n_rows local, n_rows_global = total). */
  const recnn_comm* comm;
} recnn_step_args;

/* bytes of scratch a step with these shapes needs (frame form included). */
RECNN_API int64_t recnn_step_workspace_bytes(const recnn_dims* d, int64_t n_rows, int32_t algo);

/* recnn/nn/update/ddpg.py:8-104 (with misc.py:10-55 value_update inlined). */
RECNN_API int recnn_ddpg_step(const recnn_step_args* args, void* stream);
/* recnn/nn/update/td3.py:8-150. */
RECNN_API int recnn_td3_step(const recnn_step_args* args, void* stream);

/* built-in optimizer step on one arena, exposed for recnn_b200.optim
 * (torch.optim.Adam/SGD semantics; increments *net->opt_t).
 * grad_scale: optional device scalar the gradient is multiplied by first. */
RECNN_API int recnn_optimizer_step(const recnn_optim* o, const recnn_net* net, int64_t count,
                         const float* grad_scale, void* stream);

/* ---- serving: nearest-item retrieval over the embedding table ----------------------------------
 * The step after Actor.forward in the reference's serving examples: the generated action (a 128-d
 * embedding) is matched against the item matrix -- examples/streamlit_demo.py:189-203 (faiss
 * IndexFlatL2 / IndexFlatIP / IndexFlatIP over L2-normalised rows), recnn/data/db_con.py:45-56
 * (MilvusConnection.search(search_vecs, topk) -> ids, distances).  Exact search: one
 * [n_queries, dim] x [dim, n_items] contraction on the tensor cores (3xTF32) + an exact top-k.
 * Ordering: best first; L2 reports the squared distance (as faiss / Milvus do), IP the inner product,
 * COS the cosine similarity; ties go to the smaller item id.  k <= 64. */
enum { RECNN_METRIC_L2 = 0, RECNN_METRIC_IP = 1, RECNN_METRIC_COS = 2 };
/* out[n_items]: |item|^2 (L2) or 1/|item| (COS); computed once per table ("index build") */
RECNN_API int recnn_item_norms(const float* table, int64_t n_items, int32_t dim, int32_t metric, float* out,
                               void* stream);
RECNN_API int64_t recnn_retrieve_workspace_bytes(int64_t n_queries, int64_t n_items, int32_t k);
/* ids_out int64[n_queries, k], dist_out fp32[n_queries, k]; norms from recnn_item_norms (NULL for IP) */
RECNN_API int recnn_retrieve_topk(const float* queries, int64_t n_queries, int32_t dim, const float* table,
                                  int64_t n_items, const float* norms, int32_t metric, int32_t k,
                                  int64_t* ids_out, float* dist_out, void* workspace, int64_t workspace_bytes,
                                  void* stream);

/* ---- REINFORCE with (Top-K) off-policy correction: the policy side (SURVEY 8f-2) ------------------
 * DiscreteActor (recnn/nn/models.py:76-99): probs = softmax(W2 relu(W1 s + b1) + b2), one output per item.
 * Parameter arena in nn.Module.parameters() order -- linear1.weight [H, S], linear1.bias, linear2.weight
 * [num_items, H], linear2.bias -- matrix rows padded to 16-byte multiples (recnn_discrete_layout). */
typedef struct recnn_discrete_dims {
  int32_t state_dim, hidden, num_items, reserved;
} recnn_discrete_dims;
/* out[7]: offsets of w1, b1, w2, b2; row pitches of w1, w2; total float count */
RECNN_API int recnn_discrete_layout(const recnn_discrete_dims* d, int64_t* out);
/* floats of scratch for n_rows rows: forward only (backward = 0) or recnn_reinforce_policy_grad (backward = 1) */
RECNN_API int64_t recnn_discrete_scratch_floats(const recnn_discrete_dims* d, int64_t n_rows, int32_t backward);
/* DiscreteActor.forward (models.py:95-99): probs_out fp32 [n_rows, num_items] dense */
RECNN_API int recnn_discrete_forward(const recnn_discrete_dims* d, const float* params, const float* state,
                                     int64_t n_rows, float* probs_out, float* scratch, void* stream);
/* Categorical(probs).sample() + .log_prob(sample) (models.py:107-110, 121-143): inverse CDF on `uniforms`
 * [n_rows] in [0,1) when given (replayable), else on Philox(seed, draw, row).  probs fp32 [n_rows, ld >= num_items];
 * rows are normalised by their sum and clamped to [eps, 1-eps] before the log, as torch does. */
RECNN_API int recnn_categorical_sample(const float* probs, int64_t n_rows, int32_t num_items, int64_t ld,
                                       const float* uniforms, uint64_t seed, int64_t draw, int64_t* action_out,
                                       float* log_prob_out, void* stream);
/* Categorical(probs).log_prob(action) for given actions; *oob_flag (may be NULL) is set when an id is out of range */
RECNN_API int recnn_categorical_log_prob(const float* probs, int64_t n_rows, int32_t num_items, int64_t ld,
                                         const int64_t* action, float* log_prob_out, int32_t* oob_flag, void* stream);
/* ChooseREINFORCE (recnn/nn/update/reinforce.py:10-65): the three policy losses */
enum { RECNN_REINFORCE_BASIC = 0, RECNN_REINFORCE_CORRECTED = 1, RECNN_REINFORCE_TOPK = 2 };
/* Policy loss and its gradient over the n_rows rows saved since the last policy update (the reference's
 * saved_log_probs / correction / lambda_k lists, concatenated): state [n_rows, state_dim], action int64 [n_rows]
 * (the sampled item), beta_log_prob [n_rows] (NULL for BASIC), returns [n_rows] (the normalised discounted return of
 * the env step the row was saved at, reinforce.py:44-52).  Recomputes the forward, writes the gradient of every
 * parameter into `grads` (arena geometry; overwritten, i.e. zero_grad + backward), out[0] = loss (fp32),
 * out[1] = int32 flag: an action id was outside [0, num_items) (that row contributed nothing). */
RECNN_API int recnn_reinforce_policy_grad(const recnn_discrete_dims* d, const float* params, float* grads,
                                          const float* state, const int64_t* action, const float* beta_log_prob,
                                          const float* returns, int64_t n_rows, int32_t method, int32_t top_k,
                                          float* out, float* scratch, void* stream);
/* Item-streamed form of recnn_reinforce_policy_grad for vocabularies whose [n_rows, num_items] logits do not fit in
 * memory (reinforce.py:10-65 with models.py:95-99 over a million items): the same arguments and outputs, plus
 * item_chunk >= 1.  The logits are computed item_chunk items at a time (the last chunk may be narrower) twice -- once
 * for each row's softmax statistics and the log-prob of its action, once more for d loss / d logits, consumed chunk by
 * chunk by the weight and hidden-layer gradients -- so the scratch holds one [n_rows, item_chunk] chunk instead of all
 * logits.  Deterministic for a given item_chunk; about 4/3 the logit FLOPs of the materialised entry. */
RECNN_API int64_t recnn_reinforce_streamed_scratch_floats(const recnn_discrete_dims* d, int64_t n_rows,
                                                          int32_t item_chunk);
RECNN_API int recnn_reinforce_policy_grad_streamed(const recnn_discrete_dims* d, const float* params, float* grads,
                                                   const float* state, const int64_t* action,
                                                   const float* beta_log_prob, const float* returns, int64_t n_rows,
                                                   int32_t method, int32_t top_k, int32_t item_chunk, float* out,
                                                   float* scratch, void* stream);

/* ---- data parallel: all-reduce over NVLink peer memory ------------------------------------------
 * BASELINE north_star: "partition the embedding gather + update across the 8 GPUs of one box with
 * an allreduce of the Actor/Critic gradients over NVLink".  The reference itself is single-process
 * (recnn/nn/update/ddpg.py:82-100 is where the gradients are complete and consumed), so these entry
 * points have no reference counterpart; they are what a torch.distributed launcher binds:
 *   every rank:  recnn_comm_create -> recnn_comm_local_handle -> (all-gather the handles with any
 *   host transport) -> recnn_comm_connect -> put the communicator in recnn_step_args.comm.
 * One process per GPU, at most 8 ranks on one node; the staging buffers are cudaMalloc memory shared
 * with cudaIpc and read by the peers' kernels directly (no NCCL call on the step's path). */
RECNN_API int recnn_comm_create(int32_t rank, int32_t world, int64_t capacity_floats, recnn_comm** out);
RECNN_API int32_t recnn_comm_handle_bytes(void);
RECNN_API int recnn_comm_local_handle(const recnn_comm* comm, void* out_handle);
/* all_handles: `world` handles of recnn_comm_handle_bytes() each, in rank order */
RECNN_API int recnn_comm_connect(recnn_comm* comm, const void* all_handles);
/* buf[i] <- sum over ranks of buf[i], in place, identical bits on every rank (n <= capacity_floats);
 * every rank must issue the same sequence of collectives on ONE stream. */
RECNN_API int recnn_comm_allreduce(const recnn_comm* comm, float* buf, int64_t n, void* stream);
RECNN_API int recnn_comm_destroy(recnn_comm* comm);

#ifdef __cplusplus
}
#endif
#endif /* RECNN_B200_H */
