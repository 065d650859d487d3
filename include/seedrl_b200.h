/* seedrl_b200.h -- C-ABI of libseedrl_b200.so: the B200 (sm_100a) hot path of a
 * SEED-RL V-trace learner.  Plain C, no torch / C++ types in any signature.
 *
 * Conventions (all entry points):
 *   - return 0 on success, non-zero error code otherwise; the message is
 *     available from seedrl_last_error() (thread-local).
 *   - every device pointer is caller-owned (torch or cudaMalloc), never freed
 *     or retained beyond the call unless a handle documents it.
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued, not synced.
 *   - tensors are dense, row-major, fp32 unless stated; time-major [T, B, ...]
 *     exactly like the reference's learner (agents/vtrace/learner.py:418-432).
 *   - there is NO CPU fallback anywhere behind this ABI.
 *
 * Each entry point cites the reference interface it replaces
 * (paths relative to google-research/seed_rl).
 */
#ifndef SEEDRL_B200_H_
#define SEEDRL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEEDRL_OK 0
#define SEEDRL_ERR_INVALID_ARGUMENT 3   /* tensorflow.error.Code values, so the  */
#define SEEDRL_ERR_OUT_OF_RANGE 11      /* RPC layer can forward them unchanged  */
#define SEEDRL_ERR_INTERNAL 13          /* (grpc/service.proto:51-56)            */
#define SEEDRL_ERR_CANCELLED 1
#define SEEDRL_ERR_UNAVAILABLE 14

typedef void* seedrl_stream_t;

const char* seedrl_last_error(void);
int seedrl_abi_version(void);
/* Number of kernels launched by this library since load (bench.py's
 * `gpu_launches` evidence). */
uint64_t seedrl_kernel_launch_count(void);

/* ------------------------------------------------------------------------
 * (a1) V-trace targets.   Replaces common/vtrace.py:34-148
 * `from_importance_weights`.  Inputs [T, B] (B may be a flattened B*C for the
 * "extra trailing dims" case, vtrace.py:49-51), bootstrap [B].  A NaN clip
 * threshold means `None` (no clipping, vtrace.py:111-114,138-142).
 * Outputs vs, pg_advantages [T, B].
 */
int seedrl_vtrace_from_importance_weights(
    int T, int B,
    const float* target_action_log_probs, const float* behaviour_action_log_probs,
    const float* discounts, const float* rewards, const float* values,
    const float* bootstrap_value,
    float clip_rho_threshold, float clip_pg_rho_threshold, float lambda_,
    float* vs, float* pg_advantages, seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a3) Categorical distribution.  Replaces
 * common/parametric_distribution.py:66-74,83-97 (tfd.Categorical log_prob /
 * entropy) and the sampling of dmlab/networks.py:121-122.
 * logits [N, A]; actions int64 [N] (tf.int64, dmlab/networks.py:121).
 */
int seedrl_categorical_log_prob(int N, int A, const float* logits,
                                const int64_t* actions, float* log_prob,
                                seedrl_stream_t stream);
int seedrl_categorical_entropy(int N, int A, const float* logits, float* entropy,
                               seedrl_stream_t stream);
/* Gumbel-max sample: action = argmax_k(logits[k] + g[k]).  If gumbel_noise is
 * non-NULL ([N, A] fp32) it is used as g (bit-exact, test mode); otherwise g is
 * drawn in-kernel from Philox4x32-10 keyed by (seed, offset). */
int seedrl_categorical_sample(int N, int A, const float* logits,
                              const float* gumbel_noise, uint64_t seed,
                              uint64_t offset, int64_t* actions,
                              seedrl_stream_t stream);
/* Same draw, with the Philox offset read from and then incremented in device memory (*counter_dev):
 * capturable in a CUDA graph (central inference replays one graph per batch). */
int seedrl_categorical_sample_counter(int N, int A, const float* logits, const float* gumbel_noise,
                                      uint64_t seed, uint64_t* counter_dev, int64_t* actions,
                                      seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a2) Fused V-trace loss: the part of agents/vtrace/learner.py:82-157
 * `compute_loss` after the network unroll, PLUS its analytic gradient
 * (what tape.gradient, learner.py:264, produces for the network outputs).
 */
typedef struct seedrl_loss_config {
  float discounting;        /* FLAGS.discounting  learner.py:59  */
  float lambda_;            /* FLAGS.lambda_      learner.py:60  */
  float baseline_cost;      /* learner.py:57 */
  float kl_cost;            /* learner.py:58 */
  float max_abs_reward;     /* learner.py:61; 0 disables clipping */
  float clip_rho_threshold;     /* compute_loss uses the default 1.0; NaN = None */
  float clip_pg_rho_threshold;  /* compute_loss uses the default 1.0; NaN = None */
  float target_entropy;     /* learner.py:52; used iff has_target_entropy */
  int32_t has_target_entropy;
  float entropy_cost_adjustment_speed; /* `mul`, learner.py:54,226 */
} seedrl_loss_config;

/* Indices into loss_terms[SEEDRL_LOSS_TERMS] (device, fp32), in the order the
 * reference logs them (learner.py:138-157). */
enum {
  SEEDRL_LT_TOTAL = 0, SEEDRL_LT_POLICY = 1, SEEDRL_LT_V = 2, SEEDRL_LT_ENTROPY = 3,
  SEEDRL_LT_KL = 4, SEEDRL_LT_ENTROPY_ADJ = 5, SEEDRL_LT_V_MEAN = 6,
  SEEDRL_LT_V_L2_ERROR = 7, SEEDRL_LT_MEAN_ENTROPY = 8, SEEDRL_LT_ENTROPY_COST = 9,
  SEEDRL_LT_MEAN_KL = 10, SEEDRL_LT_MAX_ACTION_ABS = 11,
  SEEDRL_LOSS_TERMS = 16
};

/* T1 = unroll_length + 1 rows, as in compute_loss.
 *   learner_logits [T1,B,A], learner_baseline [T1,B]   (network outputs)
 *   behaviour_logits [T1,B,A], actions int64 [T1,B]     (agent_outputs)
 *   rewards [T1,B], done uint8 [T1,B]                    (env_outputs)
 *   entropy_cost_param: device scalar; entropy_cost = exp(mul * param)
 *                       (learner.py:225-234)
 * Outputs: loss_terms[16]; dlogits [T1,B,A] and dbaseline [T1,B] = d total_loss
 * / d learner outputs (row T1-1 is zero: the bootstrap only enters through
 * stop_gradient'ed V-trace outputs); d_entropy_cost_param (device scalar);
 * optional vs / pg_advantages [T1-1,B] (may be NULL).
 * `scratch` must hold seedrl_vtrace_loss_scratch_bytes(T1,B,A) bytes and be
 * ZERO-INITIALISED ONCE by the caller; every launch leaves it zeroed again
 * (self-resetting completion ticket), so it can be reused without a memset. */
size_t seedrl_vtrace_loss_scratch_bytes(int T1, int B, int A);
int seedrl_vtrace_loss_fwd_bwd(
    int T1, int B, int A,
    const float* learner_logits, const float* learner_baseline,
    const float* behaviour_logits, const int64_t* actions,
    const float* rewards, const uint8_t* done,
    const seedrl_loss_config* cfg, const float* entropy_cost_param,
    float* loss_terms, float* dlogits, float* dbaseline,
    float* d_entropy_cost_param, float* vs_out, float* pg_advantages_out,
    void* scratch, seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a4) Optimizer apply.  Replaces optimizer.apply_gradients
 * (agents/vtrace/learner.py:272-273) with tf.keras Adam semantics
 * (dmlab/vtrace_main.py:46-51): ONE launch over the flat parameter arena.
 *   lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the caller's host code from
 *   `iterations`; here: m=b1 m+(1-b1) g; v=b2 v+(1-b2) g^2;
 *   p -= lr_t * m/(sqrt(v)+eps).   g is pre-multiplied by grad_scale (1 for the
 *   reference's cross-replica SUM, 1/N for a mean).
 * clamp_index >= 0 clamps that one element to [clamp_lo, clamp_hi] after the
 * update (the entropy_cost_param constraint, learner.py:229-231). */
int seedrl_adam_apply(size_t n, float* params, const float* grads, float* m,
                      float* v, float lr_t, float beta1, float beta2, float eps,
                      float grad_scale, int64_t clamp_index, float clamp_lo,
                      float clamp_hi, seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a5) Policy network.  Replaces dmlab/networks.py:63-171 `ImpalaDeep`
 * (__call__/_unroll/_torso/_head, _Stack) and common/utils.py:714-732
 * batch_apply; SEEDRL_NET_SHALLOW is the IMPALA-paper shallow net (not in the
 * reference, SURVEY 0).  Parameters live in ONE flat fp32 arena in
 * tf.Module.trainable_variables order with Keras layouts (conv HWIO, dense
 * [in,out], LSTM [in,4H] gates i,f,c,o) followed by the scalar
 * entropy_cost_param; seedrl_net_param_* describe it.
 */
enum { SEEDRL_NET_DEEP = 0, SEEDRL_NET_SHALLOW = 1 };

typedef struct seedrl_net_config {
  int32_t net;            /* SEEDRL_NET_* */
  int32_t num_actions;    /* A */
  int32_t obs_h, obs_w, obs_c;   /* uint8 NHWC observation */
} seedrl_net_config;

typedef struct seedrl_net seedrl_net;   /* opaque: layer table + offsets only */

int seedrl_net_create(const seedrl_net_config* cfg, seedrl_net** out);
void seedrl_net_destroy(seedrl_net* net);
int seedrl_net_num_param_tensors(const seedrl_net* net);       /* 39 for deep */
size_t seedrl_net_num_params(const seedrl_net* net);          /* excl. entropy param */
/* Length (floats) of the flat arena: every tensor start is aligned to 64 floats,
 * the last slot is the scalar entropy_cost_param (param index == num tensors). */
size_t seedrl_net_arena_floats(const seedrl_net* net);
/* Contraction path of every 3x3 convolution (forward, data and weight gradient) and of the
 * Dense / LSTM-projection / head GEMMs:
 * 0 = fp32 SIMT (bit-reproducible fp32 reference path), 1 = tcgen05 tensor cores, bf16
 * operands with fp32 accumulation, 2 = tcgen05 with bf16x3 split operands (hi*hi + lo*hi +
 * hi*lo: fp32-faithful to ~2^-16 relative), 3 = the same bf16x3 arithmetic with the 16/32-channel
 * activations and gradients kept in HBM as bf16 hi/lo channel-group planes (the UMMA operand
 * format): TMA-fed, warp-specialised conv kernels (csrc/conv_planes.cu; deep net only). */
int seedrl_net_set_conv_mode(seedrl_net* net, int mode);
/* LSTM recurrence: 2 (default) = one persistent kernel for all T steps each way with CTA = (batch
 * tile, 16 hidden units) and one barrier counter per batch tile (csrc/lstm_tiled.cu); 0 = a GEMM + a
 * pointwise kernel per time step (the reference the tiled kernels are tested against).  1 (an earlier
 * persistent form, since removed) is rejected with SEEDRL_ERR_INVALID_ARGUMENT. */
int seedrl_net_set_lstm_mode(seedrl_net* net, int mode);
/* name is written into buf (NUL-terminated); shape into dims[0..3], rank returned. */
int seedrl_net_param_info(const seedrl_net* net, int index, char* name_buf,
                          size_t name_buf_len, int64_t* dims, size_t* offset);
/* Bytes of activation workspace for an unroll of T1 x B frames kept for backward. */
size_t seedrl_net_workspace_bytes(const seedrl_net* net, int T1, int B);

/* Forward unroll (is_training=True, unroll=True): inputs time-major,
 *   prev_actions int64 [T1,B], reward [T1,B], done uint8 [T1,B],
 *   observation uint8 [T1,B,H,W,C], h0/c0 [B,256].
 * outputs policy_logits [T1,B,A], baseline [T1,B], h_out/c_out [B,256]. */
int seedrl_net_forward(const seedrl_net* net, const float* params, int T1, int B,
                       const int64_t* prev_actions, const float* reward,
                       const uint8_t* done, const uint8_t* observation,
                       const float* h0, const float* c0,
                       float* policy_logits, float* baseline,
                       float* h_out, float* c_out,
                       void* workspace, size_t workspace_bytes,
                       seedrl_stream_t stream);
/* Backward of the same unroll (must follow seedrl_net_forward on the same
 * workspace).  grads (flat arena layout, same offsets as params) is OVERWRITTEN
 * with d loss / d params. */
int seedrl_net_backward(const seedrl_net* net, const float* params, int T1, int B,
                        const int64_t* prev_actions, const float* reward,
                        const uint8_t* done, const uint8_t* observation,
                        const float* dlogits, const float* dbaseline,
                        float* grads, void* workspace, size_t workspace_bytes,
                        seedrl_stream_t stream);
/* Overlap of the data-parallel exchange (SURVEY 8e; the reference's strategy.run + cross-replica SUM,
 * agents/vtrace/learner.py:255-280, tests/utils_test.py:640-650): seedrl_net_backward plus a
 * cudaEvent_t recorded on `stream` once the first arena bucket -- floats
 * [0, seedrl_net_grad_split(net)): heads, Dense, LSTM -- is final, so its all-reduce can run on a side
 * stream during the convolution torso's backward. */
int seedrl_net_backward_overlap(const seedrl_net* net, const float* params, int T1, int B,
                                const int64_t* prev_actions, const float* reward, const uint8_t* done,
                                const uint8_t* observation, const float* dlogits, const float* dbaseline,
                                float* grads, void* workspace, size_t workspace_bytes,
                                void* head_ready_event, seedrl_stream_t stream);
size_t seedrl_net_grad_split(const seedrl_net* net);
/* The tcgen05 / persistent kernels never spin forever: a barrier wait that expires sets an
 * error flag in the workspace and the kernel bails out (its results are then garbage).
 * seedrl_net_forward clears the flag; this call copies it back (synchronising `stream`) and
 * returns SEEDRL_ERR_INTERNAL if any kernel of the last forward/backward on this workspace
 * set it.  (No reference analogue: TF raises from the op; here the caller polls at a point
 * that is synchronous anyway -- when it reads the loss.) */
int seedrl_net_check_error(const seedrl_net* net, int T1, int B, void* workspace,
                           size_t workspace_bytes, seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a7/a8) Per-environment state on the GPU.  Replaces
 * common/utils.py:119-257 UnrollStore.append/reset (scatter_nd_update on host
 * variables) and :461-543 Aggregator.{reset,add,read,replace} for one field.
 * `state` is [num_envs, full_length, row_bytes] bytes; `index` int32 [num_envs].
 */
int seedrl_store_append_field(uint8_t* state, const int32_t* index,
                              const int32_t* env_ids, int n, int full_length,
                              size_t row_bytes, const uint8_t* values,
                              seedrl_stream_t stream);
/* index[env]++ for env in env_ids; writes completed env ids (index reached
 * full_length) compacted IN env_ids ORDER into completed_ids and their count
 * into *num_completed (device int32). */
int seedrl_store_advance(int32_t* index, const int32_t* env_ids, int n,
                         int full_length, int32_t* completed_ids,
                         int32_t* num_completed, seedrl_stream_t stream);
/* For each completed env: copy its full unroll rows to `unrolls`
 * ([n_completed, full_length, row_bytes], env-major like the reference, or
 * time-major [full_length, n_completed, row_bytes] if time_major != 0, which
 * removes make_time_major, common/utils.py:735-761), then move the last
 * `overlap+1` rows to the front. */
int seedrl_store_gather_field(uint8_t* state, const int32_t* completed_ids,
                              int n_completed, int full_length, size_t row_bytes,
                              int overlap, int time_major, uint8_t* unrolls,
                              seedrl_stream_t stream);
/* (a6) Every per-environment row move of one inference batch in ONE launch: the reads of the
 * previous action / agent state (Aggregator.read, common/utils.py:504-516), their write-back
 * (Aggregator.replace, :519-543) and the append of all fields of the step to the unroll store
 * (UnrollStore.append, :187-190) -- agents/vtrace/learner.py:381-383,394-403 issues one TF op per
 * table.  mode 0 gather rows[j] = table[env_ids[j]]; 1 scatter; 2 append at index[env].  The
 * caller guarantees unique env_ids for scatter/append (the reference asserts it, :533-540). */
#define SEEDRL_MAX_ROW_JOBS 16
typedef struct seedrl_row_job {
  void* table;          /* [num_envs(, full_length), row_bytes] */
  void* rows;           /* [n, row_bytes] */
  size_t row_bytes;
  int32_t mode;
  int32_t full_length;  /* append only */
} seedrl_row_job;
int seedrl_rows_multi(const seedrl_row_job* jobs, int njobs, const int32_t* env_ids, int n,
                      const int32_t* index, seedrl_stream_t stream);
/* Zero-copy minibatch assembly (SURVEY 8(f) rank 2; replaces the queue-element copy, tf.stack and
 * make_time_major of agents/vtrace/learner.py:418-432): like seedrl_store_gather_field with
 * time_major = 1, but unroll i lands in column col0 + i of the caller's batch tensor
 * [full_length, batch_cols, row_bytes]. */
int seedrl_store_gather_field_into(uint8_t* state, const int32_t* completed_ids, int n_completed,
                                   int full_length, size_t row_bytes, int overlap, uint8_t* batch,
                                   int batch_cols, int col0, seedrl_stream_t stream);
int seedrl_store_finish(int32_t* index, const int32_t* completed_ids,
                        int n_completed, int overlap, seedrl_stream_t stream);
int seedrl_store_reset(uint8_t* state, int32_t* index, const int32_t* env_ids,
                       int n, int full_length, size_t row_bytes, int overlap,
                       seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * (a10) Inference batcher (host side).  Replaces the server-side dynamic
 * batcher grpc/ops/grpc.cc:591-861 (`DynamicFn`, `Computation`): callers claim
 * k contiguous slots of a fixed-size batch, copy their payload straight into a
 * pinned host slab, and block until the batch has been computed; the learner
 * thread waits for a full batch, runs it, publishes outputs and releases.
 * >= 2 batches in flight (grpc.cc:656-661).  No torch, no CUDA calls except
 * cudaHostAlloc/cudaFreeHost for the slabs.
 */
typedef struct seedrl_batcher seedrl_batcher;
/* in/out_row_bytes: bytes per batch row for each input / output field. */
int seedrl_batcher_create(int batch_size, int num_slabs, int n_in,
                          const size_t* in_row_bytes, int n_out,
                          const size_t* out_row_bytes, int pinned,
                          seedrl_batcher** out);
void seedrl_batcher_destroy(seedrl_batcher* b);
/* Caller side: claim k rows; returns slab id + first row (grpc.cc:638-663).
 * k > batch_size or a claim that would straddle a batch => OUT_OF_RANGE
 * (the reference CHECK-fails, grpc.cc:653). */
int seedrl_batcher_claim(seedrl_batcher* b, int k, int* slab, int* row);
void* seedrl_batcher_input_ptr(seedrl_batcher* b, int slab, int field, int row);
void* seedrl_batcher_output_ptr(seedrl_batcher* b, int slab, int field, int row);
/* Caller side: mark k rows written; when the slab is full the compute side wakes. */
int seedrl_batcher_commit(seedrl_batcher* b, int slab, int k);
/* Caller side: block until the slab's outputs are published (or shutdown ->
 * SEEDRL_ERR_CANCELLED "Server shutdown.", grpc.cc:771-787).  The caller then reads
 * its rows through seedrl_batcher_output_ptr and calls seedrl_batcher_release once
 * per successful claim; the slab is recycled when every claimant has released. */
int seedrl_batcher_wait_outputs(seedrl_batcher* b, int slab, int* status);
int seedrl_batcher_release(seedrl_batcher* b, int slab);
/* Compute side: block until some slab is full; returns its id
 * (SEEDRL_ERR_CANCELLED after shutdown). timeout_ms < 0 = forever. */
int seedrl_batcher_next_full(seedrl_batcher* b, int timeout_ms, int* slab);
/* Compute side: outputs are in place; wake the callers.  status != 0 is
 * propagated to every caller of this batch. */
int seedrl_batcher_publish(seedrl_batcher* b, int slab, int status);
int seedrl_batcher_shutdown(seedrl_batcher* b);

/* ------------------------------------------------------------------------
 * Per-category kernel timing for bench.py's profiling pass: between begin and end
 * every kernel launch of this library is followed by a CUDA event on its stream (a
 * kernel's time = the gap to the previous event, i.e. back-to-back device time);
 * end() synchronises and returns summed milliseconds and launch counts per category
 * (arrays of seedrl_profile_num_categories() entries).  Never on in a timed region. */
int seedrl_profile_num_categories(void);
const char* seedrl_profile_category_name(int i);
int seedrl_profile_begin(seedrl_stream_t stream);
int seedrl_profile_end(double* ms_per_category, uint64_t* launches_per_category);

/* ------------------------------------------------------------------------
 * R2D2 (SURVEY 8(a) row a11, BASELINE cfg 5): the agent network, then the post-network pieces.
 *
 * seedrl_r2d2_net_* <- atari/networks.py:221-340 (DuelingLSTMDQNNet: __call__/_unroll/_torso/_head)
 *   and :176-218 (_unroll_cell).  Parameters: one flat fp32 arena in
 *   tf.Module.trainable_variables order (_advantage, _body, _core, _value), Keras layouts.
 *   forward: time-major prev_actions int64 [T,B], reward [T,B], done uint8 [T,B], frames uint8
 *   [T,B,H,W,C] ALREADY STACKED (C = stack_size; seedrl_r2d2_stack_frames), h0/c0 [B,512] ->
 *   q_values [T,B,A], action int32 [T,B] (argmax, first maximum; may be NULL), h_out/c_out.
 *   backward: dq [T,B,A] -> grads (arena layout, overwritten); must follow the forward of the same
 *   (T,B) on the same workspace.  mode: 0 fp32 SIMT GEMMs, 2 (default) tcgen05 bf16x3.
 *   Errors: SEEDRL_ERR_INVALID_ARGUMENT for null / undersized buffers (the reference raises from
 *   TF shape checks); seedrl_r2d2_net_check_error as seedrl_net_check_error. */
typedef struct seedrl_r2d2_net seedrl_r2d2_net;
int seedrl_r2d2_net_create(int num_actions, int obs_h, int obs_w, int channels, seedrl_r2d2_net** out);
void seedrl_r2d2_net_destroy(seedrl_r2d2_net* net);
int seedrl_r2d2_net_num_param_tensors(const seedrl_r2d2_net* net);      /* 18 */
size_t seedrl_r2d2_net_num_params(const seedrl_r2d2_net* net);
size_t seedrl_r2d2_net_arena_floats(const seedrl_r2d2_net* net);
int seedrl_r2d2_net_set_mode(seedrl_r2d2_net* net, int mode);
int seedrl_r2d2_net_set_lstm_mode(seedrl_r2d2_net* net, int mode);   /* as seedrl_net_set_lstm_mode: 0 or 2 */
int seedrl_r2d2_net_param_info(const seedrl_r2d2_net* net, int index, char* name_buf, size_t name_buf_len,
                               int64_t* dims4, int* rank, size_t* offset_floats);
size_t seedrl_r2d2_net_workspace_bytes(const seedrl_r2d2_net* net, int T, int B);
int seedrl_r2d2_net_forward(const seedrl_r2d2_net* net, const float* params, int T, int B,
                            const int64_t* prev_actions, const float* reward, const uint8_t* done,
                            const uint8_t* frames, const float* h0, const float* c0, float* q_values,
                            int32_t* action, float* h_out, float* c_out, void* workspace,
                            size_t workspace_bytes, seedrl_stream_t stream);
/* `frames`: the stacked frames the forward of this unroll ran on (the first convolution's weight
 * gradient gathers its operand from them; nothing is kept of them in the workspace). */
int seedrl_r2d2_net_backward(const seedrl_r2d2_net* net, const float* params, int T, int B,
                             const uint8_t* frames, const uint8_t* done, const float* dq, float* grads,
                             void* workspace, size_t workspace_bytes, seedrl_stream_t stream);
int seedrl_r2d2_net_check_error(const seedrl_r2d2_net* net, int T, int B, void* workspace,
                                size_t workspace_bytes, seedrl_stream_t stream);

/*
 * seedrl_r2d2_stack_frames <- atari/networks.py:57-173 (stack_frames): frames uint8 [T,B,P]
 *   (P = prod(observation_shape), one channel), state int32 [B,P] bit-packed (LSB byte =
 *   oldest of the stack_size-1 kept frames), done [T,B].  stacked uint8 [T,B,P,stack_size],
 *   newest first, channels that cross an episode boundary zeroed (the reference returns the
 *   same values as float32; /255 is folded into the first convolution here).  Errors: the
 *   reference's "Only up to stack size 4 is supported due to bit-packing." */
int seedrl_r2d2_stack_frames(int T, int B, int P, int stack_size, const uint8_t* frames,
                             const int32_t* state_in, const uint8_t* done, uint8_t* stacked,
                             int32_t* state_out, seedrl_stream_t stream);
/* <- agents/r2d2/learner.py:258-330 (compute_loss_and_priorities_from_agent_outputs) with
 *   value_function_rescaling / inverse (:180-192) and n_step_bellman_target (:195-255), plus the
 *   gradient of mean_b(importance_weight_b * loss_b) (:604) w.r.t. q_train.  The greedy action
 *   of the online network is re-derived as argmax_a q_train (first maximum, like tf.argmax).
 *   loss, priorities: [B]; dq: [T,B,A]; scratch: seedrl_r2d2_loss_scratch_bytes. */
size_t seedrl_r2d2_loss_scratch_bytes(int T, int B, int n_steps);
int seedrl_r2d2_loss_fwd_bwd(int T, int B, int A, const float* q_train, const float* q_target,
                             const int64_t* replay_action, const float* reward, const uint8_t* done,
                             const float* importance_weights, float gamma, int n_steps, float eta,
                             float value_rescaling_eps, float* loss, float* priorities, float* dq,
                             void* scratch, seedrl_stream_t stream);
/* <- common/utils.py:327-352 (PrioritizedReplay.sample, priority_exp != 0): prob_i =
 *   prio_i^alpha / sum over the first `limit` slots; index_j = inverse CDF of uniforms[j] in
 *   [0,1) (the reference draws with tf.random.categorical: same distribution, different
 *   stream); weights_j = ((1/limit)/prob_{index_j})^beta / max_j.  probs_out may be NULL. */
int seedrl_replay_sample(int limit, const float* priorities, float priority_exp,
                         float importance_sampling_exp, int num_samples, const float* uniforms,
                         int64_t* indices, float* weights, float* probs_out, seedrl_stream_t stream);
/* <- tf.clip_by_global_norm (agents/r2d2/learner.py:608, clip_norm = 40) over the flat gradient
 *   arena: g *= clip_norm / max(||g||_2, clip_norm); *norm_out = ||g||_2 (may be NULL). */
size_t seedrl_clip_scratch_bytes(void);
int seedrl_clip_by_global_norm(size_t n, float* grads, float clip_norm, float* norm_out,
                               void* scratch, seedrl_stream_t stream);

/* ------------------------------------------------------------------------
 * Single-kernel test hooks: let the GPU parity tests localise a failure to one
 * kernel of the network schedule.  Not part of the drop-in surface.
 * in_mode: 0 fp32 input, 1 relu(input), 2 uint8 input / 255. */
int seedrl_debug_conv3x3(int cin, int cout, int in_mode, int N, int H, int W,
                         const void* in, const float* w, const float* bias,
                         const float* mask, const float* res, float* out,
                         seedrl_stream_t stream);
int seedrl_debug_conv3x3_flip(int cin, int cout, const float* w, float* wt,
                              seedrl_stream_t stream);
size_t seedrl_debug_wgrad_partial_bytes(void);
/* Host-side: the kernels' tall-image position -> pixel map (-1 = zero padding); which = 0
 * padded-input positions, 1 output positions.  CPU-only check of the multiply-high division. */
int seedrl_debug_conv_pixels(int N, int H, int W, int which, int start, int count, int* out);
/* 0: every shape takes vtrace_loss_kernel; 1 (default): large aligned batches take the
 * TMA-streamed vtrace_loss_stream_kernel.  Lets the tests run both on the same inputs. */
int seedrl_debug_set_loss_stream(int enabled);
/* K positions per pipeline stage of the tensor-core weight-gradient kernel: the largest of 512 / 256 / 128
 * not above `kc` whose stages fit shared memory is used (default 512). */
int seedrl_debug_set_wgrad_chunk(int kc);
/* Output positions per tile of the tensor-core forward / data-gradient kernel: the largest
 * of 512 / 256 / 128 not above `mt` that keeps two CTAs per SM is used (default 512). */
int seedrl_debug_set_conv_tile(int mt);
int seedrl_debug_set_gemm_bk(int bk);     /* gemm_tc_kernel K elements per staged block: 64 or 32 */
/* 0 = the im2col convolutions (IMPALA shallow net, R2D2 body) materialise their matrices instead of
 * gathering them while the GEMM stages its operand (default 1; bit-identical results). */
int seedrl_debug_set_gemm_gather(int on);
/* 1 = conv_mode 3 keeps the dense first-layer backward (pool backward + full-resolution weight
 * gradient) instead of csrc/conv_first.cu's gather from the pooled gradient (A/B parity tests). */
int seedrl_debug_set_first_layer_dense(int on);
/* The fused first layer (conv 4->16 on uint8 frames + bias + max-pool 3x3/2 SAME) on its own:
 * pooled plane tensors (raw, ReLU'd) + arg-max taps [N,Ho,Wo,16]. */
int seedrl_debug_conv0pool(int N, int H, int W, const uint8_t* frames, const float* w, const float* bias,
                           void* praw, void* prelu, uint8_t* idx, int* err, seedrl_stream_t stream);
int seedrl_debug_conv3x3_wgrad(int cin, int cout, int in_mode, int N, int H, int W,
                               const void* x, const float* dy, float* dw, float* db,
                               float* partial, size_t partial_bytes,
                               seedrl_stream_t stream);
/* tcgen05 (tensor-core, bf16 x bf16 -> fp32) 3x3 convolution: packs fp32 HWIO weights
 * (flip != 0: flipped + transposed, i.e. the data-gradient; split != 0: bf16x3 hi/lo
 * operands, fp32-faithful) into wq_scratch (>= 2*9*max(cin,16)*cout*2 bytes) and runs the implicit-GEMM kernel.  variant bit0/bit1 swap the
 * LBO/SBO fields of the A/B shared-memory descriptors (bring-up aid); *error_flag becomes 1
 * if the kernel's bounded mbarrier wait expires. */
int seedrl_debug_conv3x3_tc(int cin, int cout, int in_mode, int split, int N, int H, int W,
                            const void* in, const float* w, const float* bias,
                            const float* mask, const float* res, float* out, int flip,
                            int variant, void* wq_scratch, int* error_flag,
                            seedrl_stream_t stream);
/* tcgen05 weight gradient (MN-major operands, one TMEM accumulator per tap). */
int seedrl_debug_conv3x3_wgrad_tc(int cin, int cout, int in_mode, int split, int N, int H, int W,
                                  const void* x, const float* dy, float* dw, float* db,
                                  float* partial, size_t partial_bytes, int* error_flag,
                                  seedrl_stream_t stream);
int seedrl_debug_maxpool(int backward, int N, int H, int W, int C, const float* x_or_dy,
                         float* y_or_dx, uint8_t* idx, seedrl_stream_t stream);
/* C[M,N] (=|+=) op(A) op(B) on the tensor cores (tcgen05, bf16 or bf16x3 operands, fp32
 * accumulate): ta: A stored [K,M]; tb: B stored [N,K]; epilogue bias / relu / mask / accumulate
 * as seedrl_debug_sgemm.  ws (may be NULL) takes split-K partials. */
int seedrl_debug_gemm_tc(int ta, int tb, int split, int M, int N, int K, const float* A, int lda,
                         const float* B, int ldb, float* C, int ldc, const float* bias,
                         const float* mask, int ldm, int relu, int accumulate, int a_relu,
                         float* ws, size_t ws_bytes, int* error_flag, seedrl_stream_t stream);
/* out[n] = sum_m X[m*ld + n] (the bias gradients, reference Dense / Conv2D bias variables); ws (may be
 * NULL) is scratch for the row-slab path taken by tall dense matrices (ld == N, N a power of two). */
int seedrl_debug_colsum(int M, int N, const float* X, int ld, float* out, float* ws, size_t ws_bytes,
                        seedrl_stream_t stream);
int seedrl_debug_sgemm(int ta, int tb, int M, int N, int K, const float* A, int lda,
                       const float* B, int ldb, float* C, int ldc, const float* bias,
                       const float* mask, int ldm, int relu, int accumulate, int a_relu,
                       seedrl_stream_t stream);

/* ---- plane-tensor convolution path (conv_mode 3) test hooks: single kernels of
 * csrc/conv_planes.cu, so the GPU parity tests can localise a failure.  Not on the product path. */
size_t seedrl_debug_planes_bytes(int N, int H, int W, int C);
int seedrl_debug_to_planes(int N, int H, int W, int C, int relu, const float* x, void* out,
                           seedrl_stream_t stream);
int seedrl_debug_from_planes(int N, int H, int W, int C, const void* in, float* y,
                             seedrl_stream_t stream);
int seedrl_debug_convp(int cin, int cout, int N, int H, int W, const void* in, const float* w,
                       const float* bias, const void* mask, const void* res, int flip,
                       void* out_raw, void* out_relu, float* out_nhwc, void* wq_scratch,
                       int* error_flag, seedrl_stream_t stream);
int seedrl_debug_wgradp(int cin, int cout, int N, int H, int W, const void* x, const void* dy,
                        float* dw, float* db, float* partial, size_t partial_bytes,
                        int* error_flag, seedrl_stream_t stream);
int seedrl_debug_poolp(int backward, int N, int H, int W, int C, const void* in, void* out_raw,
                       void* out_relu, float* out_nhwc, uint8_t* idx, seedrl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif  /* SEEDRL_B200_H_ */
