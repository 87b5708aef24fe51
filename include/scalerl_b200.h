/* scalerl_b200 -- C ABI of the B200-native IMPALA learner hot path.
 *
 * The reference (jianzhnie/ScaleRL) is 100 % Python and has no FFI; the interface these entry points
 * replace is the Python one of scalerl/algorithms/impala (file:line given per function).  A host
 * binds them with ctypes (see INTEGRATION.md and scalerl_b200/_lib.py).  Plain pointers and sizes
 * only -- no torch types.  Every pointer is a DEVICE pointer unless the name ends in `_host`.
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Return value: 0 on
 * success, otherwise a cudaError_t (>0) or a negative SRL_E* argument error; srl_last_error()
 * returns a message for the calling thread.  Nothing here synchronises the stream.
 */
#ifndef SCALERL_B200_H_
#define SCALERL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRL_EINVAL (-1)   /* bad argument (shape / alignment / NULL) */
#define SRL_ESTATE (-2)   /* call order violated */

const char* srl_last_error(void);
int srl_version(void);

/* ---- V-trace -------------------------------------------------------------------------------------------
 * replaces vtrace.from_importance_weights (scalerl/algorithms/impala/vtrace.py:78-172).
 * log_rhos, discounts, rewards, values: f32 [T,B] row-major; bootstrap_value f32 [B]; outputs f32 [T,B].
 * clip thresholds < 0 mean None (no clipping), as the Python API's clip_*=None.
 * variant: 0 = column-sequential (float4 over B when B%4==0), 1 = warp-shuffle affine scan over T. */
int srl_vtrace_from_importance_weights(const float* log_rhos, const float* discounts, const float* rewards,
                                       const float* values, const float* bootstrap_value, int T, int B,
                                       float clip_rho_threshold, float clip_pg_rho_threshold,
                                       float* vs, float* pg_advantages, int variant, void* stream);

/* replaces vtrace.from_logits (vtrace.py:43-75): logits f32 [T,B,A], actions i64 [T,B].
 * Outputs (any may be NULL except vs/pg): vs, pg_advantages, log_rhos, behavior_alp, target_alp, all f32 [T,B]. */
int srl_vtrace_from_logits(const float* behavior_policy_logits, const float* target_policy_logits,
                           const int64_t* actions, const float* discounts, const float* rewards,
                           const float* values, const float* bootstrap_value, int T, int B, int A,
                           float clip_rho_threshold, float clip_pg_rho_threshold,
                           float* vs, float* pg_advantages, float* log_rhos, float* behavior_action_log_probs,
                           float* target_action_log_probs, void* stream);

/* ---- fused learner tail: learn() pre-processing + V-trace + the three losses + head gradients ----------
 * replaces impala_atari.py:293-330 + loss_fn.py:5-23 + the autograd step from total_loss to
 * (policy_logits, baseline).  Inputs are the [T+1,B] batch rows as they lie in the trajectory batch
 * (impala_atari.py:122-151): the kernel applies the [1:] / [:-1] shifts itself.
 *   behavior_logits f32 [T+1,B,A] (batch['policy_logits']), target_logits f32 [T+1,B,A] and baseline f32 [T+1,B]
 *   (learner outputs), action i64 [T+1,B], reward f32 [T+1,B], done u8/bool [T+1,B].
 * Outputs: vs, pg_advantages f32 [T,B]; dlogits f32 [T,B,A]; dbaseline f32 [T,B];
 *   losses f32 [4] = {pg_loss, baseline_loss (x baseline_cost), entropy_loss (x entropy_cost), total}.
 * scratch: zero-initialised f32 [3*ceil(B/4)+4] workspace (block partials + ticket; re-armed by the kernel). */
int srl_impala_loss_and_head_grads(const float* behavior_logits, const float* target_logits, const float* baseline,
                                   const int64_t* action, const float* reward, const uint8_t* done,
                                   int T, int B, int A, float discounting, int reward_clip_abs_one,
                                   float clip_rho_threshold, float clip_pg_rho_threshold,
                                   float baseline_cost, float entropy_cost,
                                   float* vs, float* pg_advantages, float* dlogits, float* dbaseline,
                                   float* losses, float* scratch, void* stream);

/* ---- row-wise policy ops: the pieces of loss_fn.py / vtrace.action_log_probs as stand-alone, differentiable operators ------
 * (used by the autograd drop-ins scalerl_b200/algorithms/impala/{loss_fn,vtrace}.py; the learner step itself uses the fused tail)
 * forward : logp[n] = log_softmax(logits[n])[actions[n]] (vtrace.py:31-40; loss_fn.py:16-23), ent[n] = sum_a p log p (loss_fn.py:9-13);
 *           logits f32 [N,A], actions i64 [N]; either output may be NULL (actions may be NULL when logp is).
 * backward: dlogits[n][a] = w_logp[n] * (1{a == actions[n]} - p[a]) + w_ent[n] * p[a] * (log p[a] - ent[n]) -- the gradient of
 *           sum_n w_logp[n] logp[n] + w_ent[n] ent[n]; a NULL weight array means zeros.
 * srl_reduce_sum: out[0] = scale * sum x[i] (square = 0) or scale * sum x[i]^2 (square = 1), fixed summation order
 *           (loss_fn.py:5-6 compute_baseline_loss = 0.5 * sum(adv^2)). */
int srl_policy_rows_forward(const float* logits, const int64_t* actions, int64_t N, int A, float* logp, float* ent, void* stream);
int srl_policy_rows_backward(const float* logits, const int64_t* actions, const float* w_logp, const float* w_ent, int64_t N, int A,
                             float* dlogits, void* stream);
int srl_reduce_sum(const float* x, int64_t n, int square, float scale, float* out, void* stream);
/* actions[n] ~ softmax(logits[n]) through the inverse CDF of uniforms[n] in [0,1) (torch.multinomial of AtariNet.forward in training
 * mode, atari_model.py:130-132); uniforms == NULL: argmax (evaluation mode, :133-134).  logits f32 [N,A], actions i64 [N]. */
int srl_sample_actions(const float* logits, const float* uniforms, int64_t N, int A, int64_t* actions, void* stream);

/* ---- learner context: encoder fwd/bwd on tcgen05 + heads + optimizer ------------------------------------
 * replaces AtariNet.forward (scalerl/algorithms/utils/atari_model.py:77-143, use_lstm=False) and
 * ImpalaTrainer.learn (impala_atari.py:270-349) for one GPU's shard of the batch.                         */
typedef struct srl_learner srl_learner_t;

typedef struct srl_config {
  int32_t T;                 /* rollout_length                                   */
  int32_t B;                 /* batch columns processed by THIS GPU              */
  int32_t A;                 /* num_actions (<= 31)                              */
  int32_t optimizer;         /* 0 = RMSprop (reference, impala_atari.py:99-105), 1 = Adam */
  int32_t reward_clip_abs_one;
  int32_t precision;         /* encoder operand precision: 0 = bf16 (default, the measured configuration); 1 = fp32-accurate:
                              * every bf16 operand tensor gets a low twin bf16(v - bf16(v)) and each tensor-core product runs as
                              * hi*hi + hi*lo + lo*hi into the fp32 TMEM accumulator (16 significant operand bits, tighter than
                              * kind::tf32's 11) -- the whole-step parity mode SURVEY.md §7.9 asks for; ~3x the MMAs */
  float discounting, baseline_cost, entropy_cost;
  float clip_rho_threshold, clip_pg_rho_threshold;   /* < 0: None */
  float max_grad_norm;       /* clip_grad_norm_ threshold (rl_args.py:108)       */
  float learning_rate, alpha, epsilon;               /* RMSprop (rl_args.py:112-117) */
  float adam_beta1, adam_beta2, adam_eps;
  int32_t use_lstm;          /* 1: AtariNet(use_lstm=True): 2-layer LSTM core between the encoder and the heads (config 5) */
} srl_config_t;

/* Number of fp32 elements of the flat parameter buffer for A actions, and the element offset / count of
 * each of the 12 AtariNet tensors in state_dict order (conv1.weight, conv1.bias, ..., baseline.bias),
 * PyTorch layouts.  Segments are padded to multiples of 4 floats. offsets/counts: int64[12], indexed in state_dict order;
 * in memory the small tensors come first and fc.weight last (offsets[6] is the largest), so [0, offsets[6]) is the
 * "small" gradient block and [offsets[6], total) is fc.weight. */
int64_t srl_param_layout(int A, int64_t* offsets, int64_t* counts);

/* Same with the 8 LSTM tensors (nn.LSTM state_dict order: weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0, *_l1) appended
 * after fc.weight when use_lstm != 0: offsets/counts are int64[20] (entries 12..19 = LSTM; unused when use_lstm == 0). */
int64_t srl_param_layout_ex(int A, int use_lstm, int64_t* offsets20, int64_t* counts20);

/* params / grads / opt_state0 / opt_state1: flat f32 device buffers of srl_param_layout() (srl_param_layout_ex() with use_lstm) elements, owned
 * by the caller (so torch can expose state_dict views and NCCL can all-reduce `grads` in place).
 * opt_state1 is only used by Adam (may be NULL for RMSprop). */
int srl_learner_create(const srl_config_t* cfg, float* params, float* grads, float* opt_state0, float* opt_state1,
                       srl_learner_t** out);
int srl_learner_destroy(srl_learner_t* L);
/* Diagnostics builds only (SRL_DEFINES=SRL_KSTAMP; tests/diag/diag_timeline.py): `buffer` = 1 + 3*2000 uint64 of device memory, zeroed by the
 * caller; every kernel then appends {kernel id, %globaltimer at entry, %globaltimer when its stream predecessor had completed} (word 0 = count).
 * NULL switches the stamps off.  The product build returns SRL_ESTATE. */
int srl_debug_kernel_timeline(void* buffer);
/* bytes of device workspace held by the context */
int64_t srl_learner_workspace_bytes(const srl_learner_t* L);
/* update a hyper-parameter that does not change buffer sizes (lr, costs, clip...) */
int srl_learner_set_config(srl_learner_t* L, const srl_config_t* cfg);

/* run-time switch of one learner context: "column_fusion" (default 1; 0 = three kernels head_fwd / impala_tail / head_bwd
 * instead of the fused column kernel -- the environment variable SRL_NO_COLUMN_FUSION is read once, at creation). */
int srl_learner_set_option(srl_learner_t* L, const char* name, int value);

/* optimizer step count (Adam's bias-correction t; torch.optim state['step']): restore it when resuming from a checkpoint
 * (host counter and the device-resident counter the captured graphs read).  Both synchronise `stream`. */
int srl_learner_set_step(srl_learner_t* L, int64_t step, void* stream);
int64_t srl_learner_get_step(srl_learner_t* L, void* stream);

/* re-derive the packed bf16 operand copies from the fp32 master parameters now (optional: every forward does it) */
int srl_learner_pack_weights(srl_learner_t* L, void* stream);

/* AtariNet.forward for n_rows*B frames: obs u8 [rows,B,4,84,84], reward f32 [rows,B], action i64 [rows,B]
 * -> policy_logits f32 [rows,B,A], baseline f32 [rows,B].  rows <= T+1. */
int srl_learner_forward(srl_learner_t* L, const uint8_t* obs, const float* reward, const int64_t* action, int rows,
                        float* policy_logits, float* baseline, void* stream);

/* forward + V-trace + losses + full backward.  Leaves SUM-reduced gradients (loss_fn.py sums) in `grads`
 * and {pg, baseline, entropy, total} in losses[4]; vs/pg_advantages (f32 [T,B]) may be NULL. */
int srl_learner_forward_backward(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                 const int64_t* action, const float* behavior_logits,
                                 float* losses, float* vs, float* pg_advantages, void* stream);

/* use_lstm variants (SURVEY.md §8 row a17).  h0/c0: initial LSTM state f32 [2,B,513+A] (create_rnn_state_buffers,
 * impala_atari.py:108-120); rows of the forward must be T+1.  hT/cT (may be NULL) receive the state after the last row. */
int srl_learner_forward_lstm(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done, const int64_t* action,
                             const float* h0, const float* c0, float* policy_logits, float* baseline, float* hT, float* cT, void* stream);
int srl_learner_forward_backward_lstm(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                      const int64_t* action, const float* behavior_logits, const float* h0, const float* c0,
                                      float* losses, float* vs, float* pg_advantages, void* stream);

/* The same step in two halves, for overlapping the gradient all-reduce with the backward pass:
 *   _begin : forward + V-trace/loss + head backward + the fc layer's backward.  On return (in stream order) the
 *            fc.weight / fc.bias segments of `grads` (95 % of the bytes) are final -> start their all-reduce.
 *   _finish: conv3 / conv2 / conv1 backward; afterwards the remaining segments are final.
 * srl_learner_forward_backward == _begin followed by _finish. */
int srl_learner_forward_backward_begin(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                       const int64_t* action, const float* behavior_logits,
                                       float* losses, float* vs, float* pg_advantages, void* stream);
int srl_learner_backward_finish(srl_learner_t* L, const uint8_t* obs, void* stream);

/* clip_grad_norm_(max_grad_norm) over `grads` (after the caller's all-reduce, if any) + optimizer step.
 * grad_norm_out: f32 [2] = {total L2 norm, clip coefficient} (may be NULL).  The bf16 operand copies of the weights
 * are re-derived at the start of the next srl_learner_forward* call. */
int srl_learner_apply_gradients(srl_learner_t* L, float* grad_norm_out, void* stream);

/* Data-parallel apply step over peer memory, replacing ncclAllReduce + srl_learner_apply_gradients (impala_atari.py:344-346
 * on every rank): reduce-scatter of the flat gradient through NVLink loads, global-norm clip, optimizer and all-gather in ONE
 * cooperative kernel (see heads_optim.cu).  grads[i] / exchange[i] / ctl[i] (i < world) are rank i's gradient buffer, its
 * exchange buffer (4 * ceil(n/4 / world) + 4 floats: the reduced slice the peers pull) and its 1 KiB control block, all
 * mapped into this process (symmetric memory / CUDA IPC); grads[rank] must be the buffer given to srl_learner_create; the
 * control blocks start zeroed.  Every rank must call it once per step.  On return (stream order) the
 * local gradient buffer holds the SUM over ranks, as after ncclAllReduce. */
typedef struct {
  void* grads[8]; void* exchange[8]; void* ctl[8]; int rank; int world;
  void* grads_multicast;   /* NVLS multicast address of the gradient buffers (NULL: peer loads).  When set, the reduce-scatter is one
                            * multimem.ld_reduce per 16 bytes (the NVSwitch adds the copies) and the all-gather one multimem.st */
} srl_dp_peers_t;
int srl_learner_apply_gradients_dp(srl_learner_t* L, const srl_dp_peers_t* peers, float* grad_norm_and_coef_out, void* stream);

/* Weight-publish snapshot (impala_atari.py:348, actor_model.load_state_dict(learner_model.state_dict())): copies the flat fp32
 * parameters to `dst` (same layout, srl_param_layout elements) on `stream` -- unless losses[3] (the step's total loss, device
 * f32[4]; may be NULL = unconditional) is NaN/Inf, in which case `dst` keeps the last good weights.  The caller then copies
 * `dst` to the actors' host memory asynchronously while the next step already updates the live parameters. */
int srl_learner_snapshot_params(srl_learner_t* L, float* dst, const float* losses, void* stream);

/* borrow internal activations / operand copies for tests: name in {"a1","a2","a3","h","logits","baseline",
 * "dlogits","dbaseline","dh","da3","da2","da1","wpack"}; returns device pointer + element count. */
int srl_learner_debug_buffer(srl_learner_t* L, const char* name, void** ptr, int64_t* count);

/* per-kernel timing of one learner step: when enabled every kernel launch of forward_backward /
 * apply_gradients is bracketed by cudaEventRecord on the caller's stream; profile_collect() synchronises
 * on those events and writes milliseconds per slot (-1 for slots not executed) to a HOST array of
 * srl_profile_slot_count() floats. */
int srl_learner_set_profiling(srl_learner_t* L, int enable);
int srl_profile_slot_count(void);
const char* srl_profile_slot_name(int slot);
int srl_learner_profile_collect(srl_learner_t* L, float* ms_out_host);

/* pin / unpin caller-owned HOST memory (trajectory ring slots: the pageable torch.stack + .to(device) of impala_atari.py:248-265
 * becomes direct DMA; actor parameters in shared memory: the target of the weight publish, impala_atari.py:348).  Registering a
 * range that a stale or enclosing registration already covers succeeds. */
int srl_host_register(void* ptr_host, int64_t bytes);
int srl_host_unregister(void* ptr_host);

/* asynchronous device-to-device copy on `stream` (used by tests to read the borrowed buffers) */
int srl_memcpy_d2d(void* dst, const void* src, int64_t bytes, void* stream);

/* ---- LSTM core (AtariNet use_lstm=True; atari_model.py:52-55,109-120; SURVEY.md §8 row a17) -------------------------------
 * 2-layer LSTM(H, H), H = 513 + A, stepped with the state multiplied by (1 - done_t) before every step.
 * weights8 / grads8: 8 device pointers in nn.LSTM state_dict order {weight_ih_l0 [4H,H], weight_hh_l0 [4H,H], bias_ih_l0 [4H],
 * bias_hh_l0 [4H], *_l1 ...} (fp32, caller-owned); gradients are ACCUMULATED into grads8 (zero them before the step).
 * forward : core f32 [T1,B,H], done u8 [T1,B], h0/c0 f32 [2,B,H] -> out f32 [T1,B,H], hT/cT f32 [2,B,H] (may be NULL)
 * backward: dout f32 [T1-1,B,H] (steps 0..T-1; the bootstrap row T carries no gradient) -> dcore f32 [T1-1,B,H] */
typedef struct srl_lstm srl_lstm_t;
int srl_lstm_create(int T1, int B, int H, const float* const* weights8, float* const* grads8, srl_lstm_t** out);
int srl_lstm_destroy(srl_lstm_t* L);
int srl_lstm_forward(srl_lstm_t* L, const float* core, const uint8_t* done, const float* h0, const float* c0, float* out,
                     float* hT, float* cT, void* stream);
int srl_lstm_backward(srl_lstm_t* L, const float* dout, const uint8_t* done, float* dcore, void* stream);
const char* srl_lstm_last_error(void);

/* ---- prioritized-replay sampler (BASELINE.json configs[3]; SURVEY.md §8f) ---------------------------------------------------
 * Device-resident float64 sum/min segment trees; replaces PrioritizedReplayBuffer's tree arithmetic
 * (scalerl/data/replay_buffer.py:305-381 over scalerl/data/segment_tree.py:7-196).  Index results are identical to the
 * reference's Python-float trees given identical leaf values.  The transition storage itself stays with the caller. */
typedef struct srl_per srl_per_t;
int srl_per_create(int64_t memory_size, double alpha, srl_per_t** out);
int srl_per_destroy(srl_per_t* P);
int64_t srl_per_size(const srl_per_t* P);
int64_t srl_per_capacity(const srl_per_t* P);
int srl_per_add(srl_per_t* P, int64_t n, void* stream);                                  /* _add x n  (replay_buffer.py:318-322) */
int srl_per_update_priorities(srl_per_t* P, const int64_t* idxs, const double* priorities, int64_t n, void* stream);   /* :346-351 */
/* pairs skipped so far by srl_per_update_priorities because idx was outside [0, size) or priority <= 0 (the reference asserts
 * both, replay_buffer.py:346-351); synchronises `stream`; -1 on error */
int64_t srl_per_invalid_updates(srl_per_t* P, void* stream);
int srl_per_sample(srl_per_t* P, const double* uniforms, int batch, double beta, int64_t* idxs, double* weights64,
                   float* weights32, void* stream);                                      /* :353-381, uniforms f64 [batch] in [0,1) */
int srl_per_debug_trees(srl_per_t* P, double* sum_out, double* min_out, double* max_priority_out, void* stream);
const char* srl_per_last_error(void);

/* ---- trajectory ring -> time-major batch (the stacking step of ImpalaTrainer.get_batch, impala_atari.py:248-251) -----------
 * staging: B trajectory slots on the DEVICE, each one contiguous record of slot_bytes holding every key of create_buffers
 * (impala_atari.py:135-147) for T+1 steps; offsets6_host (HOST array) = byte offsets of {obs u8[T+1,4,84,84], reward f32[T+1],
 * done u8[T+1], action i64[T+1], policy_logits f32[T+1,A], episode_return f32[T+1]} inside a slot.
 * Outputs: the time-major batch tensors [T+1,B,...] (episode_return may be NULL). */
int srl_unpack_slots(const uint8_t* staging, int64_t slot_bytes, const int64_t* offsets6_host, int T, int B, int A,
                     uint8_t* obs, float* reward, uint8_t* done, int64_t* action, float* policy_logits, float* episode_return,
                     void* stream);

/* ---- stand-alone optimizer ops (flat f32 buffers of n elements) ------------------------------------------
 * srl_grad_norm_clip_coef: coef[0] = ||g||_2, coef[1] = min(1, max_norm/(||g||+1e-6)); scratch f32[>=1028]. */
int srl_grad_norm_clip_coef(const float* grads, int64_t n, float max_norm, float* coef, float* scratch, void* stream);
int srl_rmsprop_step(float* params, const float* grads, float* square_avg, int64_t n, const float* coef,
                     float lr, float alpha, float eps, void* stream);
int srl_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* coef,
                  float lr, float beta1, float beta2, float eps, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCALERL_B200_H_ */
