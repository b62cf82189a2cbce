/*
 * parl_b200 — C ABI of the B200 (sm_100a) actor-learner hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): plain pointers and sizes, no
 * torch / C++ types.  Every entry point names the PaddlePaddle/PARL code whose
 * arithmetic it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *   - All data pointers are DEVICE pointers owned by the caller (e.g.
 *     torch.Tensor.data_ptr()); the library never allocates or frees
 *     user-visible memory.  `workspace` is caller-allocated scratch.
 *   - Work is enqueued on `stream` (a cudaStream_t passed as void*); no call
 *     synchronises the device or blocks the host.
 *   - Return value: RL_OK (0) or a negative RL_ERR_* code; rl_last_error()
 *     returns a thread-local message.  No exceptions cross the ABI.
 *   - "time-major" = [T, B, ...] contiguous; "env-major" = the reference's flat
 *     [B*T, ...] with index b*T + t (examples/IMPALA/actor.py:79-89).
 *   - Losses are written to device memory (`losses`), never read back here.
 */
#ifndef PARL_B200_H_
#define PARL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_OK 0
#define RL_ERR_BAD_ARG (-1)
#define RL_ERR_ALIGN (-2)
#define RL_ERR_CUDA (-3)
#define RL_ERR_UNSUPPORTED (-4)
#define RL_ERR_WORKSPACE (-5)

#define RL_LAYOUT_TIME_MAJOR 0
#define RL_LAYOUT_ENV_MAJOR 1

typedef void* rl_stream_t; /* cudaStream_t */

int rl_abi_version(void);
const char* rl_last_error(void);
/* Number of SMs / device name probe used by the host side for grid sizing. */
int rl_device_sm_count(int device);
/* Cap the CTA count of the persistent network kernels (conv forward / dgrad / wgrad) launched AFTER the call
 * (0 = one CTA per SM).  A pipelined engine caps its actor-side and learner-side kernels so that both streams'
 * grids are resident together instead of serialising; process-wide setting, read at launch (baked into a graph
 * at capture). */
int rl_set_sm_limit(int max_ctas);

/* Bytes of zero-initialised scratch the loss kernels need for a problem with
 * `n_cols` independent columns (B) — partial sums + the last-block ticket.
 * The caller zeroes it ONCE (cudaMemset / torch.zeros); kernels leave it zeroed. */
size_t rl_loss_workspace_bytes(int n_cols);

/* Triage hook: 1 forces the cp.async tile path of rl_vtrace_loss_fwd_bwd, 0 (default) lets the
 * TMA tensor-map path run when the layout allows it. */
/* 1: the per-env-step chain kernels (observation gather, TMA-window convs, GEMMs, env step) are launched with
 * programmatic stream serialization: each starts its prologue while the previous kernel of the stream drains and
 * blocks on griddepcontrol.wait before touching dependent memory.  0 (default): plain stream order — measured equal
 * for the graph-replayed rollout and slower for the pipelined step (profiles/r02_pdl_ab.txt). */
int rl_debug_set_pdl(int enable);
int rl_debug_set_tma(int disable);
/* Triage hook for rl_vtrace_loss_fwd_bwd: 0 = default (the v8 kernel for time-major, TMA-able shapes with T <= 64,
 * B % 4 == 0, even A <= 18 and int32 actions; the general v4 kernel otherwise), 4 = v4 always, 8 / 9 = v8 without /
 * with programmatic dependent launch (measured equal: profiles/r02_k1_matrix_g.jsonl), 10 / 11 = v8 with 256-byte / no L2
 * promotion in the logits tensor maps (no effect: profiles/r02_k1_l2_promotion.jsonl). */
int rl_debug_set_vtrace_path(int mode);

/* ------------------------------------------------------------------------
 * a1  V-trace returns.
 * Replaces parl/algorithms/paddle/impala/vtrace.py:36-139
 * (from_importance_weights).  All inputs [T,B] float32 time-major,
 * bootstrap [B]; outputs vs, pg_advantages [T,B].  clip thresholds < 0 mean
 * "None" (no clipping), matching vtrace.py:104-107,130-133.
 * ---------------------------------------------------------------------- */
int rl_vtrace_from_importance_weights(
    const float* behaviour_actions_log_probs, const float* target_actions_log_probs,
    const float* discounts, const float* rewards, const float* values,
    const float* bootstrap_value, int T, int B,
    float clip_rho_threshold, float clip_pg_rho_threshold,
    float* vs, float* pg_advantages, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a1+a2+a3  Fused IMPALA loss: log-softmax, entropy, KL, V-trace backward
 * scan, policy-gradient + value + entropy loss AND its gradient w.r.t. the
 * network outputs, one launch.
 * Replaces parl/algorithms/paddle/impala/impala.py:148-208 (post-network part
 * of IMPALA.learn), impala.py:25-79 (VTraceLoss) and vtrace.py:99-139.
 *
 *   target_logits, behaviour_logits : [T,B,A] f32   (T = sample_batch_steps,
 *                                      the LAST row is only the bootstrap row)
 *   actions  : [T,B] int32 (actions_i64=0) or int64 (actions_i64=1)
 *   rewards  : [T,B] f32 ; dones : [T,B] u8 (bool) ; values : [T,B] f32
 *   layout   : RL_LAYOUT_TIME_MAJOR or RL_LAYOUT_ENV_MAJOR (applies to all)
 *   losses   : [5] f32 device = {total, pi_loss, vf_loss, entropy, kl}
 *              (SUM reductions over the (T-1)*B kept rows; kl = MEAN over T*B)
 *   d_logits : [T,B,A] f32 = d total / d target_logits (row T-1 = 0)
 *   d_values : [T,B]   f32 = d total / d values        (row T-1 = 0)
 *   vs_out, pg_adv_out : optional [T-1,B] time-major f32 (may be NULL)
 * ---------------------------------------------------------------------- */
int rl_vtrace_loss_fwd_bwd(
    const float* target_logits, const float* behaviour_logits, const void* actions, int actions_i64,
    const float* rewards, const uint8_t* dones, const float* values,
    int T, int B, int A, int layout,
    float gamma, float clip_rho_threshold, float clip_pg_rho_threshold,
    float vf_loss_coeff, float entropy_coeff,
    float* losses, float* d_logits, float* d_values, float* vs_out, float* pg_adv_out,
    void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a10/a11  On-device vectorised actor pool (K5 env step + K7 sampling).
 * Replaces parl/env/vector_env.py:41-63 (VectorEnv.step, auto-reset),
 * the mock envs parl/tests/gym.py:117-207, FrameStack
 * (parl/env/atari_wrappers.py:270-307) and per-row action sampling
 * (examples/IMPALA/atari_agent.py:39-40, parl/algorithms/torch/ppo.py:164-177).
 * RNG: Philox4x32-10, counter (env_offset+b, step, block, stream), key = seed.
 *
 * Episode bookkeeping (all envs): ep_ret f32[B], ep_len i32[B] running values;
 * totals f32[4] = {#completed, sum return, sum length, -}; optional ring of the
 * most recent completed episodes (ring_ret f32[cap], ring_len i32[cap],
 * ring_head u32[1]) — the device analogue of MonitorEnv.next_episode_results()
 * (examples/IMPALA/actor.py:93-102).
 * ---------------------------------------------------------------------- */

/* Atari-shaped synthetic env.  Writes frame (step+1) of every env into
 * `frame_out` ([B,HW] uint8 plane of the caller's frame ring), reward/done of
 * step `step`, and age_out = done ? 0 : min(age_in+1, 3) (frames of the virtual
 * 4-stack that belong to the current episode).  If `logits` != NULL also samples
 * actions_out[b] ~ Categorical(logits[b,:A]) with the exact inverse-CDF rule.
 * reset=1: only emit frame `step` into frame_out and zero age/episode state.
 * step_dev: optional device-resident step index overriding `step` (lets a captured CUDA graph of
 * a whole rollout be replayed with advancing counters). */
int rl_env_atari_synth_step(
    uint8_t* frame_out, float* reward_out, uint8_t* done_out,
    const uint8_t* age_in, uint8_t* age_out,
    const float* logits, int A, int32_t* actions_out,
    float* ep_ret, int32_t* ep_len, float* totals,
    float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap,
    int B, int HW, uint64_t seed, uint32_t step, const uint32_t* step_dev, uint32_t env_offset, float p_done,
    int reset, rl_stream_t stream);

/* rl_env_atari_synth_step for step row t of a frame ring `planes` [P,B,7056] (84x84 frames; the new frame goes to
 * planes[t+4]) fused with rl_obs_stack_gather(out_dtype 4) of the NEXT step: obs_next [B,21,21,64] uint8 receives
 * obs(t+1) — the new frame is taken from shared memory, the older frames of the stack from the ring.  Bit-identical to
 * the two separate calls; saves one launch per env step of the actor chain (VectorEnv.step + the agent's obs handling,
 * parl/env/vector_env.py:41-63, examples/IMPALA/actor.py:60-75). */
int rl_env_atari_synth_step_gather(
    uint8_t* planes, int t, float* reward_out, uint8_t* done_out, const uint8_t* age_in, uint8_t* age_out,
    const float* logits, int A, int32_t* actions_out,
    float* ep_ret, int32_t* ep_len, float* totals, float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap,
    int B, uint64_t seed, uint32_t step, const uint32_t* step_dev, uint32_t env_offset, float p_done,
    uint8_t* obs_next, rl_stream_t stream);

/* Materialise observations from the frame ring: obs(t,b) channel j (0 = oldest)
 * = plane[t + 3 - min(3-j, age[t,b])].  planes [P,B,HW] u8, ages [>=t_begin+t_count, B] u8.
 * Output [t_count*B, 4, HW] in time-major or env-major sample order;
 * out_dtype 0 = uint8, 1 = float32 (value * scale), both [n,4,HW] (NCHW);
 * out_dtype 2 = bfloat16 [n,HW,4] (NHWC, value * scale) — the network input transform fused in;
 * out_dtype 3 = bfloat16 [n,21,21,64]: conv1's space-to-depth form (8x8/4/pad-1 conv == 2x2/1 conv over 4x4
 *               pixel blocks, channel = (dy*4+dx)*4+c, zero outside the image), 84x84 frames only; with
 *               ages == NULL `planes` is an already stacked uint8 tensor [t_count*B, 4, 84, 84];
 * out_dtype 4 = uint8   [n,21,21,64]: the same space-to-depth layout with the bytes untouched (scale unused) — the
 *               input of rl_conv2d_s1_u8in_bf16_{fwd,wgrad}, which apply the /255 of the reference model
 *               (benchmark/torch/a2c/atari_model.py:41, examples/IMPALA/atari_model.py) while widening to bf16
 *               in shared memory. */
int rl_obs_stack_gather(
    const uint8_t* planes, const uint8_t* ages, int B, int HW, int t_begin, int t_count,
    int out_layout, int out_dtype, float scale, void* out, rl_stream_t stream);

/* MuJoCo-shaped synthetic env: obs ~ N(0,1)^obs_dim, reward in {0,1}, done ~ p_done
 * (optionally also at max_episode_steps; 0 = no limit).  On done the returned obs is
 * the reset obs (vector_env.py:56-57) — every obs is a fresh draw. */
int rl_env_mujoco_synth_step(
    float* obs_out, float* reward_out, uint8_t* done_out,
    float* ep_ret, int32_t* ep_len, float* totals,
    float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap,
    int B, int obs_dim, int max_episode_steps,
    uint64_t seed, uint32_t step, uint32_t env_offset, float p_done, int reset, rl_stream_t stream);

/* CartPole physics (gym classic-control constants, Euler, float32), auto-reset
 * with U(-0.05,0.05)^4.  state [B,4] in/out, obs_out [B,4], actions [B] int32. */
int rl_env_cartpole_step(
    float* state, float* obs_out, float* reward_out, uint8_t* done_out, const int32_t* actions,
    float* ep_ret, int32_t* ep_len, float* totals,
    float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap,
    int B, int max_episode_steps, uint64_t seed, uint32_t step, uint32_t env_offset, int reset,
    rl_stream_t stream);

/* VecNormalizeEnv on the device (f2; parl/env/mujoco_wrappers.py:95-168 as benchmark/torch/ppo/env_utils.py uses it:
 * one wrapper — one set of running statistics — PER ENV, fed one sample per step, float64).  State arrays (caller
 * owned, initialise mean 0 / var 1 / count 1e-4 / ret 0): ob_mean, ob_var [B,D], ob_count, ret, ret_mean, ret_var,
 * ret_count [B].
 *   reward_step = 1: VecNormalizeEnv.step — ret = ret*gamma + reward; (term_obs != NULL and done: the finished
 *     episode's terminal observation updates the observation statistics first); reward <- clip(reward /
 *     sqrt(ret_var + eps), +-cliprew) IN PLACE; ret = 0 where done; then the observation handed on (obs_in; the reset
 *     observation where done) is filtered: statistics update (if `update`) and clip((x-mean)/sqrt(var+eps), +-clipob).
 *   reward_step = 0: VecNormalizeEnv.reset — only the observation filter.
 * obs_out may alias obs_in. */
int rl_vecnormalize_step(const float* obs_in, const float* term_obs, float* obs_out, float* reward,
                         const uint8_t* done, double* ob_mean, double* ob_var, double* ob_count, double* ret,
                         double* ret_mean, double* ret_var, double* ret_count, int B, int D, int update,
                         int norm_ob, int norm_ret, int reward_step, double clipob, double cliprew,
                         double gamma, double eps, rl_stream_t stream);

/* Standalone samplers.  logp_out may be NULL. */
int rl_sample_categorical(
    const float* logits, int N, int A, uint64_t seed, uint32_t step, uint32_t env_offset,
    int32_t* actions, float* logp_out, rl_stream_t stream);
int rl_sample_gaussian(
    const float* mean, const float* logstd, int N, int D, uint64_t seed, uint32_t step, uint32_t env_offset,
    float* action, float* logp_out, rl_stream_t stream);

/* Scratch for the flat (scan-free) loss kernels below: n_rows elements, `extra`
 * additional per-CTA partial columns (PPO-Gaussian: D).  Zeroed once by the caller. */
size_t rl_flat_workspace_bytes(long long n_rows, int extra);

/* ------------------------------------------------------------------------
 * a4  A2C loss + gradient.  Replaces parl/algorithms/torch/a2c.py:40-60
 * (post-network part of A2C.learn; SUM reductions).
 *   logits [N,A] f32, values [N], actions [N] i32/i64, advantages [N], target_values [N]
 *   losses [4] = {total, pi_loss, vf_loss, entropy};  d_logits [N,A], d_values [N]
 * ---------------------------------------------------------------------- */
int rl_a2c_loss_fwd_bwd(
    const float* logits, const float* values, const void* actions, int actions_i64,
    const float* advantages, const float* target_values, long long N, int A,
    float vf_loss_coeff, float entropy_coeff,
    float* losses, float* d_logits, float* d_values,
    void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* a5  Segment GAE of the A2C actor on a (T,B) rollout, float64 arithmetic.
 * Replaces parl/utils/rl_utils.py:34-51 (calc_gae via scipy.signal.lfilter) as driven by
 * benchmark/torch/a2c/actor.py:82-102: a segment ends at dones[t]==1 (next value 0) or at
 * the rollout end (next value = bootstrap_value[b] = V(next_obs)).  Time-major [T,B]. */
int rl_gae_scan_segments(
    const float* rewards, const float* values, const uint8_t* dones, const float* bootstrap_value,
    int T, int B, double gamma, double lam, float* advantages, float* target_values, rl_stream_t stream);

/* a6  PPO GAE.  Replaces benchmark/torch/ppo/storage.py:45-64
 * (RolloutStorage.compute_returns; float32, bit-exact operation order).  dones[t] is the
 * done flag observed BEFORE step t (float32 0/1); last_value/last_done [B]. */
int rl_gae_scan(
    const float* rewards, const float* values, const float* dones,
    const float* last_value, const float* last_done, int T, int B,
    float gamma, float gae_lambda, float* advantages, float* returns, rl_stream_t stream);

/* a7  PPO clipped-surrogate loss + gradient.  Replaces parl/algorithms/torch/ppo.py:102-138.
 * Pass exactly one of `logits` [N,A] (Categorical, actions i32/i64) or `mean` [N,D] with
 * `logstd` [D] (Normal(mean, exp(logstd)), actions = float32 [N,D]).
 *   adv_stats : device {mean, 1/(unbiased std + 1e-8)} from rl_adv_stats (norm_adv=True),
 *               or NULL (norm_adv=False).  Multi-GPU callers all-reduce the moments instead.
 *   losses [4] = {value_loss, action_loss, entropy_loss, total}  (MEAN reductions)
 *   d_logits_or_mean [N,A|D], d_logstd [D] (Gaussian only), d_values [N] */
int rl_adv_stats(const float* adv, long long N, float* stats, rl_stream_t stream);
int rl_ppo_loss_fwd_bwd(
    const float* logits, const float* mean, const float* logstd, const void* actions, int actions_i64,
    const float* values, const float* batch_value, const float* batch_return,
    const float* batch_logprob, const float* batch_adv, const float* adv_stats,
    long long N, int A_or_D, float clip_param, float value_loss_coef, float entropy_coef,
    int use_clipped_value_loss,
    float* losses, float* d_logits_or_mean, float* d_logstd, float* d_values,
    void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* a8  TD target + (weighted) MSE loss + gradient.  Replaces parl/algorithms/torch/dqn.py:64-69;
 * with q_online_next != NULL parl/algorithms/torch/ddqn.py:64-72; with weights != NULL the
 * PER variant benchmark/fluid/Prioritized_DQN/per_alg.py:48-69 (td_abs = |target - Q(s,a)|).
 *   q, q_target_next, q_online_next [M,A]; action [M]; reward, terminal (f32 0/1) [M]
 *   losses [1] = mean loss; d_q [M,A]; td_abs [M] or NULL */
int rl_td_loss_fwd_bwd(
    const float* q, const float* q_target_next, const float* q_online_next,
    const void* action, int action_i64, const float* reward, const float* terminal, const float* weights,
    long long M, int A, float gamma, float* losses, float* d_q, float* td_abs,
    void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* f4  Continuous-control critic TD (DDPG / TD3 / SAC).  Replaces parl/algorithms/torch/ddpg.py:63-73,
 * td3.py:78-94, sac.py:90-99:
 *   target = reward + (1 - terminal) * gamma * (min(Q1', Q2') - alpha * log pi(a'|s'))
 *   loss   = mse(Q1, target) + mse(Q2, target)          (means over the N samples)
 * q2 / d_q2 NULL: single critic (DDPG); q2_target_next NULL: no min; next_log_prob NULL: no entropy term.
 *   all arrays [N] f32, terminal 0/1; losses [3] = total, mse1, mse2; d_q = 2 (Q - target) / N; target_out [N] or NULL */
int rl_twin_q_td_loss_fwd_bwd(
    const float* q1, const float* q2, const float* q1_target_next, const float* q2_target_next,
    const float* next_log_prob, const float* reward, const float* terminal, long long N, float gamma, float alpha,
    float* losses, float* d_q1, float* d_q2, float* target_out,
    void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* REINFORCE on probabilities.  Replaces parl/algorithms/torch/policy_gradient.py:54-75. */
int rl_pg_loss_fwd_bwd(
    const float* prob, const void* action, int action_i64, const float* reward, long long N, int A,
    float* losses, float* d_prob, void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a9  HBM-resident replay.  Replaces benchmark/fluid/Prioritized_DQN/proportional_per.py:18-157
 * (SumTree + ProportionalPER), benchmark/torch/dqn/replay_memory.py:59-113 (frame-context
 * sampling) and parl/utils/replay_memory.py:51-95 (gather by index).
 *   tree  : double[2*capacity-1], reference heap indexing (leaf i at capacity-1+i), zero-initialised
 *   state : double[2] = {_min (init 10.0), _max_priority (init 1.0)}
 * ---------------------------------------------------------------------- */
int rl_per_store(double* tree, double* state, int capacity, int write_pos, int n, const float* delta,
                 double alpha, double eps, rl_stream_t stream);
int rl_per_update(double* tree, double* state, int capacity, const int32_t* tree_idx, const float* priorities,
                  int n, double alpha, double eps, rl_stream_t stream);
/* Stratified sample of seg_num leaves.  u [seg_num] float32 in [0,1) or NULL (Philox(seed, draw)).
 * weights = (size*p/total / (size*_min/total))^-beta. */
int rl_per_sample(const double* tree, const double* state, int capacity, int seg_num, const float* u,
                  uint64_t seed, uint32_t draw, double beta, double size,
                  int32_t* tree_idx, int32_t* elem_idx, float* weights, rl_stream_t stream);
/* Frame-ring gather (benchmark/torch/dqn/replay_memory.py:59-85): for every start index the n_out (<= ctx+1) frames
 * start .. start+n_out-1 (positions modulo curr_size), frames at or before the last episode end among the first
 * ctx-1 positions zeroed.  `lanes` interleaved transition streams (one per lock-stepped env): position q of lane l
 * is row q*lanes + l and a start index encodes (q0, l) as q0*lanes + l; lanes = 1 is the reference's single ring.
 * n_out = ctx+1: the learner's (obs, next_obs) window; n_out = ctx: the actor's current stacked observation. */
int rl_replay_gather_frames(const uint8_t* frames, const uint8_t* is_over, const int32_t* idx, int n,
                            int curr_size, int context_len, int HW, int lanes, int n_out, uint8_t* out,
                            rl_stream_t stream);
int rl_gather_rows(const void* src, const int32_t* idx, long long n, int row_bytes, void* out, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * Learner update on a flat parameter buffer (global-norm clip + Adam), no host sync.
 * Replaces the optimizer calls of the reference learners:
 *   parl/algorithms/paddle/impala/impala.py:113-117,210-213 (ClipGradByGlobalNorm(40) + Adam),
 *   parl/algorithms/torch/a2c.py:65-69 / ppo.py:144-147 (clip_grad_norm_ + Adam), dqn.py:68-71.
 * rl_grad_global_norm: out_norm[0] = ||grad||_2 (deterministic).  workspace >= 256+4*1184 B, zeroed once.
 * rl_adam_step: grad is first divided by grad_div (e.g. world size for MEAN losses), then scaled by
 *   clip_mode 0: 1 ; 1 (torch): min(1, max_norm/(norm+1e-6)) ; 2 (paddle): max_norm/max(norm, max_norm)
 *   where norm = grad_norm[0]/grad_div; lr from lr_device[0] if non-NULL else `lr`;
 *   step = 1-based update count (bias correction), read from step_device[0] instead when that is non-NULL (an
 *   int32 on the device: lets a captured CUDA graph of the update be replayed); zero_grad=1 clears grad in the same pass.
 * ---------------------------------------------------------------------- */
int rl_grad_global_norm(const float* grad, long long n, float* out_norm, void* workspace, size_t workspace_bytes,
                        rl_stream_t stream);
int rl_adam_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                 const float* lr_device, float lr, float beta1, float beta2, float eps, int step,
                 float grad_div, const float* grad_norm, float max_norm, int clip_mode, int zero_grad,
                 const int32_t* step_device, rl_stream_t stream);

/* out[i] = cast(src[idx[i]]) (idx < 0 -> 0): rebuilds every bf16 (out_bf16 = 1) or float32 (0) operand copy of the
 * network kernels from the flat float32 master buffer in one launch; idx is the index permutation of the copies,
 * built once by the host (parl_b200.kernels.PackPlan).  idx and out 16-byte aligned. */
int rl_gather_cast(const float* src, const int32_t* idx, long long n, void* out, int out_bf16, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a13 / K6  Dense contraction on the tcgen05 tensor cores (TMA-staged tiles, fp32 accumulation in TMEM):
 *   C[M,N] = act(A[M,K] . B[N,K]^T + bias[N])      A, B bf16 row-major ("x . W^T"), C bf16 or f32.
 * Replaces the nn.Linear forward of the reference models (e.g. benchmark/torch/a2c/atari_model.py:46-49,
 * executed there by cuBLAS through torch).  lda/ldb/ldc in elements; lda, ldb multiples of 8.
 * ---------------------------------------------------------------------- */
int rl_gemm_bf16_tn(const void* A, const void* B, const float* bias, void* C, int M, int N, int K,
                    int lda, int ldb, int ldc, int relu, int out_f32, rl_stream_t stream);
/* 1 (default): outputs of at least 2 x 2 tiles of width >= 128 run as 2 x 2 thread-block clusters whose CTAs multicast
 * their operand half-tiles to each other (each operand byte leaves L2 once per cluster); 0: single-CTA form only. */
int rl_debug_set_gemm_cluster(int enable);
/* Hidden layer + small heads in one call (the actor's fc 5184->512 followed by the policy head,
 * benchmark/torch/a2c/atari_model.py:46-49,60-66): H = act(A.B^T + bias) [M,N] bf16 as rl_gemm_bf16_tn(_splitk), then
 * out2 = bf16(H).W2^T + b2 for N2 <= 32 head rows (W2 [N2,N] bf16, out2 [M,ldo2] float32, fp32 accumulation in a fixed
 * order).  The heads kernel follows the GEMM (and its split-K reduce): mma.sync.m16n8k16 tiles of 16 rows, four warps
 * each reducing a quarter of N, for N2 <= 24; otherwise a warp-per-row kernel.  N % 128 == 0, N <= 1024, N2*N*2 <= 48 KB.  workspace as rl_gemm_bf16_tn_splitk (may be NULL). */
int rl_gemm_bf16_tn_heads(const void* A, const void* B, const float* bias, void* H, int M, int N, int K, int lda, int ldb,
                          int ldh, int relu, const void* W2, const float* b2, int N2, float* out2, int ldo2,
                          void* workspace, size_t workspace_bytes, rl_stream_t stream);
/* 1 (default): the heads of rl_gemm_bf16_tn_heads run as a warp-level mma.sync kernel after H is complete; 0: the
 * warp-per-row CUDA-core kernel (fused with the split-K reduce where that applies). */
int rl_debug_set_heads_mma(int enable);
/* rl_gemm_bf16_tn with an optional split-K workspace — the actor-side nn.Linear (atari_model.py:46-49 evaluated on
 *  the 5-env batch of examples/IMPALA/actor.py:60-62; here 512..4096 envs per GPU).  Workspace (>= splits * ceil(M/128)*128 * ceil(N/BN)*BN * 4 bytes; 8 MB
 * covers every shape that splits): when the output has fewer tiles than half the SMs and K >= 1024, the reduction is
 * split over up to 8 CTAs per tile (fp32 partials, fixed-order second pass with the bias/ReLU epilogue).  Same
 * result contract as rl_gemm_bf16_tn; workspace NULL = never split. */
int rl_gemm_bf16_tn_splitk(const void* A, const void* B, const float* bias, void* C, int M, int N, int K,
                           int lda, int ldb, int ldc, int relu, int out_f32, void* workspace, size_t workspace_bytes,
                           rl_stream_t stream);
/* Backward-through-ReLU form: C[M,N] = (A . B^T) * (mask > 0), mask [M, ldm] bf16 = the saved post-ReLU activation
 * of the layer whose input gradient is being formed (dX = dY . W, B = W^T stored [N, K]). */
int rl_gemm_bf16_tn_masked(const void* A, const void* B, void* C, const void* mask, int M, int N, int K,
                           int lda, int ldb, int ldc, int ldm, int out_f32, rl_stream_t stream);

/* NHWC bf16 convolution forward (+bias, optional ReLU) as an implicit GEMM on tcgen05: the conv layers of
 * the Atari actor-critic (benchmark/torch/a2c/atari_model.py:26-44; executed there by cuDNN through torch).
 *   in [N,Hin,Win,Cin] bf16, weight_krsc [Cout, KH*KW*Cin] bf16 with K ordered (r, s, c), bias [Cout] f32,
 *   out [N,Hout,Wout,Cout] bf16.  Cin, Cout in {32, 64}; KH*KW*Cin a multiple of 64. */
int rl_conv2d_nhwc_bf16_fwd(const void* in, const void* weight_krsc, const float* bias, void* out,
                            int N, int Hin, int Win, int Cin, int Cout, int KH, int KW, int stride, int pad,
                            int relu, rl_stream_t stream);

/* Stride-1 NHWC bf16 convolution forward in TMA-window form (no operand gather): a conv over the flattened
 * pixel sequence is a sum of shifted GEMMs; one TMA load per 128-position tile brings the input window into
 * shared memory and every filter tap is a tcgen05.mma whose descriptor starts (r*W+s) rows further down.
 * Stride-2/4 layers use it through space-to-depth of their input.  in [N,H,W,Cin], weight [Cout, KH*KW*Cin]
 * ordered (r,s,c); out_mode 0: out [N,H-KH+1,W-KW+1,Cout]; out_mode 1 (20x20 outputs only): out is the
 * zero-padded 2x2 space-to-depth tensor [N,12,12,4*Cout] that feeds a following 4x4/stride-2/pad-2 conv.
 * Cin in {64,128}, Cout in {32,64}, 128+(KH-1)*W+(KW-1) <= 256. */
int rl_conv2d_s1_nhwc_bf16_fwd(const void* in, const void* weight_krsc, const float* bias, void* out,
                               int N, int H, int W, int Cin, int Cout, int KH, int KW, int relu, int out_mode,
                               rl_stream_t stream);
int rl_debug_set_shiftconv_base_offset(int enable);
/* 0 (default): one MMA group per filter tap; 1: column-tap-fused tile (the KW taps of a filter row share one
 * A-operand read, N' = KW*Cout accumulator columns, shifted sum in the epilogue) — measured slower on B200, kept as
 * an experiment and cross-check. */
int rl_debug_set_shiftconv_form(int form);
/* The same forward for conv1 of the Atari models on the uint8 observation: in_u8 [N,H,W,64] uint8 (space-to-depth,
 * rl_obs_stack_gather out_dtype 4); operand = bf16(byte * in_scale), converted in shared memory by four extra warps,
 * bit-identical to feeding rl_conv2d_s1_nhwc_bf16_fwd the out_dtype-3 tensor at half the input traffic.
 * Built for KH = KW = 2, Cin = 64, Cout = 32. */
int rl_conv2d_s1_u8in_bf16_fwd(const void* in_u8, float in_scale, const void* weight_krsc, const float* bias, void* out,
                               int N, int H, int W, int Cout, int KH, int KW, int relu, int out_mode,
                               rl_stream_t stream);

/* Data gradient of rl_conv2d_s1_nhwc_bf16_fwd in the same TMA-window form (transposed conv = shifted GEMMs run
 * backwards).  dout_grid [N,H,W,Cout] is the output gradient ON THE INPUT GRID (zeros where y>=H-KH+1 or
 * x>=W-KW+1); weight_t_krsc [Cin, KH*KW*Cout] with element [ci][(r,s,co)] = W[co][(r,s,ci)];
 * act_mask (optional) [N,H,W,Cin] is the saved post-ReLU input activation: din *= (act_mask > 0).
 * out_mode 0: din on a [N,OGH,OGW,Cin] grid (OGH>=H, OGW>=W; untouched cells stay as they are);
 * out_mode 2 (H=W=12, Cin=128): din of the 2x2-block conv scattered to conv1's gradient grid [N,21,21,32]. */
int rl_conv2d_s1_nhwc_bf16_dgrad(const void* dout_grid, const void* weight_t_krsc, const void* act_mask, void* din,
                                 int N, int H, int W, int Cout, int Cin, int KH, int KW, int out_mode,
                                 int OGH, int OGW, rl_stream_t stream);

/* Weight gradient of rl_conv2d_s1_nhwc_bf16_fwd in TMA-window form: dW[co][(r,s,ci)] = sum_q dout_grid[q,co] *
 * in[q + r*W + s, ci] with the position index as the GEMM reduction dimension (tcgen05, MN-major operands,
 * accumulators resident in TMEM over the CTA's whole position range, deterministic two-stage reduction).
 * dout_grid [N,H,W,Cout] on the input grid (zeros at invalid positions), in [N,H,W,Cin], dw_krsc [Cout, KH*KW*Cin]
 * float32 (accumulate=1 adds to it).  (Cout, Cin) = (64, 64|128), or (32, 64) where the 64-byte dout rows are the
 * SWIZZLE_64B N-operand of a role-swapped product.  db (optional, [Cout] float32) receives the bias gradient
 * sum_q dout_grid[q, :] from the same pass (one extra tcgen05.mma per K step against a tile of ones).
 * Workspace: rl_conv_wgrad_workspace_bytes. */
size_t rl_conv_wgrad_workspace_bytes(int KH, int KW, int Cin);
int rl_conv2d_s1_nhwc_bf16_wgrad(const void* dout_grid, const void* in, float* dw_krsc, float* db, int N, int H, int W,
                                 int Cin, int Cout, int KH, int KW, int accumulate,
                                 void* workspace, size_t workspace_bytes, rl_stream_t stream);
/* Weight (+ bias) gradient of rl_conv2d_s1_u8in_bf16_fwd: `in_u8` [N,H,W,64] uint8, same workspace rule (Cin = 64). */
int rl_conv2d_s1_u8in_bf16_wgrad(const void* dout_grid, const void* in_u8, float in_scale, float* dw_krsc, float* db,
                                 int N, int H, int W, int Cout, int KH, int KW, int accumulate,
                                 void* workspace, size_t workspace_bytes, rl_stream_t stream);
int rl_debug_set_wgrad_lane_map(int mode);
/* out[c] = sum_r x[r,c] for a [rows, C] bf16 matrix (bias gradients); C a multiple of 8 with C/8 dividing 256;
 * workspace >= 1184*C*4 bytes. */
int rl_colsum_bf16(const void* x, long long rows, int C, float* out, void* workspace, size_t workspace_bytes,
                   rl_stream_t stream);

/* Bandwidth-bound glue of the learner network (bf16, in HBM):
 *   rl_bias_act_bf16          x[M,N] = act(x + bias[N]) in place (epilogue of a library GEMM);
 *   rl_mask_scatter_grid_bf16 ReLU backward + re-gridding: dst[n,y,x,:] = src[n,y,x,:] * (act[n,y,x,:] > 0) from a
 *                             compact [N,PH,PW,C] gradient onto a [N,GH,GW,C] grid (other cells untouched). */
int rl_bias_act_bf16(void* x, const float* bias, long long M, int N, int relu, rl_stream_t stream);
int rl_mask_scatter_grid_bf16(const void* src, const void* act, void* dst, long long N, int PH, int PW, int GH, int GW,
                              int C, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a13  K6 for the MLP model family: whole-network forward / backward in ONE launch, fp32 on the CUDA cores.
 * Replaces the torch/paddle eager execution of benchmark/torch/ppo/mujoco_model.py:27-53 (17-64-64 tanh ->
 * {mean 6, value 1}), benchmark/torch/QuickStart/cartpole_model.py:21-38 (4-20 tanh -> 2),
 * examples/DQN/cartpole_model.py:21-41 (4-128-128 relu -> 2).
 *   n_layers (1..4) linear layers; dims[n_layers+1] = {in, h1, ..., out} (each 1..128); hidden layers use
 *   `act` (0 relu, 1 tanh, 2 none), the last layer is linear.  Parameters are handed over as n_seg row
 *   SEGMENTS in torch nn.Linear layout: segment s holds rows [.., +seg_rows[s]) of layer seg_layer[s]
 *   (segments of one layer are stacked in the order given — e.g. the policy and value heads of an
 *   actor-critic are two segments of the last layer), seg_w[s] [rows, in] float32, seg_b[s] [rows] or NULL.
 *   dims, seg_layer, seg_rows, seg_w, seg_b, seg_dw, seg_db are HOST arrays (of device pointers where typed so).
 * rl_mlp_fwd: x [n, in] -> out [n, out]; with out2 != NULL the output columns are delivered as two dense
 *   tensors, out [n, split] and out2 [n, out-split] (policy head / value head).  rl_mlp_bwd takes d_out /
 *   d_out2 the same way.
 * rl_mlp_bwd: recomputes the hidden activations from x, back-propagates d_out [n, out] and writes
 *   (accumulate=0) or adds (1) the parameter gradients into seg_dw[s] / seg_db[s] (same shapes as the
 *   parameters); deterministic two-stage reduction through `workspace` (rl_mlp_workspace_bytes). */
size_t rl_mlp_workspace_bytes(int n_layers, const int* dims);
int rl_mlp_fwd(const float* x, int n, int n_layers, const int* dims, int n_seg, const int* seg_layer,
               const int* seg_rows, const float* const* seg_w, const float* const* seg_b, int act, float* out,
               float* out2, int split, rl_stream_t stream);
int rl_mlp_bwd(const float* x, int n, int n_layers, const int* dims, int n_seg, const int* seg_layer,
               const int* seg_rows, const float* const* seg_w, const float* const* seg_b, int act,
               const float* d_out, const float* d_out2, int split, float* const* seg_dw, float* const* seg_db,
               int accumulate, void* workspace, size_t workspace_bytes, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * a10 + a11 + a13  Fused on-device actor pool for MLP policies: ONE launch runs T lock-step steps of all B envs
 * — policy/value forward (network as in rl_mlp_fwd; outputs = [action_dim policy outputs | value if has_value]),
 * action sampling (policy_kind 0: categorical, exact inverse CDF; 1: diagonal Gaussian with logstd [action_dim]),
 * env step (env_kind 0: MuJoCo-shaped synthetic env of rl_env_mujoco_synth_step; 1: CartPole physics of
 * rl_env_cartpole_step), auto-reset, episode bookkeeping — and writes the trajectory time-major.
 * Replaces per step: agent.sample -> envs.step -> rollout.append (benchmark/torch/ppo/train.py:91-101,
 * benchmark/torch/a2c/actor.py:56-80) and its RPC.  Bit-identical to stepping the stand-alone kernels.
 *   obs_cur [B, obs_dim] in/out: the observation every env is in (initialise with the env's reset kernel);
 *   global step index of row t = step0 + t (RNG counter);
 *   outputs: obs_out [T,B,obs_dim], act_out [T,B] int32 | [T,B,action_dim] f32, logp_out [T,B] (opt),
 *   val_out [T+1,B] (opt; row T = value of the observation after the last step), logits_out [T,B,action_dim]
 *   (opt, categorical), rew_out [T,B] f32, done_out [T,B] u8.
 *   vecnorm_state (optional; host array of the 7 device state arrays of rl_vecnormalize_step in its order
 *   {ob_mean, ob_var, ob_count, ret, ret_mean, ret_var, ret_count}), vecnorm_cfg host {clipob, cliprew, gamma, eps},
 *   vecnorm_flags bit0 update | bit1 normalise observations | bit2 normalise rewards: a VecNormalizeEnv per env
 *   between the env and the policy (obs_cur / obs_out / rew_out then hold NORMALISED values; episode statistics
 *   keep raw rewards, as MonitorEnv sits below VecNormalizeEnv in wrap_rms). */
int rl_rollout_mlp(int n_layers, const int* dims, int n_seg, const int* seg_layer, const int* seg_rows,
                   const float* const* seg_w, const float* const* seg_b, int act, int env_kind, int policy_kind,
                   int T, int B, int action_dim, int has_value, const float* logstd, float* obs_cur,
                   float* ep_ret, int32_t* ep_len, float* totals, float* ring_ret, int32_t* ring_len,
                   uint32_t* ring_head, int ring_cap, uint64_t seed, uint32_t step0, uint32_t env_offset,
                   float p_done, int max_episode_steps, float* obs_out, void* act_out, float* logp_out,
                   float* val_out, float* logits_out, float* rew_out, uint8_t* done_out,
                   double* const* vecnorm_state, const double* vecnorm_cfg, int vecnorm_flags, rl_stream_t stream);

/* ------------------------------------------------------------------------
 * Off-policy continuous control (DDPG / TD3 / SAC).  Replaces the per-step loop of
 * benchmark/torch/{td3,sac,ddpg}/train.py: agent.sample -> env.step -> rpm.append -> rpm.sample_batch.
 *
 * rl_explore_mlp: ONE launch runs K lock-step steps of B MuJoCo-shaped synthetic envs (the env of
 *   rl_env_mujoco_synth_step): actor forward, exploration rule, env step, episode bookkeeping, and writes every
 *   transition straight into the rows of a replay ring of rm_max_size rows:
 *     rm_obs / rm_next_obs [cap, obs_dim] f32, rm_action [cap, action_dim] f32, rm_reward [cap] f32,
 *     rm_terminal [cap] i32.  Step t of env b goes to row (rm_pos + t*B + b) % rm_max_size (the order of K
 *     successive batch appends); K*B > rm_max_size is rejected (a launch would overwrite its own rows).
 *   Actor: n_layers-1 (1..3) ReLU hidden layers and a head, fp32 parameters read in place (row segments as in
 *     rl_mlp_fwd; widths <= 512); head 0: tanh(out) [action_dim] (TD3 / DDPG), head 1: out = [mean | log_std]
 *     [2*action_dim], log_std clamped to [-20, 2] (SAC).  The actor is not evaluated in mode 0.
 *   mode 0 (warm-up): a = 2u - 1, u = 24-bit uniform word (d % 4) of philox(env, step, d / 4, STREAM_ACTION);
 *   mode 1 (deterministic + noise, head 0): a = clip(tanh(out) + expl_noise * z, -1, 1), z Gaussian on STREAM_GAUSS
 *     (expl_noise = 0 is the deterministic policy);
 *   mode 2 (SAC, head 1): a = tanh(mean + exp(log_std) * z).
 *   Env: reward / done from STREAM_REWDONE at (env, step), next observation at step + 1 on STREAM_OBS; done also at
 *     the time limit (max_episode_steps > 0); terminal = done and not the time-limit step.  The env auto-resets: the
 *     next_obs of a done step is the first observation of the next episode (terminal rows mask it by 1 - terminal).
 *   obs_cur [B, obs_dim] in/out carries the observations between launches; step index of row t = step0 + t.
 *   The rows of every layer are split over a thread-block cluster of up to 8 CTAs that keeps the actor resident in
 *   shared memory for all K steps; an actor that does not fit 8 CTAs is rejected.
 *
 * rl_replay_sample_uniform: n rows drawn uniformly from the first min(*size_dev, capacity) rows of a ring of
 *   `capacity` rows, gathered densely:
 *   obs_out / next_obs_out [n, obs_dim], action_out [n, act_dim], reward_out / terminal_out [n] (f32), idx_out [n]
 *   (optional).  Row i of draw d = *draw_dev is (x * size) >> 32, x = word 0 of philox(i, d, 0, STREAM_REPLAY).
 *   size and draw are read from device memory, so a captured graph draws fresh rows on every replay. */
int rl_explore_mlp(int n_layers, const int* dims, int n_seg, const int* seg_layer, const int* seg_rows,
                   const float* const* seg_w, const float* const* seg_b, int head, int mode, int K, int B,
                   int action_dim, float expl_noise, float* obs_cur, float* ep_ret, int32_t* ep_len, float* totals,
                   float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap, uint64_t seed,
                   uint32_t step0, uint32_t env_offset, float p_done, int max_episode_steps, float* rm_obs,
                   float* rm_action, float* rm_reward, int32_t* rm_terminal, float* rm_next_obs, int rm_max_size,
                   int rm_pos, rl_stream_t stream);
int rl_replay_sample_uniform(const float* obs, const float* action, const float* reward, const int32_t* terminal,
                             const float* next_obs, int obs_dim, int act_dim, const int32_t* size_dev,
                             const int32_t* draw_dev, int capacity, int n, uint64_t seed, float* obs_out, float* action_out,
                             float* reward_out, float* terminal_out, float* next_obs_out, int32_t* idx_out,
                             rl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PARL_B200_H_ */
