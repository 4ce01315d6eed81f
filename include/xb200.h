/*
 * xb200.h - C-ABI of the B200-native rollout->update hot path for agi-brain/xuance (v1.4.4 @ 4f0b05b).
 *
 * The reference has NO native/FFI layer (SURVEY.md section 8b): its hot path is Python classes resolved
 * through registries.  This header is therefore the boundary a maintainer would bind from those classes
 * (ctypes stubs in INTEGRATION.md); every entry point cites the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream, allocates
 *     nothing, and returns 0 on success, a negative XB_E* code for a rejected argument, or a positive
 *     cudaError_t if the launch failed
 *   - row-major layouts; [N,T,...] buffers are the reference's `create_memory` layout
 *     (xuance/common/memory_tools.py:12-40) so that flat slot = env*T + step = the index handed to sample()
 *   - scalar fields (actions of a Discrete space, rewards, values, terminals, old_logp, returns, advantages)
 *     are float32, exactly as the reference stores them (memory_tools.py:15; SURVEY appendix B #1)
 */
#ifndef XB200_H_
#define XB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XB_OK 0
#define XB_EINVAL (-1)   /* bad size / null pointer */
#define XB_EALIGN (-2)   /* pointer or row size not aligned as the entry point requires */
#define XB_ERANGE (-3)   /* argument outside the supported range (documented per call) */

/* observation output formats of xb_gather_obs */
#define XB_OBS_U8 0        /* byte copy (bit-exact gather)                                          */
#define XB_OBS_F32_NHWC 1  /* float32 = u8/255.0 (correctly rounded division), same element order   */
#define XB_OBS_F32_NCHW 2  /* float32 = u8/255.0, channel planes (HWC -> CHW per row)               */
#define XB_OBS_BF16_NHWC 3 /* bfloat16(round-to-nearest-even of u8/255.0f), same element order      */
#define XB_OBS_F16_NHWC 4  /* float16 (rn) of u8/255.0f, same element order                         */

int xb_version(void);
const char *xb_error_string(int code);
/* sm_count, compute capability of the current device; returns cudaError on failure */
int xb_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* ---------------------------------------------------------------- K1: rollout / replay store ---------
 * Replaces store_element(): `memory[:, ptr] = data`  (memory_tools.py:43-61), as used by
 * DummyOnPolicyBuffer.store :232-240, DummyOffPolicyBuffer.store :364-372, PerOffPolicyBuffer.store :537-543.
 * rows:    dst[N, T, row_bytes] (bytes)  <- src[N, row_bytes]   at step t      (row_bytes % 4 == 0)
 * scalars: dst[F, N, T] (float32)        <- src[F, N]           at step t      (F may be 0)
 * One launch does both; pass rows_dst = NULL to store scalars only. */
int xb_rollout_store(void *rows_dst, const void *rows_src, int64_t row_bytes,
                     float *scal_dst, const float *scal_src, int F,
                     int N, int T, int t, void *stream);

/* ---------------------------------------------------------------- K2: GAE / returns scan -------------
 * Replaces DummyOnPolicyBuffer.finish_path (memory_tools.py:242-265) for ALL envs and ALL path segments of a
 * rollout in one launch.  rew/val/term/adv/ret are [N,T] float32.  seg_end[N,T] (uint8) marks the last step
 * of each finished path, bootstrap[N,T] holds the `val` passed to finish_path at that step, covered[N] is the
 * number of leading steps of env i that belong to finished paths (steps >= covered[i] get adv = ret = 0, as in
 * the reference where they are never written).
 *   use_gae=1:  delta_t = r_t + (1-d_t)*gamma*V_{t+1} - V_t ;  A_t = delta_t + (1-d_t)*gamma*lam*A_{t+1}
 *               ret_t = A_t + V_t   (float32; warp-level scan of the affine maps, so +-few ulp of the loop)
 *   use_gae=0:  ret_t = r_t + gamma*ret_{t+1} (float64 scan, as scipy.lfilter), A_t = r_t + gamma*V_{t+1} - V_t */
int xb_gae_scan(const float *rew, const float *val, const float *term,
                const uint8_t *seg_end, const float *bootstrap, const int32_t *covered,
                float *adv, float *ret, int N, int T, float gamma, float lam, int use_gae, void *stream);

/* ---------------------------------------------------------------- K3: minibatch gather ---------------
 * Replaces sample_batch(): `memory[(env_idx, step_idx)]` (memory_tools.py:64-84) as used by
 * DummyOnPolicyBuffer.sample :267-287 and the replay buffers' sample().  idx[B] are flat slots (env*T+step);
 * idx == NULL means identity (rows 0..B-1), which turns xb_gather_obs into the u8 -> float preprocessing of
 * AC_CNN_Atari.forward / Basic_CNN.forward (xuance/torch/rl_models/representations/cnn.py:45-50,98-102).
 * xb_gather_rows: dst[B,row_bytes] <- src[idx[b]]            (row_bytes % 4 == 0; bulk-async path if % 16 == 0)
 * xb_gather_obs : dst[B, H*W*C] in `format` <- u8 src rows; H*W*C % 16 == 0; NCHW needs C == 4, W % 4 == 0. */
int xb_gather_rows(const void *src, const int64_t *idx, int64_t B, int64_t row_bytes, void *dst, void *stream);
int xb_gather_obs(const uint8_t *src, const int64_t *idx, int64_t B, int H, int W, int C,
                  void *dst, int format, void *stream);

/* Gathers F float32 fields fields[F, slots] at idx[B] into out[F, B]; if adv_field >= 0 that field is
 * replaced by (x - mean) / (std + 1e-8) with the POPULATION std over the B gathered values
 * (memory_tools.py:280-282).  stats_out[2] receives (mean, std).  scratch: >= xb_scratch_doubles() doubles
 * plus one trailing int32 counter, zeroed once by the caller (the kernels re-zero it).
 * world-size > 1 is handled above the ABI (all-reduce of the partial sums). */
int64_t xb_scratch_doubles(void);
int xb_gather_scalars(const float *fields, int64_t slots, const int64_t *idx, int64_t B, int F,
                      float *out, int adv_field, float *stats_out, double *scratch, void *stream);
/* adv[b] <- (adv[b] - stats[0]) / (stats[1] + 1e-8) with GIVEN statistics: the second half of memory_tools.py:281-282 for a
 * minibatch that is sharded over ranks (its global mean / population std are all-reduced once per epoch). */
int xb_adv_normalize(float *adv, int64_t B, const float *stats, void *stream);

/* ---------------------------------------------------------------- K4: fused PPO-Clip loss fwd+bwd ----
 * Replaces ppo_learner.py:46-60 plus the autograd backward of those lines down to (logits, value):
 *   logp = log_softmax(logits)[a]; ratio = exp(logp - old_logp)
 *   a_loss = -mean(min(clamp(ratio,1-eps,1+eps)*adv, adv*ratio)); c_loss = mean((v-ret)^2); e = mean(H)
 *   loss = a_loss - ent_coef*e + vf_coef*c_loss
 * Writes dlogits[B,A] = dloss/dlogits, dvalue[B] = dloss/dvalue (means over B_total >= B rows so a
 * rank-local shard of a global minibatch produces correctly scaled gradients) and
 * stats[8] = {a_loss, c_loss, entropy, mean(v), clip_fraction, loss, 0, 0} * (B/B_total weighting applied,
 * i.e. sums over the local rows divided by B_total).  actions are float32 (reference quirk).  A <= 64.
 * loss_kind 0 = PPO-Clip (above); 1 = plain policy gradient a_loss = -mean(adv*logp) (old_logp unused): A2C
 * (a2c_learner.py:46-52) with adv = advantages, PG (pg_learner.py:44-47) with adv = returns and vf_coef = 0. */
int xb_ppo_loss_fwd_bwd(const float *logits, const float *value, const float *actions,
                        const float *old_logp, const float *adv, const float *ret,
                        int64_t B, int A, int64_t B_total, float clip_range, float vf_coef, float ent_coef,
                        int loss_kind, float *dlogits, float *dvalue, float *stats, double *scratch, void *stream);

/* ---------------------------------------------------------------- K4-G: Gaussian-policy PPO loss ------
 * K4 for a diagonal Gaussian policy (GaussianActorHead + DiagGaussianDistribution, actor_head.py:45-72,
 * distributions.py:165-197): torch.distributions.Normal(mu, exp(log_std)) with log-prob and entropy summed over D,
 *   logp_b = sum_d [-(a-mu)^2/(2 sigma^2) - log sigma - log sqrt(2 pi)];  H = sum_d [1/2 + log sqrt(2 pi) + log sigma]
 * and the same surrogate, value loss, loss_kind, B_total scaling and stats[8] layout as xb_ppo_loss_fwd_bwd.
 * mu[B,D] is the head's output after activation_action, log_std[D] the head's parameter, actions[B,D] float32.
 * Writes dmu[B,D], dvalue[B] and dlog_std[D] = sum_b dloss/dlogp_b * ((a-mu)^2/sigma^2 - 1) - ent_coef*B/B_total,
 * a reduction over every row that is bit-identical from run to run (fixed-order double sums, no float atomics).
 * scratch: the K4 scratch (xb_scratch_doubles()); col_scratch: xb_gaussian_scratch_doubles(D) doubles for the
 * per-dimension block partials (need not be zeroed).  1 <= D <= 64 (XB_ERANGE above). */
int64_t xb_gaussian_scratch_doubles(int D);
int xb_ppo_gaussian_loss_fwd_bwd(const float *mu, const float *log_std, const float *value, const float *actions,
                                 const float *old_logp, const float *adv, const float *ret, int64_t B, int D,
                                 int64_t B_total, float clip_range, float vf_coef, float ent_coef, int loss_kind,
                                 float *dmu, float *dvalue, float *dlog_std, float *stats, double *scratch,
                                 double *col_scratch, void *stream);

/* ---------------------------------------------------------------- K5: prioritized-replay trees -------
 * Replaces SumSegmentTree/MinSegmentTree (xuance/common/segtree_tool.py:4-220) and their use in
 * PerOffPolicyBuffer (memory_tools.py:505-598).  One (sum,min) pair PER ENV, float32 nodes, heap layout
 * tree[env][2*cap] (node 1 = root, leaves at cap..2cap-1); parents are fl32(l+r) / min(l,r).
 * insert : leaf[ptr] = max_prio[env]^alpha in both trees for every env           (:545-548)
 * sample : per env, k stratified draws: p_total = sum(0,size-1) with the reference's association order,
 *          mass_j = fl(fl(u_j*seg) + fl(j*seg)), find_prefixsum_idx; weights = p_j/p_min computed as the
 *          reference does (:563-572); u[N,k] float32 uniforms supplied by the caller
 *          outputs: step_out[N,k] int64, flat_out[N*k] int64 (= env*S + step), w_out[N,k] float64
 * update : leaf = p^alpha (p==0 -> 1e-8), later duplicates win, parents recomputed, max_prio updated (:588-598) */
/* out[i] = x[i]^y evaluated exactly as glibc 2.39 powf does (the routine numpy's float32 ** python-float calls, i.e.
 * what memory_tools.py:547,596 evaluate); exported so the parity tests can check the restatement on its own. */
int xb_powf_libm(const float *x, float y, float *out, int64_t n, void *stream);
int xb_per_insert(float *sum_tree, float *min_tree, float *max_prio, int N, int cap, int ptr, float alpha,
                  void *stream);
int xb_per_sample(const float *sum_tree, const float *min_tree, const float *u, int N, int cap, int size,
                  int k, int64_t S, float size_pow_neg_beta,
                  int64_t *step_out, int64_t *flat_out, double *w_out, void *stream);
int xb_per_update(float *sum_tree, float *min_tree, float *max_prio, const int64_t *idx, const float *prio,
                  int N, int cap, int k, float alpha, void *stream);

/* ---------------------------------------------------------------- K6: DQN TD target + loss fwd+bwd ---
 * Replaces dqn_learner.py:41-46 / perdqn_learner.py:44-50: predictQ = Q[b, a_b]; y = r + gamma*(1-d)*max_a Q'
 * loss = mean((predictQ - y)^2); dq[B,A] = dloss/dQ; td[B] = y - predictQ; stats[4] = {loss, mean predictQ,0,0}
 * (sums over local rows / B_total).  q_sel != NULL selects double-Q (ddqn_learner.py:39-44): q_sel[B,A] are the EVAL
 * network's values at the next observation, y uses q_next[b, argmax_a q_sel[b,a]] instead of the max. */
int xb_dqn_td_fwd_bwd(const float *q_eval, const float *q_next, const float *q_sel, const float *actions, const float *rew,
                      const float *term, int64_t B, int A, int64_t B_total, float gamma,
                      float *dq, float *td, float *stats, double *scratch, void *stream);

/* ---------------------------------------------------------------- K9: QMIX selection / mixing / TD ----
 * Replaces, for one parameter-sharing group with use_rnn=True (episodes padded to T, `filled` mask):
 * select  : qmix_learner.py:42-66 + iql_learner.py:57-59 - gather Q(o_t, a_t) from the eval net outputs
 *           q_all[B,n,T+1,A], the double-Q / max next value from the target outputs q_tgt at step t+1, both
 *           multiplied by agent_mask*filled and written agent-minor [B*T, n] (the layout Q_tot concatenates,
 *           value_factorization.py:137-142); also filled_sum[0] = sum(filled).  actions/masks are float32.
 *           avail (nullable; use_actions_mask, iql_learner.py:60-81 + value_factorization.py:86-89): uint8
 *           [B,n,T+1,avail_ld], unavailable actions count as -1e10 in the double-Q arg-max over the eval values
 *           and in the target values of step t+1.
 *           select_bwd scatters d(q_eval_taken) back into a zeroed dq_all.
 * mix     : QMIX_Mixer.forward epilogue (q_mix_head.py:81-94) on precomputed hypernet outputs:
 *           hidden = elu(q . |w1_raw|[n,H] + b1) ; q_tot = hidden . |w2_raw| + b2   (n <= 16), and its backward
 *           (abs' = sign, elu' = exp) producing dq, dw1_raw, db1, dw2_raw (db2 = dq_tot).
 * td      : qmix_learner.py:34-35,76-84 masked TD loss; writes dq_tot and stats[2] = {loss_Q, mean(q_tot)}. */
int xb_qmix_select_fwd(const float *q_all, const float *q_tgt, const float *actions, const float *agent_mask,
                       const float *filled, const uint8_t *avail, int avail_ld, int B, int n, int T, int A,
                       int double_q, float *q_eval_taken, float *q_next_taken, float *filled_sum, double *scratch,
                       void *stream);
int xb_qmix_select_bwd(const float *d_taken, const float *actions, const float *agent_mask, const float *filled,
                       int B, int n, int T, int A, float *dq_all, void *stream);
int xb_qmix_mix_fwd(const float *q, const float *w1_raw, const float *b1, const float *w2_raw, const float *b2,
                    int64_t R, int n, int H, float *q_tot, void *stream);
int xb_qmix_mix_bwd(const float *dq_tot, const float *q, const float *w1_raw, const float *b1, const float *w2_raw,
                    int64_t R, int n, int H, float *dq, float *dw1_raw, float *db1, float *dw2_raw, void *stream);
int xb_qmix_td(const float *q_tot, const float *q_tot_next, const float *rewards, const float *terminals,
               const float *filled, const float *filled_sum, int B, int n, int T, float gamma, float grad_scale,
               float *dq_tot, float *stats, double *scratch, void *stream);

/* Tensor-core forward of the whole mixer (hypernet GEMMs + epilogue in ONE kernel; tcgen05.mma with TMEM
 * accumulators, bf16 hi/lo split operands, 3 MMAs per product, fp32 accumulate): q_tot[R] from states[R,S], q[R,n]
 * and the raw Linear parameters of QMIX_Mixer (q_mix_head.py:52-64): w_l1[4] / b_l1[4] are HOST arrays of 4 device
 * pointers to the first-layer weights [32,S] / biases [32] of hyper_w_1, hyper_b_1, hyper_w_2, hyper_b_2 (in that
 * order), wb1[n*32,32] = hyper_w_1[2], wb2[32,32] = hyper_w_2[2], wb2c[1,32] = hyper_b_2[2].  Requires dim_hidden =
 * dim_hypernet_hidden = 32, n <= 8 and the staged operands to fit 220 KB of shared memory (else XB_ERANGE and the
 * caller uses cuBLAS + xb_qmix_mix_fwd).  Forward only: used for the target mixer / inference. */
int xb_qmix_mix_fused_fwd(const float *states, const float *q, const float *const *w_l1_host,
                          const float *const *b_l1_host, const float *wb1, const float *bias_wb1, const float *wb2,
                          const float *bias_wb2, const float *wb2c, const float *bias_wb2c, int64_t R, int S, int n,
                          int H, int HH, float *q_tot, void *stream);

/* ---------------------------------------------------------------- K8: SAC loss stages ----------------
 * Replaces the elementwise/reduction parts of SAC_Learner.update (xuance/torch/learners/policy_gradient/
 * sac_learner.py:52-88).  `alpha` is a DEVICE scalar (exp(log_alpha)).
 * actor : p_loss = mean(alpha*log_pi - min(q1,q2)); writes dlog_pi, dq1, dq2 (torch.min ties split 1/2),
 *         stats[4] = {Ploss, mean(min q), mean(log_pi), 0}
 * critic: backup = r + (1-d)*gamma*(target_q - alpha*log_pi_next); q_loss = mse(q1,backup)+mse(q2,backup);
 *         writes dq1, dq2, backup; stats[2] = {Qloss, 0} */
int xb_sac_actor_loss(const float *log_pi, const float *q1, const float *q2, const float *alpha, int64_t B,
                      int64_t B_total, float *dlog_pi, float *dq1, float *dq2, float *stats, double *scratch,
                      void *stream);
int xb_sac_critic_loss(const float *q1, const float *q2, const float *target_q, const float *log_pi_next,
                       const float *rew, const float *term, const float *alpha, float gamma, int64_t B,
                       int64_t B_total, float *dq1, float *dq2, float *backup, float *stats, double *scratch,
                       void *stream);

/* ---------------------------------------------------------------- K7: flat-bucket optimiser step -----
 * Replaces clip_grad_norm_ + torch.optim.Adam.step on the learner's parameters (ppo_learner.py:61-65;
 * Adam eps=1e-5, no weight decay, no amsgrad) over ONE flat float32 bucket (params/grads/exp_avg/exp_avg_sq
 * are each a single contiguous array - the same bucket the NCCL all-reduce uses).
 * xb_grad_sumsq  : norm_out[0] = sqrt(sum g^2) * grad_scale   (deterministic two-level reduction)
 * xb_adam_step   : g' = g * grad_scale * min(1, max_norm/(norm+1e-6)) (max_norm <= 0: no clip);
 *                  m = m + (g'-m)*(1-b1); v = v*b2 + g'*g'*(1-b2); p -= step_size * m/(sqrt(v)/bc2_sqrt + eps)
 *                  hyper (device, float32[4]) = {step_size = lr/(1-b1^t), bc2_sqrt = sqrt(1-b2^t), unused, unused}
 *                  write_back_grad != 0 stores g' into g (what clip_grad_norm_ leaves in .grad)
 * xb_soft_update : target = target*(1-tau) + tau*source    (SoftActorCritic.soft_update, actor_critic.py:155-158)
 */
int xb_grad_sumsq(const float *g, int64_t n, float grad_scale, float *norm_out, double *scratch, void *stream);
int xb_adam_step(float *p, float *g, float *m, float *v, int64_t n, const float *hyper,
                 float beta1, float beta2, float eps, float max_norm, const float *norm, float grad_scale,
                 int write_back_grad, void *stream);
int xb_soft_update(float *target, const float *source, int64_t n, float tau, void *stream);

/* ---------------------------------------------------------------- K10/K11: device-side rollout glue ---
 * SURVEY.md section 8f-1: what OnPolicyAgent.get_actions does after the network (core/on_policy.py:128-169) and what
 * Agent._process_observation / RunningMeanStd.update do before it (agents/base/agent.py:262-279,
 * common/statistic_tools.py:117-185), each as ONE launch writing straight into device buffers (e.g. the K1 staging
 * rows of the rollout buffer), so that a vector-env step costs one H2D of observations and one D2H of N int32 actions.
 *
 * xb_categorical_act: CategoricalDistribution over logits[N,A] (modules/distributions.py:128-162), A <= 64.
 *   forced_actions != NULL : a_n = (int)forced_actions[n]          (log_prob / entropy of given actions)
 *   else uniforms != NULL  : a_n = min{i : u_n < p_0+..+p_i}, u in [0,1) (stochastic_sample; inverse CDF in index order,
 *                            last index if rounding leaves the total mass below u_n)
 *   else                   : a_n = first argmax_i p_i               (deterministic_sample)
 *   outputs (each nullable, at least one): actions_f32[N] (the float32 the buffers store), actions_i32[N] (for the
 *   host-side env step), logp[N] = log_softmax(logits)[a], entropy[N] = -sum p log p.
 * xb_gaussian_act: DiagGaussianDistribution over Normal(mu[N,D], exp(log_std[D])) (distributions.py:165-197), D <= 64.
 *   forced_actions[N,D] != NULL : a = forced_actions                (log_prob / entropy of given actions)
 *   else noise[N,D] != NULL     : a = mu + noise * sigma, rounded after the product and after the sum as Normal.rsample
 *                                 (noise: standard normal draws supplied by the caller)
 *   else                        : a = mu                            (deterministic_sample)
 *   outputs (each nullable, at least one): actions_f32[N,D] (what the env steps with and the buffer stores),
 *   logp[N] = sum_d Normal.log_prob(a), entropy[N] = sum_d Normal.entropy().
 * xb_rms_update_normalize: x[N,D] float32.
 *   update != 0: (mean, var)[D] <- parallel-variance merge with the batch moments, float32 in the reference's operation
 *                order; `count` is the running count BEFORE the merge (host state, Python float in the reference).
 *   out != NULL: out = clip((x - mean) / (sqrt(var) + eps), -clip_range, clip_range) with the UPDATED statistics
 *                (PPO_Agent.train calls obs_rms.update(obs) and then _process_observation(obs), ppo_agent.py:115-116).
 */
int xb_categorical_act(const float *logits, const float *uniforms, const float *forced_actions, int N, int A,
                       float *actions_f32, int32_t *actions_i32, float *logp, float *entropy, void *stream);
int xb_gaussian_act(const float *mu, const float *log_std, const float *noise, const float *forced_actions, int N, int D,
                    float *actions_f32, float *logp, float *entropy, void *stream);
int xb_rms_update_normalize(const float *x, int N, int64_t D, float *mean, float *var, double count, int update,
                            float *out, float clip_range, float eps, void *stream);

/* ---------------------------------------------------------------- K12: tensor-core layers (tcgen05 / TMEM) ------
 * The pixel encoders' convolutions and hidden layer (NatureCNN of AC_CNN_Atari / Basic_CNN: rl_models/representations/cnn.py:
 * 45-50, 84-101; layers.py:16-65), forward, data gradient and weight gradient, that cuDNN runs as CUDA-core fp32 kernels
 * (85 % of the fp32 PPO update).  Every float32 operand travels as 1-3 bfloat16 "planes" (x = sum of its planes; plane q =
 * bf16 of the residual left by the planes before it: 1 plane is exact for integers <= 256 such as raw uint8 pixels, 2
 * planes are exact to 2^-16, 3 planes to 2^-24); products are accumulated in float32 in TMEM, one accumulator per order of
 * magnitude (plane-index sum), added smallest first in the epilogue.  planes_a <= planes_b; kept products: index sum <
 * planes_b.
 * xb_split_bf16       : x (float32[n]) -> planes[0] = bf16(x), planes[1] = bf16(x - planes[0]), [planes[2] = ...]
 * xb_pack_conv_weight : torch [N, C, KH, KW] float32 (* scale) -> bf16 planes of [N, (kh, kw, c)] (also a Linear over a
 *                       [C,H,W] flatten).  scale = 1/255 folds `observations / 255.0` (cnn.py:98) into the first layer,
 *                       whose A operand is then the raw uint8 pixel as ONE exact bf16 plane.
 * xb_gemm_gather_tc   : D[m,n] = sum_{t,c} in[b, y*sy+dy[t], x*sx+dx[t], c] * W[n, t*C+c] (+bias, ReLU), m = (b,y,x) over
 *                       [B,OY,OX], n < N; in / W as bf16 planes (NHWC, [N,K]); a work item is (128 sites, n_tile columns),
 *                       planes_b * n_tile <= 256, n_tile % 32 == 0, N % n_tile == 0; result as float32 and / or
 *                       planes_out bf16 planes written to columns [out_c0, out_c0+N) of row
 *                       (b*out_H + y*oys+oy0)*out_W + x*oxs+ox0 of a matrix with out_ld elements per row
 *                       (out_ld % 8 == out_c0 % 8 == 0).  C % 8 == 0, (T*C) % 64 == 0, T <= 64; dy / dx are HOST arrays
 *                       (copied into the launch parameters).  relu_mask (nullable, bf16, the output's pixel index in a
 *                       matrix of mask_ld elements per pixel from column mask_c0; mask_ld = 0: addressed exactly like
 *                       the output): result zeroed where mask <= 0 - the ReLU derivative applied to a data gradient,
 *                       mask = plane 0 of the saved activation.  colsum (nullable, float32 [ceil(M/128)][N]): row i =
 *                       column sums of the result rows of M tile i (after bias / ReLU / mask; deterministic) - the
 *                       partials of the bias gradient of the layer whose output gradient this call produces
 *                       (finish with xb_wgrad_reduce(colsum, tiles, N, 1, 1, 1, 1.0, db)).  Forward conv: dy = kh - pad, (sy,sx) = stride; Linear: one tap;
 *                       data gradients: flipped taps over the output gradient, one call per stride phase.
 * xb_wgrad_gather_tc  : weight gradient of the same gathered GEMM: partials[s, (t,c), n] = sum over the sites of split s of
 *                       in[b, y*sy+dy[t], x*sx+dx[t], c] * G[site*g_ld + n]; G = output gradient planes.  Both operands
 *                       are fed MN-major (16-byte units transposed into the core matrices); one work item =
 *                       (128 columns of (t,c), n_tile columns, split).  partials: float32 [splits, T*C, N].
 * xb_wgrad_reduce     : dw[N, C, KH, KW] (torch layout) (+)= scale * sum_s partials[s, (kh,kw,c), n], splits added in a fixed
 *                       order; `partials` is scratch: with more than 256 splits groups of rows are folded in place first. */
int xb_split_bf16(const float *x, int64_t n, int planes, void *out /* bf16 [planes, n] */, void *stream);
/* K3 variant that feeds K12: gathers uint8 rows (sample_batch, memory_tools.py:64-84; idx NULL = rows 0..B-1) and writes
 * dst[q, b, :] = plane q of float32(x)/255.0f for q < planes (bf16 [planes, B, row_bytes], planes 2 or 3), or with
 * planes == 1 the raw pixel value as one exact bf16 plane (the 1/255 lives in the packed weights); row_bytes % 16 == 0. */
int xb_gather_obs_planes(const uint8_t *src, const int64_t *idx, int64_t B, int64_t row_bytes, int planes, void *dst,
                         void *stream);
int xb_pack_conv_weight(const float *w, int N, int C, int KH, int KW, int planes, float scale,
                        void *out /* bf16 [planes, N, KH*KW*C] */, void *stream);
/* One operand form of one weight (xb_pack_weights): torch weight w [N, C, KH, KW] float32 (a Linear layer over a flattened
 * [C, H, W] feature map is N x C x H x W) -> bf16 planes out [planes][rows][cols] of scale * w, with
 *   mode 0: rows = N, cols = (kh, kw, c)            the B operand of the forward GEMM (= xb_pack_conv_weight)
 *   mode 1: rows = (kh, kw, c), cols = N            its transpose: the B operand of a Linear layer's data gradient
 *   mode 2: rows = C, cols = (tap, n), tap t = (kh[t], kw[t])   the B operand of one stride phase of a convolution's data
 *                                                    gradient (flipped taps in the order of the launch's chunks) */
#define XB_PACK_MAX_JOBS 16
#define XB_PACK_MAX_TAPS 16
typedef struct XbPackJob {
    const float *w;
    void *out;
    int N, C, KH, KW;
    int mode, n_taps;
    signed char kh[XB_PACK_MAX_TAPS], kw[XB_PACK_MAX_TAPS];
    float scale;
    int planes;
} XbPackJob;
/* Every operand form an encoder needs for one update in ONE launch: jobs is a HOST array (copied into the launch parameters),
 * n_jobs <= XB_PACK_MAX_JOBS.  Replaces one xb_pack_conv_weight / transpose / xb_split_bf16 launch per form. */
int xb_pack_weights(const XbPackJob *jobs, int n_jobs, void *stream);
int xb_gemm_gather_tc(int planes_a, int planes_b, const void *in, int64_t in_plane, const void *w, int64_t w_plane,
                      const float *bias, const void *relu_mask, int64_t mask_ld, int mask_c0, int B, int IH, int IW, int C,
                      int OY, int OX, int sy, int sx, int T, const int8_t *dy, const int8_t *dx, int N, int n_tile, int relu,
                      void *out_planes, int64_t out_plane, int planes_out, float *out_f32, int out_H, int out_W, int oys,
                      int oxs, int oy0, int ox0, int64_t out_ld, int out_c0, float *colsum, void *stream);
/* xb_gemm_gather_tc for a convolution whose input is stored in a PADDED-ROW layout [planes][B * hp_in][W][C] (hp_in rows per
 * image of which the first / last are zero padding), with the A operand fetched by TMA: a work item is box_h consecutive
 * grid rows x box_px sites (<= 128 GEMM rows); chunk i (64 K values = box_c = 64 channels of one pixel; a 32-channel tensor
 * is passed as its 64-channel pixel-pair view) is ONE box per plane at channel c0[i], pixel w0[i] (negative = left padding,
 * zero-filled by the TMA unit), rows tile_row0 * row_step + r0[i] + k * row_step, k < box_h (the tensor is described to the
 * TMA unit as {channel, pixel, row mod row_step, row / row_step, plane}; in_rows must be a multiple of row_step).
 * relu_mask rows are the output's, in a tensor mask_W pixels wide with the pixel index shifted by mask_x0 (mask_W = 0: laid
 * out exactly like the output).  Output sites are indexed over a padded grid too: hp rows per image, rows y0..y1 valid (the
 * others are never written: the caller keeps them zero), row y lands at ((b*out_H + (y-y0)*oys + oy0)*out_W + x*oxs + ox0).
 * W is [planes_b][N][n_chunks*64] in chunk order.  Everything else as xb_gemm_gather_tc. */
int xb_gemm_box_tc(int planes_a, int planes_b, const void *in, int64_t in_plane, int C, int W, int64_t in_rows, int box_c,
                   int box_px, int box_h, int row_step, int n_chunks, const int16_t *c0, const int16_t *w0, const int16_t *r0,
                   const void *w, int64_t w_plane, const float *bias, const void *relu_mask, int mask_W, int mask_x0, int B,
                   int hp, int y0, int y1, int N, int n_tile, int relu, void *out_planes, int64_t out_plane, int planes_out,
                   float *out_f32, int out_H, int out_W, int oys, int oxs, int oy0, int ox0, int64_t out_ld, int out_c0,
                   float *colsum, void *stream);
/* The gathered GEMM with the activation tile RESIDENT in shared memory ("halo" mode): stride-1 gathers over a 64-channel
 * padded-row tensor in [planes][B*hp rows][W pixels][64] (in_rows = B*hp) - a 3x3 convolution, its data gradient, the stride
 * phases of a strided convolution's data gradient.  The sites are the positions of the haloed raster: row R (image R / hp,
 * padded row y = R % hp), column hc = pixel hc + halo_w0 (halo_w0 <= 0, halo_w columns per row; pixels outside [0, W) read
 * as zero); an M tile is 128 consecutive positions and ONE TMA box per plane holds every input its taps read.  Sub-item j
 * (n_sub <= 4: the n tiles of a forward layer or the stride phases of a data gradient) multiplies with rows j*N .. of
 * w [planes_b][n_sub*N][n_chunks*64]; its chunk i reads the site (R + dr[j*n_chunks+i], pixel + dc[..]) - a descriptor
 * offset into the resident tile.  Valid sites of sub-item j: y0 <= y <= sub_y1[j], 0 <= x <= sub_x1[j]; they land at row
 * ((b*out_H + (y-y0)*oys + sub_oy0[j])*out_W + x*oxs + sub_ox0[j]) of the output, columns out_c0 + j*N (same_cols: out_c0 for
 * every sub-item).  n_sub * n_chunks <= 16.  bias / relu / relu_mask (mask_W, mask_x0) / planes / colsum
 * ([ceil(B*hp*halo_w / 128) * n_sub][N]) as xb_gemm_box_tc. */
int xb_gemm_halo_tc(int planes_a, int planes_b, const void *in, int64_t in_plane, int W, int64_t in_rows, int halo_w, int halo_w0,
                    int n_sub, int n_chunks, const int16_t *dr, const int16_t *dc, const void *w, int64_t w_plane,
                    const float *bias, const void *relu_mask, int mask_W, int mask_x0, int B, int hp, int y0,
                    const int16_t *sub_y1, const int16_t *sub_x1, int N, int relu, void *out_planes, int64_t out_plane,
                    int planes_out, float *out_f32, int out_H, int out_W, int oys, int oxs, const int16_t *sub_oy0,
                    const int16_t *sub_ox0, int64_t out_ld, int out_c0, int same_cols, float *colsum, void *stream);
/* Weight gradient of the same convolution with both operands fetched by TMA boxes: `in` as for xb_gemm_box_tc, `g` the
 * output gradient in the padded site layout [planes_b][g_rows][box_px*box_c/64 sites][N]; a chunk of the reduction is box_h
 * grid rows (box_w * box_h <= 64 sites), N % 64 == 0; partials: float32 [splits, n_chunks*64, N] (reduce with xb_wgrad_reduce). */
int xb_wgrad_box_tc(int planes_a, int planes_b, const void *in, int64_t in_plane, int C, int W, int64_t in_rows, int box_c,
                    int box_px, int box_h, int row_step, int n_chunks, const int16_t *c0, const int16_t *w0, const int16_t *r0,
                    const void *g, int64_t g_plane, int64_t g_rows, int N, int splits, float *partials, void *stream);
/* Diagnostics (XB_K12_TIMING=1 in the environment): per CTA of the LAST K12 launch, clock64 cycles of each warp role and of its
 * barrier waits: out_host[cta][12] = {MMA total, MMA wait operands, MMA wait epilogue, MMA wait resident tile, producer total,
 * producer wait ring, producer wait tile buffer, epilogue total, epilogue wait accumulator, ...}.  Synchronises the device. */
int xb_debug_k12_timing(unsigned long long *out_host, int n_ctas);
/* Test hook: the raw shared-memory image (first out_bytes, 0xEE = untouched) after ONE TMA box load of the 4-D tensor map the
 * box mode builds - lets the tests pin the layout (pixel packing, row step, 128-byte swizzle, zero fill) byte for byte. */
int xb_debug_tma_box(const void *in, int64_t in_plane, int planes, int C, int W, int64_t rows, int box_c, int box_px, int box_h,
                     int row_step, int c0, int c1, int c2, int c3, uint32_t expect_bytes, void *out, uint32_t out_bytes,
                     void *stream);
int xb_wgrad_gather_tc(int planes_a, int planes_b, const void *in, int64_t in_plane, const void *g, int64_t g_plane,
                       int64_t g_ld, int B, int IH, int IW, int C, int OY, int OX, int sy, int sx, int T, const int8_t *dy,
                       const int8_t *dx, int N, int n_tile, int splits, float *partials, void *stream);
int xb_wgrad_reduce(float *partials, int splits, int N, int C, int KH, int KW, float scale, float *dw, int accumulate,
                    void *stream);

#ifdef __cplusplus
}
#endif
#endif /* XB200_H_ */
