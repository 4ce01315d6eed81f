// K4 fused PPO-Clip loss forward+backward, K6 DQN TD target + loss forward+backward.
// Elementwise + row reductions over tiny rows (A <= 64 logits): one thread per sample, float4 loads when the
// row width allows, deterministic two-level reduction of the logged statistics.
#include "xb_common.cuh"

// =====================================================================================================
// K4  xb_ppo_loss_fwd_bwd
// =====================================================================================================
// Mirrors torch semantics of xuance/torch/learners/policy_gradient/ppo_learner.py:46-60:
//   Categorical(logits): logp_i = z_i - logsumexp(z);  entropy = -sum p_i*logp_i
//   torch.minimum backward: ties split the gradient in half; clamp backward passes inside [lo,hi] inclusive.
template <int A_MAX>
__global__ void __launch_bounds__(256, (A_MAX <= 4 ? 3 : 1)) ppo_loss_kernel(const float *__restrict__ logits,
                                                       const float *__restrict__ value,
                                                       const float *__restrict__ actions,
                                                       const float *__restrict__ old_logp,
                                                       const float *__restrict__ adv, const float *__restrict__ ret,
                                                       int64_t B, int A, float inv_bt, float clip, float vf_coef,
                                                       float ent_coef, int loss_kind, float *__restrict__ dlogits,
                                                       float *__restrict__ dvalue, float *__restrict__ stats,
                                                       double *__restrict__ scratch) {
    __shared__ double red[6 * 32];
    double acc[6] = {0, 0, 0, 0, 0, 0};  // a_loss, c_loss, entropy, v, clipped count, (unused)
    const float lo = 1.0f - clip, hi = 1.0f + clip;
    struct Row {
        float z[A_MAX];
        float v, act, ol, ad, r;
    };
    auto load_row = [&](int64_t b, Row &in) {
        const float *zr = logits + b * A;
        if (A_MAX == 4 && A == 4) {  // the BASELINE action count: one 16-byte load per row
            const float4 z4 = *reinterpret_cast<const float4 *>(zr);
            in.z[0] = z4.x, in.z[1] = z4.y, in.z[2] = z4.z, in.z[3] = z4.w;
        } else {
#pragma unroll
            for (int i = 0; i < A_MAX; ++i)
                if (i < A) in.z[i] = zr[i];
        }
        in.v = value[b], in.act = actions[b], in.ad = adv[b], in.r = ret[b];
        in.ol = (loss_kind == 0) ? old_logp[b] : 0.f;
    };
    auto compute_row = [&](int64_t b, const Row &in) {
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < A_MAX; ++i)
            if (i < A) m = fmaxf(m, in.z[i]);
        float se = 0.f;
#pragma unroll
        for (int i = 0; i < A_MAX; ++i)
            if (i < A) se += expf(in.z[i] - m);
        const float lse = m + logf(se);
        const int a = (int)in.act;
        float ent = 0.f, logp_a = 0.f;
        float p[A_MAX], lp[A_MAX];
#pragma unroll
        for (int i = 0; i < A_MAX; ++i) {
            if (i < A) {
                lp[i] = in.z[i] - lse;
                p[i] = expf(lp[i]);
                ent -= p[i] * lp[i];
                if (i == a) logp_a = lp[i];
            }
        }
        const float ad = in.ad;
        float ratio = 1.f, smin, d_logp;
        if (loss_kind == 0) {  // PPO-Clip surrogate
            ratio = expf(logp_a - in.ol);
            const float rc = fminf(fmaxf(ratio, lo), hi);
            const float s1 = rc * ad, s2 = ad * ratio;
            smin = fminf(s1, s2);
            // d(-mean(min(s1,s2)))/d ratio
            float g1 = s1 < s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
            float g2 = s2 < s1 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
            const bool inside = ratio >= lo && ratio <= hi;
            const float d_ratio = -inv_bt * ad * ((inside ? g1 : 0.f) + g2);
            d_logp = d_ratio * ratio;  // d ratio / d logp = ratio
        } else {               // plain policy gradient: a_loss = -mean(w * logp)   (A2C: w = advantage, PG: w = return)
            smin = ad * logp_a;
            d_logp = -inv_bt * ad;
        }
        const float dent = -ent_coef * inv_bt;  // d loss / d entropy_b
        float *dz = dlogits + b * A;
        float gz[A_MAX];
#pragma unroll
        for (int i = 0; i < A_MAX; ++i) {
            if (i < A) {
                float g = d_logp * ((i == a ? 1.f : 0.f) - p[i]);  // d logp_a / d z_i
                g += dent * (-p[i] * (lp[i] + ent));               // d H / d z_i
                gz[i] = g;
            }
        }
        if (A_MAX == 4 && A == 4) {
            *reinterpret_cast<float4 *>(dz) = make_float4(gz[0], gz[1], gz[2], gz[3]);
        } else {
#pragma unroll
            for (int i = 0; i < A_MAX; ++i)
                if (i < A) dz[i] = gz[i];
        }
        const float dv = in.v - in.r;
        dvalue[b] = vf_coef * 2.f * dv * inv_bt;
        acc[0] += (double)(-smin);
        acc[1] += (double)dv * (double)dv;
        acc[2] += (double)ent;
        acc[3] += (double)in.v;
        acc[4] += (ratio < lo || ratio > hi) ? 1.0 : 0.0;
    };
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (A_MAX <= 4) {
        // two rows in flight per thread: the loads of the second row are issued before the (transcendental-heavy)
        // arithmetic of the first - the kernel is latency-bound on its global loads otherwise (ncu: long_scoreboard)
        for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += 2 * stride) {
            Row r0, r1;
            const bool two = b + stride < B;
            load_row(b, r0);
            if (two) load_row(b + stride, r1);
            compute_row(b, r0);
            if (two) compute_row(b + stride, r1);
        }
    } else {
        for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += stride) {
            Row r0;
            load_row(b, r0);
            compute_row(b, r0);
        }
    }
    grid_sum_finalize<6>(acc, scratch, red, [&](double(&t)[6]) {
        const double ib = (double)inv_bt;
        float a_loss = (float)(t[0] * ib), c_loss = (float)(t[1] * ib), e = (float)(t[2] * ib);
        stats[0] = a_loss;
        stats[1] = c_loss;
        stats[2] = e;
        stats[3] = (float)(t[3] * ib);
        stats[4] = (float)(t[4] * ib);
        stats[5] = a_loss - ent_coef * e + vf_coef * c_loss;
        stats[6] = 0.f;
        stats[7] = 0.f;
    });
}

extern "C" int xb_ppo_loss_fwd_bwd(const float *logits, const float *value, const float *actions,
                                   const float *old_logp, const float *adv, const float *ret, int64_t B, int A,
                                   int64_t B_total, float clip_range, float vf_coef, float ent_coef, int loss_kind,
                                   float *dlogits, float *dvalue, float *stats, double *scratch, void *stream) {
    if (!logits || !value || !actions || !adv || !ret || !dlogits || !dvalue || !stats || !scratch) return XB_EINVAL;
    if (loss_kind != 0 && loss_kind != 1) return XB_EINVAL;
    if (loss_kind == 0 && !old_logp) return XB_EINVAL;
    if (B <= 0 || B_total < B || A <= 0) return XB_EINVAL;
    if (A > 64) return XB_ERANGE;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t want = (B + 255) / 256;
    int grid = (int)(want < XB_MAX_PARTIALS ? want : XB_MAX_PARTIALS);
    const float inv_bt = 1.0f / (float)B_total;
    if (A == 4 && (!xb_aligned(logits, 16) || !xb_aligned(dlogits, 16))) return XB_EALIGN;
#define XB_PPO(AM)                                                                                                   \
    ppo_loss_kernel<AM><<<grid, 256, 0, s>>>(logits, value, actions, old_logp, adv, ret, B, A, inv_bt, clip_range,   \
                                              vf_coef, ent_coef, loss_kind, dlogits, dvalue, stats, scratch)
    if (A <= 4) XB_PPO(4);
    else if (A <= 8) XB_PPO(8);
    else if (A <= 18) XB_PPO(18);
    else if (A <= 32) XB_PPO(32);
    else XB_PPO(64);
#undef XB_PPO
    return xb_launch_status();
}

// =====================================================================================================
// K4-G  xb_ppo_gaussian_loss_fwd_bwd
// =====================================================================================================
// The same losses for a diagonal Gaussian policy, torch.distributions.Normal(mu, exp(log_std)) as ppo_learner.py:46-60
// uses it through DiagGaussianDistribution (log_prob and entropy summed over the action dimensions):
//   logp_b = sum_d [-(a-mu)^2 / (2 var) - log sigma - log sqrt(2 pi)],  H = sum_d [0.5 + 0.5 log(2 pi) + log sigma]
//   d logp_b / d mu_d = (a-mu)/var,  d logp_b / d log_std_d = (a-mu)^2/var - 1,  d H / d log_std_d = 1
// dlog_std is a reduction over every row: per-thread float partials, then warp / block / grid sums in double and in a
// fixed order (deterministic), the block partials in col_scratch[D][XB_MAX_PARTIALS] and the logged statistics in the
// K4 scratch, both finished by the last block to arrive.
extern "C" int64_t xb_gaussian_scratch_doubles(int D) {
    return (D <= 0 || D > 64) ? 0 : (int64_t)D * XB_MAX_PARTIALS;
}

template <int D_MAX>
__global__ void __launch_bounds__(256) ppo_gaussian_loss_kernel(
    const float *__restrict__ mu, const float *__restrict__ log_std, const float *__restrict__ value,
    const float *__restrict__ actions, const float *__restrict__ old_logp, const float *__restrict__ adv,
    const float *__restrict__ ret, int64_t B, int D, int64_t B_total, float inv_bt, float clip, float vf_coef,
    float ent_coef, int loss_kind, float *__restrict__ dmu, float *__restrict__ dvalue, float *__restrict__ dlog_std,
    float *__restrict__ stats, double *__restrict__ scratch, double *__restrict__ col_scratch) {
    __shared__ double red[6 * 32];
    __shared__ double col_red[D_MAX * 8];  // [d][warp], 8 warps of 256 threads
    __shared__ float s_inv_var[D_MAX], s_two_var[D_MAX], s_log_scale[D_MAX];
    __shared__ float s_entropy;
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (threadIdx.x < D) {
        const float sigma = expf(log_std[threadIdx.x]);
        const float var = sigma * sigma;  // Normal.log_prob: var = scale ** 2, log_scale = scale.log()
        s_inv_var[threadIdx.x] = 1.0f / var;
        s_two_var[threadIdx.x] = 2.0f * var;
        s_log_scale[threadIdx.x] = logf(sigma);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float h = 0.f;
        for (int d = 0; d < D; ++d) h += (float)(0.5 + XB_LOG_SQRT_2PI) + s_log_scale[d];
        s_entropy = h;
    }
    __syncthreads();
    const float lo = 1.0f - clip, hi = 1.0f + clip, ent = s_entropy;
    double acc[6] = {0, 0, 0, 0, 0, 0};  // a_loss, c_loss, entropy, v, clipped count, (unused)
    float col[D_MAX];                     // this thread's share of sum_b dlogp_b * ((a-mu)^2/var - 1)
#pragma unroll
    for (int d = 0; d < D_MAX; ++d) col[d] = 0.f;
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        const float *mr = mu + b * D, *ar = actions + b * D;
        float diff[D_MAX];
        float logp = 0.f;
#pragma unroll
        for (int d = 0; d < D_MAX; ++d) {
            if (d < D) {
                diff[d] = ar[d] - mr[d];
                logp += -(diff[d] * diff[d]) / s_two_var[d] - s_log_scale[d] - (float)XB_LOG_SQRT_2PI;
            }
        }
        const float ad = adv[b];
        float ratio = 1.f, smin, d_logp;
        if (loss_kind == 0) {  // PPO-Clip surrogate (same arithmetic as K4)
            ratio = expf(logp - old_logp[b]);
            const float rc = fminf(fmaxf(ratio, lo), hi);
            const float s1 = rc * ad, s2 = ad * ratio;
            smin = fminf(s1, s2);
            float g1 = s1 < s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
            float g2 = s2 < s1 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
            const bool inside = ratio >= lo && ratio <= hi;
            d_logp = -inv_bt * ad * ((inside ? g1 : 0.f) + g2) * ratio;
        } else {  // plain policy gradient: a_loss = -mean(w * logp)
            smin = ad * logp;
            d_logp = -inv_bt * ad;
        }
        float *gr = dmu + b * D;
#pragma unroll
        for (int d = 0; d < D_MAX; ++d) {
            if (d < D) {
                const float z = diff[d] * s_inv_var[d];
                gr[d] = d_logp * z;
                col[d] += d_logp * (z * diff[d] - 1.f);
            }
        }
        const float v = value[b], dv = v - ret[b];
        dvalue[b] = vf_coef * 2.f * dv * inv_bt;
        acc[0] += (double)(-smin);
        acc[1] += (double)dv * (double)dv;
        acc[2] += (double)ent;
        acc[3] += (double)v;
        acc[4] += (ratio < lo || ratio > hi) ? 1.0 : 0.0;
    }
    // per-dimension block partial: warps in shuffle order, then the block's warps in index order
#pragma unroll
    for (int d = 0; d < D_MAX; ++d) {
        if (d < D) {
            const double s = warp_sum_d((double)col[d]);
            if (lane == 0) col_red[d * 8 + warp] = s;
        }
    }
    __syncthreads();
    if (threadIdx.x < D) {
        double s = 0.0;
        for (int w = 0; w < nwarps; ++w) s += col_red[threadIdx.x * 8 + w];
        col_scratch[(int64_t)threadIdx.x * XB_MAX_PARTIALS + blockIdx.x] = s;
        __threadfence();
    }
    // statistics partials + arrival ticket (the __syncthreads inside block_sum_d orders the column stores above)
    int *ticket = reinterpret_cast<int *>(scratch + 8 * XB_MAX_PARTIALS);
    block_sum_d<6>(acc, red);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 6; ++k) scratch[k * XB_MAX_PARTIALS + blockIdx.x] = acc[k];
        __threadfence();
        is_last = (atomicAdd(ticket, 1) == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const double d_ent = -(double)ent_coef * (double)B / (double)B_total;  // d(-ent_coef * mean_b H) / d log_std_d
    for (int d = warp; d < D; d += nwarps) {
        double s = 0.0;
        for (int blk = lane; blk < (int)gridDim.x; blk += 32) s += __ldcg(&col_scratch[(int64_t)d * XB_MAX_PARTIALS + blk]);
        s = warp_sum_d(s);
        if (lane == 0) dlog_std[d] = (float)(s + d_ent);
    }
    double t[6] = {0, 0, 0, 0, 0, 0};
    for (int blk = threadIdx.x; blk < (int)gridDim.x; blk += blockDim.x) {
#pragma unroll
        for (int k = 0; k < 6; ++k) t[k] += __ldcg(&scratch[k * XB_MAX_PARTIALS + blk]);
    }
    __syncthreads();
    block_sum_d<6>(t, red);
    if (threadIdx.x == 0) {
        *ticket = 0;  // re-arm for the next launch
        const double ib = (double)inv_bt;
        float a_loss = (float)(t[0] * ib), c_loss = (float)(t[1] * ib), e = (float)(t[2] * ib);
        stats[0] = a_loss;
        stats[1] = c_loss;
        stats[2] = e;
        stats[3] = (float)(t[3] * ib);
        stats[4] = (float)(t[4] * ib);
        stats[5] = a_loss - ent_coef * e + vf_coef * c_loss;
        stats[6] = 0.f;
        stats[7] = 0.f;
    }
}

extern "C" int xb_ppo_gaussian_loss_fwd_bwd(const float *mu, const float *log_std, const float *value,
                                            const float *actions, const float *old_logp, const float *adv,
                                            const float *ret, int64_t B, int D, int64_t B_total, float clip_range,
                                            float vf_coef, float ent_coef, int loss_kind, float *dmu, float *dvalue,
                                            float *dlog_std, float *stats, double *scratch, double *col_scratch,
                                            void *stream) {
    if (!mu || !log_std || !value || !actions || !adv || !ret || !dmu || !dvalue || !dlog_std || !stats || !scratch ||
        !col_scratch)
        return XB_EINVAL;
    if (loss_kind != 0 && loss_kind != 1) return XB_EINVAL;
    if (loss_kind == 0 && !old_logp) return XB_EINVAL;
    if (B <= 0 || B_total < B || D <= 0) return XB_EINVAL;
    if (D > 64) return XB_ERANGE;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t want = (B + 255) / 256;
    int grid = (int)(want < XB_MAX_PARTIALS ? want : XB_MAX_PARTIALS);
    const float inv_bt = 1.0f / (float)B_total;
#define XB_PPO_G(DM)                                                                                                  \
    ppo_gaussian_loss_kernel<DM><<<grid, 256, 0, s>>>(mu, log_std, value, actions, old_logp, adv, ret, B, D, B_total, \
                                                      inv_bt, clip_range, vf_coef, ent_coef, loss_kind, dmu, dvalue,  \
                                                      dlog_std, stats, scratch, col_scratch)
    if (D <= 8) XB_PPO_G(8);
    else if (D <= 18) XB_PPO_G(18);
    else if (D <= 32) XB_PPO_G(32);
    else XB_PPO_G(64);
#undef XB_PPO_G
    return xb_launch_status();
}

// =====================================================================================================
// K6  xb_dqn_td_fwd_bwd
// =====================================================================================================
__global__ void __launch_bounds__(256) dqn_td_kernel(const float *__restrict__ q_eval, const float *__restrict__ q_next,
                                                     const float *__restrict__ q_sel,
                                                     const float *__restrict__ actions, const float *__restrict__ rew,
                                                     const float *__restrict__ term, int64_t B, int A, float inv_bt,
                                                     float gamma, float *__restrict__ dq, float *__restrict__ td,
                                                     float *__restrict__ stats, double *__restrict__ scratch) {
    __shared__ double red[2 * 32];
    double acc[2] = {0, 0};
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
        const int a = (int)actions[b];
        const float *qe = q_eval + b * A, *qn = q_next + b * A;
        float mx = -INFINITY;
        if (q_sel) {  // double-Q: evaluate the target net at the eval net's greedy action (ddqn_learner.py:39-44)
            const float *qs = q_sel + b * A;
            int best = 0;
            float bv = qs[0];
            for (int i = 1; i < A; ++i)
                if (qs[i] > bv) {  // first maximal index, as torch.argmax
                    bv = qs[i];
                    best = i;
                }
            mx = qn[best];
        } else {
            for (int i = 0; i < A; ++i) mx = fmaxf(mx, qn[i]);
        }
        const float pred = qe[a];
        // targetQ = rew + gamma*(1-ter)*max  evaluated left to right as torch does: (gamma*(1-ter))*max
        const float y = __fadd_rn(rew[b], __fmul_rn(__fmul_rn(gamma, __fsub_rn(1.f, term[b])), mx));
        const float e = __fsub_rn(y, pred);  // td_error = targetQ - predictQ
        td[b] = e;
        float *g = dq + b * A;
        const float ga = -2.f * e * inv_bt;  // d mean((pred-y)^2) / d pred
        for (int i = 0; i < A; ++i) g[i] = (i == a) ? ga : 0.f;
        acc[0] += (double)e * (double)e;
        acc[1] += (double)pred;
    }
    grid_sum_finalize<2>(acc, scratch, red, [&](double(&t)[2]) {
        stats[0] = (float)(t[0] * (double)inv_bt);
        stats[1] = (float)(t[1] * (double)inv_bt);
        stats[2] = 0.f;
        stats[3] = 0.f;
    });
}

extern "C" int xb_dqn_td_fwd_bwd(const float *q_eval, const float *q_next, const float *q_sel, const float *actions,
                                 const float *rew,
                                 const float *term, int64_t B, int A, int64_t B_total, float gamma, float *dq,
                                 float *td, float *stats, double *scratch, void *stream) {
    if (!q_eval || !q_next || !actions || !rew || !term || !dq || !td || !stats || !scratch) return XB_EINVAL;
    if (B <= 0 || B_total < B || A <= 0) return XB_EINVAL;
    int64_t want = (B + 255) / 256;
    int grid = (int)(want < XB_MAX_PARTIALS ? want : XB_MAX_PARTIALS);
    dqn_td_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(q_eval, q_next, q_sel, actions, rew, term, B, A,
                                                          1.0f / (float)B_total, gamma, dq, td, stats, scratch);
    return xb_launch_status();
}
