// K10 categorical act (sample / argmax + log-prob + entropy) and K11 running mean/std update + observation normalise:
// the device-side rollout glue of SURVEY.md section 8f-1.  Both are per-vector-step kernels over N <= a few hundred
// rows: launch-latency bound by construction, written so that ONE launch replaces the ~15 small launches and the
// three device->host reads the reference's rollout loop issues per step (core/on_policy.py:128-169).
#include "xb_common.cuh"

// =====================================================================================================
// K10  xb_categorical_act
// =====================================================================================================
// torch.distributions.Categorical(logits=z) semantics (modules/distributions.py:128-162):
//   logp_i = z_i - logsumexp(z), p_i = exp(logp_i), entropy = -sum p_i logp_i,
//   deterministic_sample = argmax_i p_i (first maximal index),
//   stochastic sample: inverse CDF over p in index order with the caller's uniform u in [0,1)
//     a = min{ i : u < p_0 + ... + p_i }   (a = last index if rounding leaves the total below u)
// The reference draws with torch.multinomial from torch's RNG; a stream that differs by construction, so parity of the
// draw is defined on supplied uniforms (as for PER, K5) and parity of logp / entropy on the chosen action.
template <int A_MAX>
__global__ void __launch_bounds__(128) categorical_act_kernel(const float *__restrict__ logits,
                                                              const float *__restrict__ uniforms,
                                                              const float *__restrict__ forced, int N, int A,
                                                              float *__restrict__ act_f, int32_t *__restrict__ act_i,
                                                              float *__restrict__ logp, float *__restrict__ entropy) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float *zr = logits + (int64_t)n * A;
    float z[A_MAX];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < A_MAX; ++i)
        if (i < A) {
            z[i] = zr[i];
            m = fmaxf(m, z[i]);
        }
    float se = 0.f;
#pragma unroll
    for (int i = 0; i < A_MAX; ++i)
        if (i < A) se += expf(z[i] - m);
    const float lse = m + logf(se);
    float ent = 0.f, cdf = 0.f, best_p = -1.f, lp_a = 0.f, lp_best = 0.f, lp_last = 0.f;
    int a = -1, best = 0;
    const bool sample = uniforms != nullptr && forced == nullptr;
    const float u = sample ? uniforms[n] : 0.f;
    const int want = forced ? (int)forced[n] : -1;
#pragma unroll
    for (int i = 0; i < A_MAX; ++i) {
        if (i < A) {
            const float lp = z[i] - lse;
            const float p = expf(lp);
            ent -= p * lp;
            cdf += p;
            if (sample && a < 0 && u < cdf) {
                a = i;
                lp_a = lp;
            }
            if (p > best_p) {  // strict: first maximal index, as torch.argmax
                best_p = p;
                best = i;
                lp_best = lp;
            }
            lp_last = lp;
            if (i == want) lp_a = lp;
        }
    }
    if (forced) {
        a = want;
    } else if (!sample) {
        a = best;
        lp_a = lp_best;
    } else if (a < 0) {  // u >= rounded total mass: the last action
        a = A - 1;
        lp_a = lp_last;
    }
    if (act_f) act_f[n] = (float)a;
    if (act_i) act_i[n] = a;
    if (logp) logp[n] = lp_a;
    if (entropy) entropy[n] = ent;
}

extern "C" int xb_categorical_act(const float *logits, const float *uniforms, const float *forced_actions, int N, int A,
                                  float *actions_f32, int32_t *actions_i32, float *logp, float *entropy,
                                  void *stream) {
    if (!logits || N <= 0 || A <= 0) return XB_EINVAL;
    if (!actions_f32 && !actions_i32 && !logp && !entropy) return XB_EINVAL;
    if (A > 64) return XB_ERANGE;
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = (N + 127) / 128;
#define XB_ACT(AM)                                                                                                    \
    categorical_act_kernel<AM><<<grid, 128, 0, s>>>(logits, uniforms, forced_actions, N, A, actions_f32, actions_i32, \
                                                    logp, entropy)
    if (A <= 4) XB_ACT(4);
    else if (A <= 8) XB_ACT(8);
    else if (A <= 18) XB_ACT(18);
    else if (A <= 32) XB_ACT(32);
    else XB_ACT(64);
#undef XB_ACT
    return xb_launch_status();
}

// =====================================================================================================
// K10-G  xb_gaussian_act
// =====================================================================================================
// DiagGaussianDistribution over Normal(mu, exp(log_std)) (modules/distributions.py:165-197), one thread per row:
//   a = mu + noise * sigma  (Normal.rsample: one product, one sum, each rounded - no fused multiply-add)
//   logp = sum_d [-(a-mu)^2 / (2 var) - log sigma - log sqrt(2 pi)],  entropy = sum_d [0.5 + 0.5 log(2 pi) + log sigma]
// The reference draws with Normal.sample from torch's RNG; as for K10 the draw is defined on the caller's noise.
template <int D_MAX>
__global__ void __launch_bounds__(128) gaussian_act_kernel(const float *__restrict__ mu,
                                                           const float *__restrict__ log_std,
                                                           const float *__restrict__ noise,
                                                           const float *__restrict__ forced, int N, int D,
                                                           float *__restrict__ act_f, float *__restrict__ logp,
                                                           float *__restrict__ entropy) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int64_t o = (int64_t)n * D;
    float lp = 0.f, ent = 0.f;
#pragma unroll
    for (int d = 0; d < D_MAX; ++d) {
        if (d < D) {
            const float sigma = expf(log_std[d]);
            const float m = mu[o + d];
            float a = m;
            if (forced) a = forced[o + d];
            else if (noise) a = __fadd_rn(m, __fmul_rn(noise[o + d], sigma));
            const float diff = a - m, log_scale = logf(sigma);
            lp += -(diff * diff) / (2.0f * (sigma * sigma)) - log_scale - (float)XB_LOG_SQRT_2PI;
            ent += (float)(0.5 + XB_LOG_SQRT_2PI) + log_scale;
            if (act_f) act_f[o + d] = a;
        }
    }
    if (logp) logp[n] = lp;
    if (entropy) entropy[n] = ent;
}

extern "C" int xb_gaussian_act(const float *mu, const float *log_std, const float *noise, const float *forced_actions,
                               int N, int D, float *actions_f32, float *logp, float *entropy, void *stream) {
    if (!mu || !log_std || N <= 0 || D <= 0) return XB_EINVAL;
    if (!actions_f32 && !logp && !entropy) return XB_EINVAL;
    if (D > 64) return XB_ERANGE;
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = (N + 127) / 128;
#define XB_GACT(DM) \
    gaussian_act_kernel<DM><<<grid, 128, 0, s>>>(mu, log_std, noise, forced_actions, N, D, actions_f32, logp, entropy)
    if (D <= 8) XB_GACT(8);
    else if (D <= 18) XB_GACT(18);
    else if (D <= 32) XB_GACT(32);
    else XB_GACT(64);
#undef XB_GACT
    return xb_launch_status();
}

// =====================================================================================================
// K11  xb_rms_update_normalize
// =====================================================================================================
// RunningMeanStd.update + Agent._process_observation for a float32 batch x[N,D] (common/statistic_tools.py:117-185,
// agents/base/agent.py:262-279), one thread per feature column, float32 arithmetic in the reference's operation order
// (NumPy reduces axis 0 row after row; Python-float counts are weak scalars and enter every product as float32):
//   bm = (sum_n x) / N ; bv = square(sqrt((sum_n (x-bm)^2) / N))
//   delta = bm - mean ; tot = count + N
//   mean' = mean + delta*N/tot ; var' = (var*count + bv*N + delta^2*count*N/tot) / tot
//   out   = clip((x - mean') / (sqrt(var') + 1e-8), -range, range)
// `count` is host state (a Python float in the reference) and is passed by value; the caller adds N afterwards.
__global__ void __launch_bounds__(128) rms_update_normalize_kernel(const float *__restrict__ x, int N, int D,
                                                                   float *__restrict__ mean, float *__restrict__ var,
                                                                   double count, int update, float *__restrict__ out,
                                                                   float clip_range, float eps) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    float mu = mean[d], v = var[d];
    if (update) {
        float s = 0.f;
        for (int n = 0; n < N; ++n) s = __fadd_rn(s, x[(int64_t)n * D + d]);
        const float fn = (float)N;
        const float bm = __fdiv_rn(s, fn);
        float ss = 0.f;
        for (int n = 0; n < N; ++n) {
            const float c = __fsub_rn(x[(int64_t)n * D + d], bm);
            ss = __fadd_rn(ss, __fmul_rn(c, c));
        }
        const float bstd = sqrtf(__fdiv_rn(ss, fn));
        const float bv = __fmul_rn(bstd, bstd);
        const float cnt = (float)count, tot = (float)(count + (double)N);
        const float delta = __fsub_rn(bm, mu);
        const float new_mean = __fadd_rn(mu, __fdiv_rn(__fmul_rn(delta, fn), tot));
        const float m_a = __fmul_rn(v, cnt), m_b = __fmul_rn(bv, fn);
        const float cross = __fdiv_rn(__fmul_rn(__fmul_rn(__fmul_rn(delta, delta), cnt), fn), tot);
        const float m2 = __fadd_rn(__fadd_rn(m_a, m_b), cross);
        mu = new_mean;
        v = __fdiv_rn(m2, tot);
        mean[d] = mu;
        var[d] = v;
    }
    if (out) {
        const float denom = __fadd_rn(sqrtf(v), eps);
        for (int n = 0; n < N; ++n) {
            const float y = __fdiv_rn(__fsub_rn(x[(int64_t)n * D + d], mu), denom);
            out[(int64_t)n * D + d] = fminf(fmaxf(y, -clip_range), clip_range);
        }
    }
}

extern "C" int xb_rms_update_normalize(const float *x, int N, int64_t D, float *mean, float *var, double count,
                                       int update, float *out, float clip_range, float eps, void *stream) {
    if (!x || !mean || !var || N <= 0 || D <= 0) return XB_EINVAL;
    if (!update && !out) return XB_EINVAL;
    if (D > (int64_t)1 << 30) return XB_ERANGE;
    const int grid = (int)((D + 127) / 128);
    rms_update_normalize_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(x, N, (int)D, mean, var, count, update, out,
                                                                         clip_range, eps);
    return xb_launch_status();
}
