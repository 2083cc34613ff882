// Per-row PPO loss and its gradient w.r.t. the model outputs.
// Restates ray.rllib.agents.ppo.ppo_tf_policy.PPOLoss (1.0.1) with DiagGaussian logp / kl / entropy
// (ray.rllib.models.tf.tf_action_dist.DiagGaussian), FP32 like the TF graph.
// The loss separates into a policy part (function of the logits) and a value part (function of v), which the
// tensor-core kernel evaluates in two passes; ppo_row_loss runs both.
#pragma once
#include "common.cuh"

namespace ddrl {

constexpr float kHalfLog2PiE = 1.4189385332046727f;  // 0.5*log(2*pi*e)

// Policy part.  logits[0..2A) = (mean | log_std).  Writes dl[0..2A) = scale * d(-surr + klc*KL - ent_coeff*H)/dlogits
// and s[0] = -surr, s[1] = KL(old||new), s[3] = entropy.
__device__ __forceinline__ void ppo_row_policy(const float* logits, int A, const float* __restrict__ actions,
                                               const float* __restrict__ old_logits, float old_logp, float adv, float klc,
                                               float clip_param, float entropy_coeff, float scale, float* dl, double* s) {
    float sz2 = 0.f, sls = 0.f, kl = 0.f, ent = 0.f;
    float dlp_mu[DDRL_MAX_ACT], dlp_ls[DDRL_MAX_ACT], dkl_mu[DDRL_MAX_ACT], dkl_ls[DDRL_MAX_ACT];
#pragma unroll
    for (int i = 0; i < DDRL_MAX_ACT; ++i) {
        if (i < A) {
            const float mu = logits[i], ls = logits[A + i];
            const float sd = expf(ls);
            const float z = (actions[i] - mu) / sd;
            sz2 = fmaf(z, z, sz2);
            sls += ls;
            const float omu = old_logits[i], ols = old_logits[A + i];
            const float osd = expf(ols);
            const float dm = omu - mu, var = sd * sd;
            const float q = (osd * osd + dm * dm) / var;
            kl += ls - ols + 0.5f * q - 0.5f;          // KL(old || new)
            ent += ls + kHalfLog2PiE;
            dlp_mu[i] = z / sd;                         // d logp / d mean
            dlp_ls[i] = z * z - 1.f;                    // d logp / d log_std
            dkl_mu[i] = -dm / var;
            dkl_ls[i] = 1.f - q;
        }
    }
    const float lp = -0.5f * sz2 - 0.5f * kLog2Pi * (float)A - sls;
    const float ratio = expf(lp - old_logp);
    const float lo = 1.f - clip_param, hi = 1.f + clip_param;
    const float s1 = adv * ratio, s2 = adv * fminf(fmaxf(ratio, lo), hi);
    const float surr = fminf(s1, s2);
    // d surr / d logp: min() passes the gradient to s1 on ties; clip() has zero slope outside [lo, hi]
    const float dsurr = (s1 <= s2 || (ratio >= lo && ratio <= hi)) ? s1 : 0.f;
#pragma unroll
    for (int i = 0; i < DDRL_MAX_ACT; ++i) {
        if (i < A) {
            dl[i] = scale * (-dsurr * dlp_mu[i] + klc * dkl_mu[i]);
            dl[A + i] = scale * (-dsurr * dlp_ls[i] + klc * dkl_ls[i] - entropy_coeff);
        }
    }
    s[0] = -(double)surr; s[1] = kl; s[3] = ent;
}

// Value part.  Returns scale * vf_loss_coeff * d max((v-R)^2, (v_clip-R)^2)/dv; s[2] = vf, s[4..8) = R, R^2, R-v, (R-v)^2.
__device__ __forceinline__ float ppo_row_value(float v, float vf_pred, float Rt, float vf_clip_param, float vf_loss_coeff,
                                               float scale, double* s) {
    const float e1 = v - Rt, c = vf_clip_param, dvp = v - vf_pred;
    const float e2 = vf_pred + fminf(fmaxf(dvp, -c), c) - Rt;
    const float vf1 = e1 * e1, vf2 = e2 * e2;
    const float vf = fmaxf(vf1, vf2);
    const float dvf = (vf1 >= vf2) ? 2.f * e1 : ((fabsf(dvp) <= c) ? 2.f * e2 : 0.f);
    s[2] = vf;
    s[4] = Rt; s[5] = (double)Rt * Rt; s[6] = (double)Rt - v; s[7] = s[6] * s[6];
    return scale * vf_loss_coeff * dvf;
}

// out[0..2A) = logits, out[2A] = value.  Writes dl[0..2A] (d loss / d out, already scaled by inv_global_mb) and the
// row's stat contributions s[0..8) (see ddrl_ppo_train_step in ddrl_b200.h).
__device__ __forceinline__ void ppo_row_loss(const float* out, int A, const float* __restrict__ actions,
                                             const float* __restrict__ old_logits, float old_logp, float vf_pred,
                                             float adv, float Rt, float klc, const ddrl_ppo_hyper& hp, float* dl,
                                             double* s) {
    ppo_row_policy(out, A, actions, old_logits, old_logp, adv, klc, hp.clip_param, hp.entropy_coeff, hp.inv_global_mb, dl, s);
    dl[2 * A] = ppo_row_value(out[2 * A], vf_pred, Rt, hp.vf_clip_param, hp.vf_loss_coeff, hp.inv_global_mb, s);
}

}  // namespace ddrl
