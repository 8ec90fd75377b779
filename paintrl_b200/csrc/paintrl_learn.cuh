// paintrl_learn.cuh -- the PPO learner of the reference's training script on the GPU: one launch computes the loss
// gradient of a minibatch, a second sums the per-CTA partial gradients in a fixed order, a third applies Adam, and a
// fourth packs the updated parameters into the rollout policy's device weights (paintrl_policy.cuh).
//
// ppo_grad_kernel: CTA = 128 samples (one TMEM lane per sample), 512 threads, the same split as policy_act_kernel
// (four threads per sample, each owning a quarter of the sample's hidden features).  Samples are rows of a flattened
// T x B fragment read through an index list, so the learner shuffles without copying.
//
//   forward   calls policy_act_kernel's forward functions (paintrl_policy.cuh): layer 1 FP32 FFMA + tanh.approx -> BF16
//             h1 (canonical K-major), layer 2 on tcgen05.mma (BF16 x BF16 -> FP32, sixteen K steps) into TMEM columns
//             [0, 128), head in FP32 as four partial sums added in the same order -- so logits and value equal
//             paintrl_policy_act's bit for bit
//   loss      RLlib PPO (ray 0.x ppo_policy): clipped surrogate + kl_coeff KL(old || new) + vf_loss_coeff clipped
//             value loss - entropy_coeff H, averaged over the minibatch; its gradient with respect to the head outputs
//             (dout) is computed per sample in FP32
//   backward  head and layer 1 on CUDA cores; the two 128 x 256 products on tcgen05.mma, reading the tiles already in
//             shared memory through MN-major descriptors (no re-staging):
//               dh1 [128 samples x 256] = dz2 [128 x 128] . W2^T     A = dz2 K-major, B = the W2 tile MN-major
//                                                                      -> TMEM columns [0, 256) (z2 has been read)
//               dW2^T [128 x 256]       = dz2^T . h1               A = dz2 MN-major, B = the h1 tile MN-major
//                                                                      -> TMEM columns [256, 512)
//             cross-sample sums (dW1, db1, dW3, db2, db3) go through shared memory, summed in sample order
//   output    one partial gradient per CTA (every entry written, no atomics); ppo_reduce_kernel adds the partials in CTA
//             order, so a training run is reproducible bit for bit
//
// The loss stage is a template parameter (LOSS): kLossPpo above, or kLossDqn, double DQN on the head read as a dueling
// Q-network (dqn_q_values, paintrl_policy.cuh): per sample td = Q(s, a) - y with y = r + gamma (1 - done)
// Q_target(s', argmax_o Q_online(s', o)), Huber loss (delta 1) averaged over the minibatch, and dout = g ([o == a] -
// 1 / n_out) for the n_out advantage columns and g for the value column, g = clamp(td, -1, 1) / n.  The head outputs on
// s' under the online and the target parameters come from two forward-only launches of the PPO instantiation before the
// gradient launch (paintrl_dqn_grad).  Forward, backward, the cross-sample sums and the partials are the same code.
// kLossDqnPer is kLossDqn with a per-sample importance weight w (prioritized replay, paintrl_replay.cuh): g =
// (clamp(td, -1, 1) * w) * inv_n, so w = 1 gives kLossDqn's bits; the Huber statistic is weighted the same way, a fifth
// statistic is w, and td goes to td_out in minibatch order for the priority update.
// kLossPpoDiag is kLossPpo on the diagonal-Gaussian head of A = n_out / 2 dimensions (RLlib's DiagGaussian; mean in
// column o, log sigma in column A + o, actions float64 [rows][A]): logp from pol_diag_logp (the act kernel's own
// function), KL(old || new) = sum (log sigma - log sigma_old + (sigma_old^2 + (mu_old - mu)^2) / (2 sigma^2) - 1/2),
// H = sum (log sigma + log(2 pi e) / 2), and per dimension, with q = (sigma_old^2 + (mu - mu_old)^2) / sigma^2,
//   dout[mu]        = s (g_logp u / sigma + kl_coeff (mu - mu_old) / sigma^2)
//   dout[log sigma] = s (g_logp (u^2 - 1) + kl_coeff (1 - q) - ent_coeff)
// The clipped surrogate, the value loss and the six statistics are kLossPpo's.
//
// Parameters arrive flat, in pol_num_params' layout (paintrl_policy.cuh).
#pragma once
#include "paintrl_policy.cuh"

namespace paintrl {

constexpr int kLrnStats = 6;                   // policy loss, value loss, KL, entropy, clip fraction, mean ratio
constexpr int kDqnStats = 4;                   // Huber loss, |td|, Q(s, a), target y
constexpr int kDqnPerStats = 5;                // weighted Huber loss, |td|, Q(s, a), target y, importance weight
constexpr int kLrnStatStride = 8;
constexpr int kLossPpo = 0, kLossDqn = 1, kLossDqnPer = 2, kLossPpoDiag = 3;

struct PpoGradArgs {
    int obs_dim, n_out, discrete, n, nparams;
    int forward_only;                          // 1: write the forward outputs to fwd_out and stop (tests)
    const float *params;                       // flat FP32 parameters
    const int *idx;                            // [n] rows of the flattened fragment
    const double *obs;                         // [rows][obs_dim]
    const void *actions;                       // int64 [rows] (discrete) | float64 [rows][n_out] | [rows][n_out / 2] (kLossPpoDiag)
    const float *logp_old, *value_old, *logits_old, *adv, *vtarg;   // [rows], logits_old [rows][n_out + 1]
    float clip, vf_clip, vf_coeff, ent_coeff, kl_coeff, inv_n;
    float *partial;                            // [gridDim.x][nparams]
    float *partial_stats;                      // [gridDim.x][kLrnStatStride]
    float *fwd_out;                            // forward_only: [n][n_out + 1]
    // kLossDqn: reward float32 [rows], done uint8 [rows]; the head outputs on s' under the online and the target
    // parameters, [n][n_out + 1] in minibatch order
    const float *reward;
    const unsigned char *done;
    const float *next_online, *next_target;
    float gamma;
    // kLossDqnPer: importance weights float32 [n] in, TD errors float32 [n] out, both in minibatch order
    const float *weight;
    float *td_out;
};

// dynamic shared memory.  R0 (160 KB) is reused by phase:
//   forward / backward MMAs: h1 (64 KB, A of layer 2, B of dW2) | W2 (64 KB) | dz2 (32 KB; partial heads before it)
//   after the backward MMAs: h2 and dz2 in FP32 [128][129], then dz1 in FP32 [128][257] and x [128][32] at 144 KB
constexpr int kLrnR0 = 163840;
constexpr int kLrnPadH2 = kPolH2 + 1, kLrnPadH1 = kPolH1 + 1;
constexpr size_t kLrnSmemBytes = (size_t)kLrnR0 +
                                 sizeof(float) * (kPolMaxObs * kPolH1 + kPolH1 + kPolH2 + kPolH2 * kPolMaxOut + kPolMaxOut +
                                                  kPolRows * kPolMaxOut + kPolRows * kLrnStatStride) + 64;

// MO / MX: the compile-time caps of policy_act_kernel (observation and output register arrays)
template <int MO, int MX, int LOSS = kLossPpo>
__global__ void __launch_bounds__(kPolThreads, 1) ppo_grad_kernel(PpoGradArgs a) {
    extern __shared__ __align__(1024) unsigned char lrn_smem[];
    unsigned char *sA = lrn_smem;
    unsigned char *sB = lrn_smem + kPolRows * kPolH1 * 2;
    unsigned char *sD = sB + kPolH2 * kPolH1 * 2;
    float *spart = reinterpret_cast<float *>(sD);                     // [kPolSplit - 1][kPolRows][kPolMaxOut]
    float *sH2 = reinterpret_cast<float *>(lrn_smem);                 // [128][kLrnPadH2]
    float *sDZ2 = sH2 + kPolRows * kLrnPadH2;
    float *sDZ1 = reinterpret_cast<float *>(lrn_smem);                // [128][kLrnPadH1]
    float *sX = reinterpret_cast<float *>(lrn_smem + 147456);         // [128][kPolMaxObs]
    const PolTables st(reinterpret_cast<float *>(lrn_smem + kLrnR0));
    float *sdout = reinterpret_cast<float *>(st.end());               // [128][kPolMaxOut] dLoss / d(logits | value)
    float *sstat = sdout + kPolRows * kPolMaxOut;                     // [128][kLrnStatStride]
    unsigned long long *bar_mma = reinterpret_cast<unsigned long long *>(sstat + kPolRows * kLrnStatStride);
    unsigned *tmem_slot = reinterpret_cast<unsigned *>(bar_mma + 1);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int row = tid & (kPolRows - 1), part = tid / kPolRows;
    const int j = blockIdx.x * kPolRows + row;
    const bool valid = j < a.n;
    const int src = valid ? __ldg(&a.idx[j]) : 0;
    const int nout1 = a.n_out + 1;
    const int off_b1 = a.obs_dim * kPolH1, off_w2 = off_b1 + kPolH1, off_b2 = off_w2 + kPolH1 * kPolH2, off_w3 = off_b2 + kPolH2,
              off_b3 = off_w3 + kPolH2 * nout1;
    const float *P = a.params;

    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar_mma)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {   // TMEM: z2 / dh1 in columns [0, 256), dW2^T in [256, 512)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"((unsigned)__cvta_generic_to_shared(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // W2 [256 in][128 out] -> BF16 [n][k] in the canonical K-major layout (the bytes paintrl_policy_create packs):
    // one thread per 8 consecutive k of one n, one 16-byte store
    for (int g = tid; g < kPolH1 / 8 * kPolH2; g += kPolThreads) {
        const int n = g % kPolH2, kg = g / kPolH2;
        float f[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) f[q] = __ldg(&P[off_w2 + (kg * 8 + q) * kPolH2 + n]);
        *reinterpret_cast<uint4 *>(sB + pol_w2_byte(kg * 8, n)) = pol_pack8(f);
    }
    pol_stage_tables(st, P, P, P, P, P, a.obs_dim, nout1, tid, off_b1, off_b2, off_w3, off_b3);
    float x[MO];
    pol_load_x<MO>(x, a.obs, src, a.obs_dim, valid);
    __syncthreads();

    pol_layer1<MO>(sA, st, x, a.obs_dim, row, part);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = *tmem_slot;
    const unsigned a0 = (unsigned)__cvta_generic_to_shared(sA), b0 = (unsigned)__cvta_generic_to_shared(sB),
                   d0 = (unsigned)__cvta_generic_to_shared(sD);

    if (tid == 0) pol_layer2(tmem, a0, b0, bar_mma);   // z2 [128 x 128] = h1 W2
    pol_wait(bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    const unsigned lane_base = tmem + ((unsigned)((warp & 3) * 32) << 16);
    float out[MX];
    pol_head_partial<MX>(out, lane_base, st, nout1, part);
    pol_head_store<MX>(spart, out, row, part);
    __syncthreads();

    // ---- loss and its gradient with respect to the head outputs (one thread per sample)
    if (part == 0) {
        pol_head_combine<MX>(out, spart, row);
        float dout[MX], st[kLrnStats];
#pragma unroll
        for (int o = 0; o < MX; ++o) dout[o] = 0.f;
#pragma unroll
        for (int s = 0; s < kLrnStats; ++s) st[s] = 0.f;
        if (valid && a.forward_only) {
#pragma unroll
            for (int o = 0; o < MX; ++o) if (o < nout1) a.fwd_out[(size_t)j * nout1 + o] = out[o];
        } else if (valid && (LOSS == kLossDqn || LOSS == kLossDqnPer)) {
            const int act = (int)reinterpret_cast<const long long *>(a.actions)[src];
            float q[MX], nx[MX], qn[MX];
            dqn_q_values<MX>(out, a.n_out, q);
#pragma unroll
            for (int o = 0; o < MX; ++o) nx[o] = o < nout1 ? __ldg(&a.next_online[(size_t)j * nout1 + o]) : 0.f;
            const int an = dqn_q_values<MX>(nx, a.n_out, qn);
#pragma unroll
            for (int o = 0; o < MX; ++o) nx[o] = o < nout1 ? __ldg(&a.next_target[(size_t)j * nout1 + o]) : 0.f;
            dqn_q_values<MX>(nx, a.n_out, qn);
            float qsa = 0.f, qnext = 0.f;
#pragma unroll
            for (int o = 0; o < MX; ++o) {
                if (o == act) qsa = q[o];
                if (o == an) qnext = qn[o];
            }
            const float nd = a.done[src] ? 0.f : 1.f;
            const float y = __ldg(&a.reward[src]) + a.gamma * nd * qnext;
            const float td = qsa - y, atd = fabsf(td);
            float c = fminf(fmaxf(td, -1.f), 1.f);
            float w = 1.f;
            if (LOSS == kLossDqnPer) {
                w = __ldg(&a.weight[j]);
                c = c * w;
                a.td_out[j] = td;
            }
            const float g = c * a.inv_n;
            const float inv_nout = 1.f / (float)a.n_out;
#pragma unroll
            for (int o = 0; o < MX; ++o) {
                if (o < a.n_out) dout[o] = g * ((o == act ? 1.f : 0.f) - inv_nout);
                else if (o == a.n_out) dout[o] = g;
            }
            st[0] = atd <= 1.f ? 0.5f * td * td : atd - 0.5f;
            st[1] = atd;
            st[2] = qsa;
            st[3] = y;
            if (LOSS == kLossDqnPer) {
                st[0] = st[0] * w;
                st[4] = w;
            }
        } else if (valid) {
            float v = 0.f;
#pragma unroll
            for (int o = 0; o < MX; ++o) if (o == a.n_out) v = out[o];
            float old[MX];
#pragma unroll
            for (int o = 0; o < MX; ++o) old[o] = o < a.n_out ? __ldg(&a.logits_old[(size_t)src * nout1 + o]) : 0.f;
            float logp = 0.f, kl = 0.f, ent = 0.f;
            float lse = 0.f, lseo = 0.f;
            int act = 0;
            // kLossPpoDiag: the row's head in its sdout slots (mu at [o], log sigma at [A + o]), its FP32 actions in ad
            float *head = sdout + row * kPolMaxOut;
            const int adim = a.n_out >> 1;
            const float *lgo = a.logits_old + (size_t)src * nout1;
            float ad[MX / 2];
            if (LOSS == kLossPpoDiag) {
#pragma unroll
                for (int o = 0; o < MX; ++o) if (o < nout1) head[o] = out[o];
                const double *ac = reinterpret_cast<const double *>(a.actions) + (size_t)src * adim;
#pragma unroll
                for (int o = 0; o < MX / 2; ++o) ad[o] = o < adim ? (float)ac[o] : 0.f;
                logp = pol_diag_logp<MX>(head, ad, adim);
#pragma unroll
                for (int o = 0; o < MX / 2; ++o) {
                    if (o < adim) {
                        const float mu = head[o], ls = head[adim + o], muo = __ldg(&lgo[o]), lso = __ldg(&lgo[adim + o]);
                        const float sig = pol_diag_sigma(ls), sigo = pol_diag_sigma(lso);
                        const float d = mu - muo;
                        const float q = (sigo * sigo + d * d) / (sig * sig);
                        kl += ((ls - lso) + 0.5f * q) - 0.5f;
                        ent += ls + 1.4189385332046727f;             // log sigma + log(2 pi e) / 2
                    }
                }
            } else if (a.discrete) {
                // log-softmax exactly as policy_act_kernel computes the sampled action's log-probability
                float mx = -INFINITY, mo = -INFINITY;
#pragma unroll
                for (int o = 0; o < MX; ++o) if (o < a.n_out) { mx = fmaxf(mx, out[o]); mo = fmaxf(mo, old[o]); }
                float se = 0.f, so = 0.f;
#pragma unroll
                for (int o = 0; o < MX; ++o) if (o < a.n_out) { se += __expf(out[o] - mx); so += __expf(old[o] - mo); }
                lse = mx + __logf(se);
                lseo = mo + __logf(so);
                act = (int)reinterpret_cast<const long long *>(a.actions)[src];
#pragma unroll
                for (int o = 0; o < MX; ++o) {
                    if (o < a.n_out) {
                        if (o == act) logp = out[o] - lse;
                        const float lp = out[o] - lse, lpo = old[o] - lseo;
                        const float p = expf(lp), po = expf(lpo);
                        kl += po * (lpo - lp);
                        ent -= p * lp;
                    }
                }
            } else {
                const double *ac = reinterpret_cast<const double *>(a.actions) + (size_t)src * a.n_out;
#pragma unroll
                for (int o = 0; o < MX; ++o) {
                    if (o < a.n_out) {
                        const float mu = pol_tanh(out[o]), muo = pol_tanh(old[o]);
                        const float d = (float)ac[o] - mu;
                        logp += -0.5f * d * d - 0.9189385332046727f;
                        kl += 0.5f * (muo - mu) * (muo - mu);
                    }
                }
                ent = (float)a.n_out * 1.4189385332046727f;       // N(mu, I): constant
            }
            const float A = __ldg(&a.adv[src]), R = __ldg(&a.vtarg[src]), vold = __ldg(&a.value_old[src]);
            const float r = expf(logp - __ldg(&a.logp_old[src]));
            const float rc = fminf(fmaxf(r, 1.f - a.clip), 1.f + a.clip);
            const float s1 = A * r, s2 = A * rc;
            const float g_logp = s1 <= s2 ? -A * r : 0.f;        // d(-min(s1, s2)) / d logp
            const float vf1 = (v - R) * (v - R);
            const float dv = v - vold, dvc = fminf(fmaxf(dv, -a.vf_clip), a.vf_clip);
            const float vcl = vold + dvc;
            const float vf2 = (vcl - R) * (vcl - R);
            const float g_v = vf1 >= vf2 ? 2.f * (v - R) : (fabsf(dv) <= a.vf_clip ? 2.f * (vcl - R) : 0.f);
            const float s = a.inv_n;
            if (LOSS == kLossPpoDiag) {
#pragma unroll
                for (int o = 0; o < MX / 2; ++o) {
                    if (o < adim) {
                        const float mu = head[o], ls = head[adim + o], muo = __ldg(&lgo[o]), lso = __ldg(&lgo[adim + o]);
                        const float sig = pol_diag_sigma(ls), sigo = pol_diag_sigma(lso);
                        const float u = __fdiv_rn(__fsub_rn(ad[o], mu), sig);
                        const float d = mu - muo;
                        const float is2 = 1.f / (sig * sig);
                        const float q = (sigo * sigo + d * d) * is2;
                        head[o] = s * (g_logp * (u / sig) + a.kl_coeff * (d * is2));
                        head[adim + o] = s * ((g_logp * (u * u - 1.f) + a.kl_coeff * (1.f - q)) - a.ent_coeff);
                    }
                }
#pragma unroll
                for (int o = 0; o < MX; ++o) {
                    if (o < a.n_out) dout[o] = head[o];
                    else if (o == a.n_out) dout[o] = s * a.vf_coeff * g_v;
                }
            } else
#pragma unroll
            for (int o = 0; o < MX; ++o) {
                if (o < a.n_out) {
                    if (a.discrete) {
                        const float lp = out[o] - lse;
                        const float p = expf(lp), po = expf(old[o] - lseo);
                        const float onehot = o == act ? 1.f : 0.f;
                        dout[o] = s * (g_logp * (onehot - p) + a.kl_coeff * (p - po) + a.ent_coeff * p * (lp + ent));
                    } else {
                        const float mu = pol_tanh(out[o]), muo = pol_tanh(old[o]);
                        const double *ac = reinterpret_cast<const double *>(a.actions) + (size_t)src * a.n_out;
                        dout[o] = s * (g_logp * ((float)ac[o] - mu) + a.kl_coeff * (mu - muo)) * (1.f - mu * mu);
                    }
                } else if (o == a.n_out) {
                    dout[o] = s * a.vf_coeff * g_v;
                }
            }
            st[0] = -fminf(s1, s2);
            st[1] = fmaxf(vf1, vf2);
            st[2] = kl;
            st[3] = ent;
            st[4] = fabsf(r - 1.f) > a.clip ? 1.f : 0.f;
            st[5] = r;
        }
#pragma unroll
        for (int o = 0; o < MX; ++o) sdout[row * kPolMaxOut + o] = dout[o];
#pragma unroll
        for (int o = MX; o < kPolMaxOut; ++o) sdout[row * kPolMaxOut + o] = 0.f;
#pragma unroll
        for (int q = 0; q < kLrnStats; ++q) sstat[row * kLrnStatStride + q] = st[q];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    if (!a.forward_only) {
        // ---- head backward: dz2 = (dout W3^T) * (1 - h2^2) for this thread's quarter of the row; BF16 copy into the
        // K-major A layout [sample][feature]; h2 and dz2 stay in registers until the tensor core has read the tiles
        float h2v[kPolH2 / kPolSplit], dz2v[kPolH2 / kPolSplit];
        {
            float dr[MX];
#pragma unroll
            for (int o = 0; o < MX; ++o) dr[o] = sdout[row * kPolMaxOut + o];
            unsigned char *rowbase = sD + (row >> 3) * 128 + (row & 7) * 16;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c0 = part * (kPolH2 / kPolSplit) + h * 16;
                float z[16];
                pol_ld16(lane_base + (unsigned)c0, z);
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float h2 = pol_tanh(z[c] + st.b2[c0 + c]);
                    const float *wr = st.w3 + (c0 + c) * nout1;
                    float dh = 0.f;
#pragma unroll
                    for (int o = 0; o < MX; ++o)
                        if (o < nout1) dh = fmaf(dr[o], wr[o], dh);
                    h2v[h * 16 + c] = h2;
                    dz2v[h * 16 + c] = dh * (1.f - h2 * h2);
                }
                *reinterpret_cast<uint4 *>(rowbase + (c0 >> 3) * (kPolRows / 8) * 128) = pol_pack8(&dz2v[h * 16]);
                *reinterpret_cast<uint4 *>(rowbase + ((c0 >> 3) + 1) * (kPolRows / 8) * 128) = pol_pack8(&dz2v[h * 16 + 8]);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tid == 0) {
            // dh1 [128 x 256] = dz2 W2^T: A = dz2 [sample][feature] K-major; B = the W2 tile read as [k][n], n the
            // reduction: MN-major (8 consecutive k per 16-byte row), MN groups of 8 k every 2 KB (SBO), K groups of 8 n
            // every 128 B (LBO)
            const unsigned id1 = kPolIdescBase | (1u << 16) | ((unsigned)(kPolH1 >> 3) << 17);
#pragma unroll 1
            for (int ks = 0; ks < kPolH2 / 16; ++ks)
                pol_mma(tmem, pol_smem_desc(d0 + ks * 2 * (kPolRows / 8) * 128, (kPolRows / 8) * 128, 128),
                        pol_smem_desc(b0 + ks * 2 * 128, 128, (kPolH2 / 8) * 128), id1, ks > 0 ? 1u : 0u);
            // dW2^T [128 n x 256 k] = dz2^T h1, the reduction over samples: both tiles MN-major (8 consecutive features
            // per 16-byte row), feature groups every 2 KB (SBO), sample groups every 128 B (LBO)
            const unsigned id2 = kPolIdescBase | (1u << 15) | (1u << 16) | ((unsigned)(kPolH1 >> 3) << 17);
#pragma unroll 1
            for (int ks = 0; ks < kPolRows / 16; ++ks)
                pol_mma(tmem + 256, pol_smem_desc(d0 + ks * 2 * 128, 128, (kPolRows / 8) * 128),
                        pol_smem_desc(a0 + ks * 2 * 128, 128, (kPolRows / 8) * 128), id2, ks > 0 ? 1u : 0u);
            pol_commit(bar_mma);
        }
        pol_wait(bar_mma, 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

        // ---- dW3, db2, db3 and the statistics: h2 / dz2 through shared memory, summed in sample order
#pragma unroll
        for (int c = 0; c < kPolH2 / kPolSplit; ++c) {
            sH2[row * kLrnPadH2 + part * (kPolH2 / kPolSplit) + c] = h2v[c];
            sDZ2[row * kLrnPadH2 + part * (kPolH2 / kPolSplit) + c] = dz2v[c];
        }
        __syncthreads();
        float *pg = a.partial + (size_t)blockIdx.x * a.nparams;
        {
            const int c = tid & (kPolH2 - 1), q = tid >> 7;
            float acc[kPolMaxOut / kPolSplit];
#pragma unroll
            for (int u = 0; u < kPolMaxOut / kPolSplit; ++u) acc[u] = 0.f;
            float accb = 0.f;
#pragma unroll 4
            for (int r = 0; r < kPolRows; ++r) {
                const float h2 = sH2[r * kLrnPadH2 + c];
#pragma unroll
                for (int u = 0; u < kPolMaxOut / kPolSplit; ++u) acc[u] = fmaf(h2, sdout[r * kPolMaxOut + q + kPolSplit * u], acc[u]);
                if (q == 0) accb += sDZ2[r * kLrnPadH2 + c];
                else if (q == 1 && c < nout1) accb += sdout[r * kPolMaxOut + c];
                else if (q == 2 && c < kLrnStats) accb += sstat[r * kLrnStatStride + c];
            }
#pragma unroll
            for (int u = 0; u < kPolMaxOut / kPolSplit; ++u)
                if (q + kPolSplit * u < nout1) pg[off_w3 + c * nout1 + q + kPolSplit * u] = acc[u];
            if (q == 0) pg[off_b2 + c] = accb;
            else if (q == 1 && c < nout1) pg[off_b3 + c] = accb;
            else if (q == 2 && c < kLrnStats) a.partial_stats[(size_t)blockIdx.x * kLrnStatStride + c] = accb;
        }
        // dW2: TMEM lane = n, column 256 + k
        {
            const int n = (warp & 3) * 32 + (tid & 31);
#pragma unroll 1
            for (int k0 = part * (kPolH1 / kPolSplit); k0 < (part + 1) * (kPolH1 / kPolSplit); k0 += 16) {
                float g[16];
                pol_ld16(lane_base + 256u + (unsigned)k0, g);
#pragma unroll
                for (int c = 0; c < 16; ++c) pg[off_w2 + (k0 + c) * kPolH2 + n] = g[c];
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

        // ---- layer 1 backward: dz1 = dh1 * (1 - h1^2), h1 recomputed in FP32 with the forward's arithmetic
        pol_load_x<MO>(x, a.obs, src, a.obs_dim, valid);
        if (part == 0) {
#pragma unroll
            for (int i = 0; i < MO; ++i) sX[row * kPolMaxObs + i] = x[i];
        }
#pragma unroll 1
        for (int k0 = part * (kPolH1 / kPolSplit); k0 < (part + 1) * (kPolH1 / kPolSplit); k0 += 16) {
            float g[16];
            pol_ld16(lane_base + (unsigned)k0, g);
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                float h = st.b1[k0 + c];
#pragma unroll
                for (int i = 0; i < MO; ++i)
                    if (i < a.obs_dim) h = fmaf(x[i], st.w1[i * kPolH1 + k0 + c], h);
                h = pol_tanh(h);
                sDZ1[row * kLrnPadH1 + k0 + c] = valid ? g[c] * (1.f - h * h) : 0.f;
            }
        }
        __syncthreads();
        {
            const int k = tid & (kPolH1 - 1), half = tid >> 8;
            float acc[(MO + 1) / 2];
#pragma unroll
            for (int u = 0; u < (MO + 1) / 2; ++u) acc[u] = 0.f;
            float accb = 0.f;
#pragma unroll 2
            for (int r = 0; r < kPolRows; ++r) {
                const float d = sDZ1[r * kLrnPadH1 + k];
#pragma unroll
                for (int u = 0; u < (MO + 1) / 2; ++u)
                    if (half + 2 * u < a.obs_dim) acc[u] = fmaf(sX[r * kPolMaxObs + half + 2 * u], d, acc[u]);
                accb += d;
            }
#pragma unroll
            for (int u = 0; u < (MO + 1) / 2; ++u)
                if (half + 2 * u < a.obs_dim) pg[(half + 2 * u) * kPolH1 + k] = acc[u];
            if (half == 0) pg[off_b1 + k] = accb;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// grad[p] = sum over CTAs, in CTA order, of the partial gradients; stats[s] = the minibatch means of the first nstats
__global__ void ppo_reduce_kernel(const float *partial, int nparts, int nparams, float *grad, const float *partial_stats, float inv_n,
                                  float *stats, int nstats) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < nparams) {
        float s = 0.f;
        for (int c = 0; c < nparts; ++c) s += partial[(size_t)c * nparams + p];
        grad[p] = s;
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < nstats) {
        float s = 0.f;
        for (int c = 0; c < nparts; ++c) s += partial_stats[c * kLrnStatStride + threadIdx.x];
        stats[threadIdx.x] = s * inv_n;
    }
}

// Global-norm gradient clipping (torch.nn.utils.clip_grad_norm_'s rule): norm = sqrt(sum g^2), and when norm > max_norm
// every entry is multiplied by max_norm / (norm + 1e-6).  One CTA: each thread sums a fixed stride of squares, then a
// shared-memory tree in a fixed order -- no float atomics, the same norm on every run.  Under max_norm nothing is written.
constexpr int kClipThreads = 1024;
__global__ void __launch_bounds__(kClipThreads) clip_grad_norm_kernel(float *grad, int n, float max_norm, float *norm_out) {
    __shared__ float red[kClipThreads];
    const int tid = threadIdx.x;
    float s = 0.f;
    for (int i = tid; i < n; i += kClipThreads) {
        const float g = grad[i];
        s += g * g;
    }
    red[tid] = s;
    __syncthreads();
#pragma unroll 1
    for (int w = kClipThreads / 2; w > 0; w >>= 1) {
        if (tid < w) red[tid] += red[tid + w];
        __syncthreads();
    }
    const float norm = sqrtf(red[0]);
    if (tid == 0) norm_out[0] = norm;
    if (!(norm > max_norm)) return;
    const float scale = max_norm / (norm + 1e-6f);
    for (int i = tid; i < n; i += kClipThreads) grad[i] *= scale;
}

// Adam with bias correction, torch.optim.Adam's arithmetic: m <- lerp(m, g, 1 - beta1), v <- beta2 v + (1 - beta2) g^2,
// p <- p - step_size m / (sqrt(v) / sqrt(1 - beta2^t) + eps), step_size = lr / (1 - beta1^t)
__global__ void adam_kernel(float *params, const float *grad, float *m, float *v, int n, float step_size, float beta1, float beta2,
                            float eps, float bc2_sqrt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float g = grad[i];
    const float mi = m[i] + (1.f - beta1) * (g - m[i]);
    const float vi = v[i] * beta2 + (1.f - beta2) * (g * g);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    params[i] = params[i] + (-step_size) * (mi / denom);
}

// flat FP32 parameters -> the policy engine's device weights (paintrl_policy_create's host packing, on a stream)
__global__ void policy_pack_kernel(const float *params, int obs_dim, int n_out, float *w1, float *b1, __nv_bfloat16 *w2p, float *b2,
                                   float *w3, float *b3) {
    const int nout1 = n_out + 1;
    const int off_b1 = obs_dim * kPolH1, off_w2 = off_b1 + kPolH1, off_b2 = off_w2 + kPolH1 * kPolH2, off_w3 = off_b2 + kPolH2,
              off_b3 = off_w3 + kPolH2 * nout1, total = off_b3 + nout1;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < total; p += gridDim.x * blockDim.x) {
        const float f = params[p];
        if (p < off_b1) w1[p] = f;
        else if (p < off_w2) b1[p - off_b1] = f;
        else if (p < off_b2) {
            const int e = p - off_w2;
            w2p[pol_w2_byte(e / kPolH2, e % kPolH2) / 2] = __float2bfloat16_rn(f);
        } else if (p < off_w3) b2[p - off_b2] = f;
        else if (p < off_b3) w3[p - off_w3] = f;
        else b3[p - off_b3] = f;
    }
}

}  // namespace paintrl
