// paintrl_policy.cuh -- the rollout policy of the reference's PPO script as ONE kernel per step.
//
// paint_ppo.py:179-183 trains a fully connected policy obs -> 256 -> 128 -> {logits | mean, value} (tanh, value branch
// sharing the hidden layers); its rollout workers evaluate it once per environment step and sample an action.  Here
// that is one launch for the whole batch, observations in, actions straight into the rollout fragment out:
//
//   CTA = 128 environments (one per TMEM lane), 512 threads: four threads share a row -- each computes a quarter of the
//         row's layer-1 features and reduces a quarter of its layer-2 columns (warps w, w + 4, w + 8, w + 12 own TMEM
//         lanes 32 (w % 4) ...), so the SM runs sixteen warps instead of four
//   layer 1  (obs_dim x 256, obs_dim <= 32): FP32 FFMA per thread, weights broadcast from shared memory, tanh, the
//            activations written as BF16 into shared memory in the tensor core's canonical K-major layout
//   layer 2  (256 x 128): sixteen tcgen05.mma (M 128, N 128, K 16, BF16 x BF16 -> FP32) issued by one thread, A = the
//            activations, B = the weights (pre-packed by the host in the same canonical layout, brought in with one
//            cp.async.bulk), accumulator in TMEM (128 lanes x 128 columns)
//   epilogue tcgen05.ld of each thread's row, + bias, tanh, the 128 x (n_out + 1) head in FP32 FFMA
//   sampling discrete: Gumbel-max over the logits; continuous: tanh(mean) + unit Gaussian noise, or mean + sigma x unit
//            noise with a learned log-std (the DIAG instantiations); log-probability and value; counter-based random
//            numbers (per-environment counters in device memory, so a captured CUDA graph draws fresh noise on every
//            replay)
//
// Shared-memory operand layout (no swizzle, K-major; cute::UMMA "INTERLEAVE"): 8 x 8 BF16 core matrices of 128
// contiguous bytes (row r at +16 r); core (mi, kj) of an [rows x 256] operand sits at kj * (rows / 8) * 128 + mi * 128,
// i.e. stride-byte-offset (next 8 rows) = 128 B, leading-byte-offset (next 8 columns of K) = rows * 16 B.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace paintrl {

constexpr int kPolH1 = 256, kPolH2 = 128;      // hidden sizes (paint_ppo.py:180 fcnet_hiddens)
constexpr int kPolRows = 128;                  // environments per CTA = MMA M
constexpr int kPolMaxObs = 32, kPolMaxOut = 16;
constexpr int kPolSplit = 4;                   // threads per environment row
constexpr int kPolThreads = kPolRows * kPolSplit;

struct PolicyParams {
    int obs_dim, n_out, discrete;
    const float *w1, *b1;                      // [obs_dim][256], [256]
    const __nv_bfloat16 *w2_packed;            // [128 x 256] in the canonical layout above (64 KB)
    const float *b2;                           // [128]
    const float *w3, *b3;                      // [128][n_out + 1] (last column: value), [n_out + 1]
    unsigned long long seed;
    unsigned *counters;                        // [capacity] per-environment draw counters
};

struct PolicyIO {
    const double *obs;        // [B][obs_dim]
    int batch;
    long long *act_discrete;  // [B]               (discrete)
    double *act_continuous;   // [B][n_out]        (continuous; [B][n_out / 2] for DIAG)
    float *logp, *value;      // [B]
    float *logits;            // [B][n_out + 1] or nullptr (tests)
    int sample;               // 0: value / logits only (bootstrap), 1: sample actions
    const float *epsilon;     // [1] exploration probability of the epsilon-greedy instantiations (EPS), device memory
};

__device__ __forceinline__ unsigned long long pol_mix(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// uniform in (0, 1): 24 random bits, never 0 or 1
__device__ __forceinline__ float pol_uniform(unsigned long long seed, unsigned env, unsigned ctr, unsigned k) {
    const unsigned long long h = pol_mix(seed ^ pol_mix(((unsigned long long)env << 32) | ctr) ^ ((unsigned long long)k * 0xD6E8FEB86659FD93ull));
    return ((float)(unsigned)(h >> 40) + 0.5f) * (1.0f / 16777216.0f);
}

__device__ __forceinline__ unsigned long long pol_smem_desc(unsigned smem_byte_addr, unsigned lbo_bytes, unsigned sbo_bytes) {
    // cute::UMMA::SmemDescriptor: start address [0,14), leading byte offset [16,30), stride byte offset [32,46) (all >> 4),
    // version [46,48) = 1 on sm_100, layout type [61,64) = 0 (no swizzle)
    return (unsigned long long)((smem_byte_addr & 0x3FFFFu) >> 4) | ((unsigned long long)(lbo_bytes >> 4) << 16) |
           ((unsigned long long)(sbo_bytes >> 4) << 32) | (1ull << 46);
}

// Flat parameter layout (PaintrlPolicyConfig's tensors, row-major), the learner's and policy_pack_kernel's input:
// w1 [obs][256] | b1 [256] | w2 [256][128] | b2 [128] | w3 [128][n_out + 1] | b3 [n_out + 1]
__host__ __device__ constexpr int pol_num_params(int obs_dim, int n_out) {
    return obs_dim * kPolH1 + kPolH1 + kPolH1 * kPolH2 + kPolH2 + kPolH2 * (n_out + 1) + (n_out + 1);
}

// Byte offset of W2 element (k = input feature, n = output feature) in the canonical K-major B tile [n][k] above.  The
// host packing (paintrl_policy_create), policy_pack_kernel and the learner's W2 staging all place W2 through this.
__host__ __device__ constexpr size_t pol_w2_byte(int k, int n) {
    return (size_t)(k / 8) * (kPolH2 / 8) * 128 + (size_t)(n / 8) * 128 + (size_t)(n % 8) * 16 + (size_t)(k % 8) * 2;
}

__device__ __forceinline__ float pol_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- the forward pass, called step for step by policy_act_kernel and ppo_grad_kernel (paintrl_learn.cuh), so that the
// learner's head outputs equal the act kernel's bit for bit.  The two kernels lay out shared memory differently; these
// functions take the shared-memory pointers.

// the FP32 tables in shared memory: w1 [obs_dim][256] | b1 [256] | b2 [128] | w3 [128][n_out + 1] | b3 [n_out + 1]
struct PolTables {
    float *w1, *b1, *b2, *w3, *b3;
    __device__ explicit PolTables(float *base)
        : w1(base), b1(w1 + kPolMaxObs * kPolH1), b2(b1 + kPolH1), w3(b2 + kPolH2), b3(w3 + kPolH2 * kPolMaxOut) {}
    __device__ void *end() const { return b3 + kPolMaxOut; }
};

// Each source table is read at its pointer plus an element offset: the act kernel passes the engine's five arrays, the
// learner its flat parameter vector five times with the layout's offsets.  obs_dim here and obs / obs_dim in
// pol_load_x are references to the kernels' launch-parameter fields; passed so, both kernels compile to the code they
// compiled to when each had its own copy of these loops.
__device__ __forceinline__ void pol_stage_tables(const PolTables &s, const float *w1, const float *b1, const float *b2, const float *w3,
                                                 const float *b3, const int &obs_dim, int nout1, int tid, int o_b1 = 0, int o_b2 = 0,
                                                 int o_w3 = 0, int o_b3 = 0) {
    for (int i = tid; i < obs_dim * kPolH1; i += kPolThreads) s.w1[i] = __ldg(&w1[i]);
    for (int i = tid; i < kPolH1; i += kPolThreads) s.b1[i] = __ldg(&b1[o_b1 + i]);
    for (int i = tid; i < kPolH2; i += kPolThreads) s.b2[i] = __ldg(&b2[o_b2 + i]);
    for (int i = tid; i < kPolH2 * nout1; i += kPolThreads) s.w3[i] = __ldg(&w3[o_w3 + i]);
    if (tid < nout1) s.b3[tid] = __ldg(&b3[o_b3 + tid]);
}

// observation row `src` as FP32, zero past obs_dim and for rows past the batch
template <int MO>
__device__ __forceinline__ void pol_load_x(float (&x)[MO], const double *const &obs, int src, const int &obs_dim, bool valid) {
#pragma unroll
    for (int i = 0; i < MO; ++i) x[i] = (i < obs_dim && valid) ? (float)obs[(size_t)src * obs_dim + i] : 0.f;
}

__device__ __forceinline__ uint4 pol_pack8(const float *f) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(f[0], f[1]), p1 = __floats2bfloat162_rn(f[2], f[3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(f[4], f[5]), p3 = __floats2bfloat162_rn(f[6], f[7]);
    uint4 v;
    v.x = *reinterpret_cast<unsigned *>(&p0); v.y = *reinterpret_cast<unsigned *>(&p1);
    v.z = *reinterpret_cast<unsigned *>(&p2); v.w = *reinterpret_cast<unsigned *>(&p3);
    return v;
}

// layer 1: h1 = tanh(x W1 + b1) -> BF16 into the A tile sA (canonical layout); this thread's quarter of the row's features
template <int MO>
__device__ __forceinline__ void pol_layer1(unsigned char *sA, const PolTables &s, const float (&x)[MO], int obs_dim, int row, int part) {
    unsigned char *rowbase = sA + (row >> 3) * 128 + (row & 7) * 16;
    for (int kj = part * (kPolH1 / 8 / kPolSplit); kj < (part + 1) * (kPolH1 / 8 / kPolSplit); ++kj) {
        float h[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) h[c] = s.b1[kj * 8 + c];
#pragma unroll
        for (int i = 0; i < MO; ++i) {
            if (i < obs_dim) {
                const float xi = x[i];
                const float *wr = s.w1 + i * kPolH1 + kj * 8;
#pragma unroll
                for (int c = 0; c < 8; ++c) h[c] = fmaf(xi, wr[c], h[c]);
            }
        }
        // tanh inside the conversions: written so, this compiles to the act kernel's earlier instruction sequence
        __nv_bfloat162 p0 = __floats2bfloat162_rn(pol_tanh(h[0]), pol_tanh(h[1]));
        __nv_bfloat162 p1 = __floats2bfloat162_rn(pol_tanh(h[2]), pol_tanh(h[3]));
        __nv_bfloat162 p2 = __floats2bfloat162_rn(pol_tanh(h[4]), pol_tanh(h[5]));
        __nv_bfloat162 p3 = __floats2bfloat162_rn(pol_tanh(h[6]), pol_tanh(h[7]));
        uint4 v;
        v.x = *reinterpret_cast<unsigned *>(&p0); v.y = *reinterpret_cast<unsigned *>(&p1);
        v.z = *reinterpret_cast<unsigned *>(&p2); v.w = *reinterpret_cast<unsigned *>(&p3);
        *reinterpret_cast<uint4 *>(rowbase + kj * (kPolRows / 8) * 128) = v;
    }
}

__device__ __forceinline__ void pol_wait(unsigned long long *bar, unsigned parity) {
    const unsigned b = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" ::"r"(b),
                 "r"(parity) : "memory");
}

__device__ __forceinline__ void pol_mma(unsigned tmem, unsigned long long da, unsigned long long db, unsigned idesc, unsigned accumulate) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem), "l"(da), "l"(db),
                 "r"(idesc), "r"(accumulate)
                 : "memory");
}

__device__ __forceinline__ void pol_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

// instruction descriptor (cute::UMMA::InstrDescriptor) without N: D FP32, A / B BF16, M = 128
constexpr unsigned kPolIdescBase = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(kPolRows >> 4) << 24);

// layer 2 on the tensor core, issued by one thread: D[128 x 128] = A[128 x 256] B[128 x 256]^T, both K-major, into TMEM
// columns [0, 128), then a commit that arrives on bar
__device__ __forceinline__ void pol_layer2(unsigned tmem, unsigned a0, unsigned b0, unsigned long long *bar) {
    const unsigned idesc = kPolIdescBase | ((unsigned)(kPolH2 >> 3) << 17);   // N = 128
#pragma unroll 1
    for (int ks = 0; ks < kPolH1 / 16; ++ks)
        // K step of 16 = two core matrices along K; LBO = distance between them, SBO = distance between 8-row groups
        pol_mma(tmem, pol_smem_desc(a0 + ks * 2 * (kPolRows / 8) * 128, (kPolRows / 8) * 128, 128),
                pol_smem_desc(b0 + ks * 2 * (kPolH2 / 8) * 128, (kPolH2 / 8) * 128, 128), idesc, ks > 0 ? 1u : 0u);
    pol_commit(bar);
}

// 16 consecutive FP32 columns of this warp's 32 TMEM lanes (one per thread)
__device__ __forceinline__ void pol_ld16(unsigned addr, float *v) {
    unsigned r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = __uint_as_float(r[c]);
}

// the head over this thread's quarter of its row of D (TMEM lane = row): out = (part 0: b3) + sum over the quarter's
// columns c, in column order, of tanh(z2[c] + b2[c]) w3[c]
template <int MX>
__device__ __forceinline__ void pol_head_partial(float (&out)[MX], unsigned lane_base, const PolTables &s, int nout1, int part) {
#pragma unroll
    for (int o = 0; o < MX; ++o) out[o] = (o < nout1 && part == 0) ? s.b3[o] : 0.f;
#pragma unroll 1
    for (int c0 = part * (kPolH2 / kPolSplit); c0 < (part + 1) * (kPolH2 / kPolSplit); c0 += 16) {
        float z[16];
        pol_ld16(lane_base + (unsigned)c0, z);
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const float h2 = pol_tanh(z[c] + s.b2[c0 + c]);
            const float *wr = s.w3 + (c0 + c) * nout1;
#pragma unroll
            for (int o = 0; o < MX; ++o)
                if (o < nout1) out[o] = fmaf(h2, wr[o], out[o]);
        }
    }
}

// partial heads of the row's other three threads -> spart [kPolSplit - 1][kPolRows][kPolMaxOut]; after a barrier the
// row's first thread adds them in part order
template <int MX>
__device__ __forceinline__ void pol_head_store(float *spart, const float (&out)[MX], int row, int part) {
    if (part > 0) {
#pragma unroll
        for (int o = 0; o < MX; ++o) spart[((part - 1) * kPolRows + row) * kPolMaxOut + o] = out[o];
    }
}

template <int MX>
__device__ __forceinline__ void pol_head_combine(float (&out)[MX], const float *spart, int row) {
#pragma unroll
    for (int q = 0; q < kPolSplit - 1; ++q)
#pragma unroll
        for (int o = 0; o < MX; ++o) out[o] += spart[(q * kPolRows + row) * kPolMaxOut + o];
}

// The head read as a dueling Q-network (RLlib DQN's dueling combination, without its per-stream hidden layers):
// out[0, n_out) are the advantages A, out[n_out] the state value V, and q[o] = V + (A[o] - mean A) with the mean
// summed in column order and divided by n_out.  Returns the greedy action: the first maximum over q, i.e. the lowest
// index on ties.  The epsilon-greedy act kernel and the double-DQN target both use this, so "greedy" is one rule.
template <int MX>
__device__ __forceinline__ int dqn_q_values(const float *out, int n_out, float *q) {
    float sa = 0.f, v = 0.f;
#pragma unroll
    for (int o = 0; o < MX; ++o) {
        if (o < n_out) sa += out[o];
        else if (o == n_out) v = out[o];
    }
    const float ma = sa / (float)n_out;
    float best = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int o = 0; o < MX; ++o) {
        q[o] = 0.f;
        if (o < n_out) {
            q[o] = v + (out[o] - ma);
            if (q[o] > best) { best = q[o]; arg = o; }
        }
    }
    return arg;
}

// The head read as a diagonal Gaussian over A = n_out / 2 action dimensions (RLlib's DiagGaussian): mean mu_o in
// column o, log sigma_o in column A + o.  `head` is the row's outputs in shared memory, so the runtime column offset A
// needs no dynamic register indexing.  The act kernel and the learner's kLossPpoDiag stage both call these two
// functions; with explicit round-to-nearest operations (never contracted into FMAs) they give the same bits in both
// kernels, so the first PPO minibatch after a collection sees ratios of exactly 1.
__device__ __forceinline__ float pol_diag_sigma(float log_sigma) { return expf(log_sigma); }

// log N(a; mu, diag sigma^2) = sum over o, in order, of (-u_o^2 / 2 - log sigma_o), u_o = (a_o - mu_o) / sigma_o, then
// minus A log(2 pi) / 2
template <int MX>
__device__ __forceinline__ float pol_diag_logp(const float *head, const float (&a)[MX / 2], int A) {
    float lp = 0.f;
#pragma unroll
    for (int o = 0; o < MX / 2; ++o) {
        if (o < A) {
            const float ls = head[A + o];
            const float u = __fdiv_rn(__fsub_rn(a[o], head[o]), pol_diag_sigma(ls));
            lp = __fsub_rn(__fsub_rn(lp, __fmul_rn(__fmul_rn(0.5f, u), u)), ls);
        }
    }
    return __fsub_rn(lp, __fmul_rn((float)A, 0.9189385332046727f));
}

// dynamic shared memory: A (64 KB) | B (64 KB) | w1 | b1 | b2 | w3 | b3 | barriers
// MO / MX: compile-time caps of the observation and output loops (register arrays, fully unrolled): 8 / 8 for the
// reference's spaces (6-18 observations are 8 or 32; 4 logits + value), 32 / 16 in general.  The shared-memory layout
// does not depend on them.
// EPS: epsilon-greedy over the dueling Q values instead of sampling the logits (discrete engines; DQN).  Draw k = 0 of
// the environment's counter decides (explore when pol_uniform(.., 0) < *io.epsilon), draw k = 1 picks the random
// action min((int)(pol_uniform(.., 1) * n_out), n_out - 1); otherwise the action is dqn_q_values' greedy one.  logp
// is not written.
// DIAG: the diagonal-Gaussian head (continuous engines with an even n_out, PPO with a learned log-std).  For each of
// the A = n_out / 2 dimensions, z is the Box-Muller draw of the N(tanh mu, I) head (k = 2o, 2o + 1) and the action is
// a = fl(fl(sigma z) + mu), no tanh and no clamp; A actions per row go to act_continuous, and logp is pol_diag_logp
// of those FP32 actions.
template <int MO, int MX, bool EPS = false, bool DIAG = false>
__global__ void __launch_bounds__(kPolThreads, 1) policy_act_kernel(PolicyParams pp, PolicyIO io) {
    extern __shared__ __align__(1024) unsigned char pol_smem[];
    unsigned char *sA = pol_smem;
    unsigned char *sB = pol_smem + kPolRows * kPolH1 * 2;
    const PolTables st(reinterpret_cast<float *>(sB + kPolH2 * kPolH1 * 2));
    unsigned long long *bar_w = reinterpret_cast<unsigned long long *>(st.end());              // W2 landed
    unsigned long long *bar_mma = bar_w + 1;                                                 // accumulator ready
    unsigned *tmem_slot = reinterpret_cast<unsigned *>(bar_mma + 1);
    float *spart = reinterpret_cast<float *>(tmem_slot + 2);          // [kPolSplit - 1][kPolRows][kPolMaxOut] partial heads

    const int tid = threadIdx.x, warp = tid >> 5;
    const int row = tid & (kPolRows - 1), part = tid / kPolRows;      // warp % 4 == (row / 32): the TMEM lanes this warp may read
    const int env = blockIdx.x * kPolRows + row;
    const int nout1 = pp.n_out + 1;

    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar_w)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar_mma)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // B operand: 64 KB, already in the canonical layout
        const unsigned bytes = kPolH2 * kPolH1 * 2;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar_w)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         (unsigned)__cvta_generic_to_shared(sB)),
                     "l"(pp.w2_packed), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar_w))
                     : "memory");
    }
    if (warp == 0) {   // TMEM: 128 columns for the 128 x 128 FP32 accumulator
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"((unsigned)__cvta_generic_to_shared(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    pol_stage_tables(st, pp.w1, pp.b1, pp.b2, pp.w3, pp.b3, pp.obs_dim, nout1, tid);
    float x[MO];
    pol_load_x<MO>(x, io.obs, env, pp.obs_dim, env < io.batch);
    __syncthreads();

    pol_layer1<MO>(sA, st, x, pp.obs_dim, row, part);
    // the activations were written through the generic proxy; the tensor core reads through the async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = *tmem_slot;

    if (tid == 0) {
        pol_wait(bar_w, 0);   // W2 has landed
        pol_layer2(tmem, (unsigned)__cvta_generic_to_shared(sA), (unsigned)__cvta_generic_to_shared(sB), bar_mma);
    }
    pol_wait(bar_mma, 0);     // everyone: accumulator ready
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: this thread's quarter of its row of D, + b2, tanh, head; the row's first thread adds the others'
    float out[MX];
    pol_head_partial<MX>(out, tmem + ((unsigned)((warp & 3) * 32) << 16), st, nout1, part);
    pol_head_store<MX>(spart, out, row, part);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem) : "memory");
    if (part > 0 || env >= io.batch) return;
    pol_head_combine<MX>(out, spart, row);

    // ---- outputs
    float v = 0.f;                              // out[n_out], selected without dynamic register indexing
#pragma unroll
    for (int o = 0; o < MX; ++o) if (o == pp.n_out) v = out[o];
    io.value[env] = v;
    if (io.logits) {
#pragma unroll
        for (int o = 0; o < MX; ++o) if (o < nout1) io.logits[(size_t)env * nout1 + o] = out[o];
    }
    if (!io.sample) return;
    const unsigned ctr = pp.counters[env];
    pp.counters[env] = ctr + 1u;
    if constexpr (EPS) {
        float q[MX];
        int act = dqn_q_values<MX>(out, pp.n_out, q);
        if (pol_uniform(pp.seed, (unsigned)env, ctr, 0u) < __ldg(io.epsilon))
            act = min((int)(pol_uniform(pp.seed, (unsigned)env, ctr, 1u) * (float)pp.n_out), pp.n_out - 1);
        io.act_discrete[env] = act;
        return;
    }
    if constexpr (DIAG) {
        // the row's head into its first partial-head slot, free since the combine
        float *head = spart + (size_t)row * kPolMaxOut;
#pragma unroll
        for (int o = 0; o < MX; ++o) if (o < nout1) head[o] = out[o];
        const int A = pp.n_out >> 1;
        float a[MX / 2];
#pragma unroll
        for (int o = 0; o < MX / 2; ++o) {
            a[o] = 0.f;
            if (o < A) {
                const float u1 = pol_uniform(pp.seed, (unsigned)env, ctr, (unsigned)(2 * o));
                const float u2 = pol_uniform(pp.seed, (unsigned)env, ctr, (unsigned)(2 * o + 1));
                const float z = sqrtf(-2.f * __logf(u1)) * __cosf(6.2831853071795865f * u2);      // Box-Muller
                a[o] = __fadd_rn(__fmul_rn(pol_diag_sigma(head[A + o]), z), head[o]);
                io.act_continuous[(size_t)env * A + o] = (double)a[o];
            }
        }
        io.logp[env] = pol_diag_logp<MX>(head, a, A);
        return;
    }
    if (pp.discrete) {
        // log-softmax + Gumbel-max
        float mx = -INFINITY;
#pragma unroll
        for (int o = 0; o < MX; ++o) if (o < pp.n_out) mx = fmaxf(mx, out[o]);
        float se = 0.f;
#pragma unroll
        for (int o = 0; o < MX; ++o) if (o < pp.n_out) se += __expf(out[o] - mx);
        const float lse = mx + __logf(se);
        float best = -INFINITY, best_l = 0.f;
        int arg = 0;
#pragma unroll
        for (int o = 0; o < MX; ++o) {
            if (o < pp.n_out) {
                const float u = pol_uniform(pp.seed, (unsigned)env, ctr, (unsigned)o);
                const float g = out[o] - __logf(-__logf(u));
                if (g > best) { best = g; arg = o; best_l = out[o]; }
            }
        }
        io.act_discrete[env] = arg;
        io.logp[env] = best_l - lse;
    } else {
        float lp = 0.f;
#pragma unroll
        for (int o = 0; o < MX; ++o) {
            if (o < pp.n_out) {
                const float u1 = pol_uniform(pp.seed, (unsigned)env, ctr, (unsigned)(2 * o));
                const float u2 = pol_uniform(pp.seed, (unsigned)env, ctr, (unsigned)(2 * o + 1));
                const float z = sqrtf(-2.f * __logf(u1)) * __cosf(6.2831853071795865f * u2);      // Box-Muller
                io.act_continuous[(size_t)env * pp.n_out + o] = (double)(pol_tanh(out[o]) + z);
                lp += -0.5f * z * z - 0.9189385332046727f;
            }
        }
        io.logp[env] = lp;
    }
}

constexpr size_t kPolSmemBytes = (size_t)kPolRows * kPolH1 * 2 + (size_t)kPolH2 * kPolH1 * 2 +
                                 sizeof(float) * (kPolMaxObs * kPolH1 + kPolH1 + kPolH2 + kPolH2 * kPolMaxOut + kPolMaxOut) + 64 +
                                 sizeof(float) * (kPolSplit - 1) * kPolRows * kPolMaxOut;

}  // namespace paintrl
