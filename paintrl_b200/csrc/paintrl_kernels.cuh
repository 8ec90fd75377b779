// paintrl_kernels.cuh -- the step kernels (one warp per environment).
//
// A step is two launches on the caller's stream (SURVEY.md Appendix A); the second is a programmatic dependent
// launch whose warps wait for their own environment's move phase only (per-environment release / acquire flags):
//   move_kernel   5 sub-steps of {ray vs hull, nearest vertex, closest triangle}    robot.py:302-329
//   paint_kernel  stamp   5 ball queries, colour update, overlap bookkeeping
//                                                     bullet_paint_wrapper.py:568-577, 352-434
//                 score   reward / penalty / termination                 robot_gym_env.py:289-340
//                 observe normalised pose + section/grid observation
//                                                     bullet_paint_wrapper.py:965-978, 1045-1139
//                 same-step auto-reset                                   robot_gym_env.py:370-387
//
// Texel layout ("rows and words", built by build_tables in paintrl_capi.cu): the front texels are
// cut into rows (strips along axis1), each row is sorted by the axis0 coordinate and packed 32
// texels to a word.  Per environment the "painted" predicate (first channel == 255,
// bullet_paint_wrapper.py:354, 723-725) is one bit per texel: bit = predicate differs from the fresh
// texture's.  HSI mode also keeps the int16 thickness per texel in the same slot order.
//   * stamp: per row, the words whose axis0 range can meet the shots; lane = texel, the painted
//     counts are __ballot_sync / __popc of the in-ball masks against the environment's word;
//   * 4-sector observation: per row the number of texels left of / not right of the TCP is found
//     once (static cell table + a few exact compares), so "left / right of the TCP" is a prefix /
//     suffix bit mask of each word and the sector counts are popcounts; only the TCP's own row is
//     compared texel by texel along axis1.
#pragma once
#include "paintrl_device.cuh"

namespace paintrl {

struct StepIO {
    const void *actions;
    double *obs, *reward, *penalty, *actual;
    uint8_t *done;
    int32_t *new_texels;
    double *next_obs;
    const int32_t *reset_start_idx;
};

// The environments a subset step serves (SUBSET instantiations of the step kernels): the k-th warp / move group steps
// environment ids[k] (ids != nullptr) or lo + k, for k < n.  Row k of every StepIO buffer belongs to it.
struct EnvSel {
    const int32_t *ids;
    int lo, n;
};

// `env` = the environment of the k-th warp / move group; false when it has none.  Without SUBSET the k-th environment
// (env is k itself, so the whole-batch kernels compile as they did before subsets existed).  Ids outside [0, num_envs)
// are skipped (the host validates them; the device never indexes out of bounds).
template <bool SUBSET>
__device__ __forceinline__ bool step_env(const EnvSel &sel, int k, int num_envs, int &env) {
    if (!SUBSET) { env = k; return k < num_envs; }
    if (k >= sel.n) return false;
    env = sel.ids ? __ldg(&sel.ids[k]) : sel.lo + k;
    return (unsigned)env < (unsigned)num_envs;
}

// Per-environment dynamic arrays.
struct EnvArrays {
    EnvState *states;
    MoveOut *moves;
    EnvStat *env_stats;
    unsigned *bits;        // [num_envs][n_words_pad]  flip bit per slot
    int16_t *thick;        // [num_envs][n_slots]      HSI thickness (HSI only)
    unsigned *grid_cnt;    // [num_envs][n_gcells_pad] flipped texels per grid-observation cell (grid mode only)
    unsigned *ready;       // [num_envs] 1 once the step's move phase of the environment has been published (paint consumes it)
    ShotPoses *shots;      // [num_envs] normal paint method only: pose / orientation of the five shots
    unsigned *last_mask;   // [num_envs][n_words_pad] normal paint method only: Part._last_painted_pixels as a slot mask
};

// Words of the per-environment bit-plane a warp stages in shared memory (one TMA bulk copy in,
// one out); larger planes are accessed in global memory.
constexpr int kStageWords = 512;

// Per-warp shared scratch.
template <bool STAGED>
struct alignas(128) WarpScratch {
    unsigned sbits[STAGED ? kStageWords : 32];   // the environment's flip bits (STAGED only)
    EnvState st;                                  // the environment's record
    MoveOut mv;                                   // the step's shot centres (from move_kernel)
    int rowL[kMaxRows], rowU[kMaxRows];           // texels of the row with axis0 coordinate <  / <= the TCP's
    int rowWa[kMaxRows], rowWn[kMaxRows];         // stamp candidates of the row: first word, word count
                                                  // (reused as the K != 4 section histogram)
    uint16_t cand[STAGED ? kStageWords : 2];      // flat list of the step's candidate words (STAGED only)
    double hsi_r[2 * kPaintPerAction];                         // HSI: r = distances.max() of each shot, then 1 / r^2 (stamp)
    unsigned long long bar;                       // mbarrier of the bulk copies
};
static_assert(2 * kMaxRows >= 2 * kMaxObs, "the section histogram aliases rowWa / rowWn");

// The environment's flip bits: staged in shared memory or in place in global memory (L2).
template <bool STAGED>
struct Bits {
    unsigned *g;
    unsigned *s;
    __device__ __forceinline__ unsigned ld(int w) const { return STAGED ? s[w] : __ldcg(g + w); }
    __device__ __forceinline__ void st(int w, unsigned v) const {
        if (STAGED) s[w] = v; else __stcg(g + w, v);
    }
};

// ---- TMA bulk copies (cp.async.bulk) between global memory and the warp's scratch
__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}" ::"r"(smem_addr(bar)), "r"(phase)
        : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_addr(src)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ unsigned lowmask(int n) {   // the n lowest bits; n >= 0, clamped to 32 (one BMSK)
    unsigned m;
    asm("bmsk.clamp.b32 %0, 0, %1;" : "=r"(m) : "r"(n));
    return m;
}
__device__ __forceinline__ int clamp32(int v) { return max(v, 0); }   // lowmask() clamps at 32 itself

__device__ __forceinline__ unsigned *bits_of(const DevPack &pk, const EnvArrays &ea, int env) {
    return ea.bits + (size_t)env * pk.n_words_pad;
}
__device__ __forceinline__ int16_t *thick_of(const DevPack &pk, const EnvArrays &ea, int env) {
    return ea.thick ? ea.thick + (size_t)env * pk.n_slots : nullptr;
}
__device__ __forceinline__ unsigned *grid_cnt_of(const DevPack &pk, const EnvArrays &ea, int env) {
    return ea.grid_cnt ? ea.grid_cnt + (size_t)env * pk.n_gcells_pad : nullptr;
}
__device__ __forceinline__ const double *axis_table(const DevPack &pk, int a) {
    return a == 0 ? pk.tx : (a == 1 ? pk.ty : pk.tz);
}

// ------------------------------------------------------------------------------ observation
// Per row: L = #texels with axis0 coordinate < p0, U = #texels with coordinate <= p0.  The cell of a
// coordinate is a monotone function evaluated with the same two FP64 operations for texels (host)
// and the TCP (here), so texels of lower cells are < p0, those of higher cells are > p0, and only
// the TCP's own cell of each row is compared value by value.
template <typename WS>
__device__ __forceinline__ void row_ranks(const DevPack &pk, const Ax &ax, double p0, int lane, WS &ws) {
    const double f = floor((p0 - pk.cx_o0) * pk.cx_inv);
    const double *kx = axis_table(pk, ax.a0);
    for (int r = lane; r < pk.n_rows; r += 32) {
        const int n = __ldg(&pk.row_count[r]);
        int L, U;
        if (!(f >= 0.0)) {
            L = U = 0;
        } else if (f >= (double)pk.ncx) {
            L = U = n;
        } else {
            const int *cs = pk.cell_start + (size_t)r * (pk.ncx + 1) + (int)f;
            const int i0 = __ldg(cs), i1 = __ldg(cs + 1);
            const double *k = kx + (size_t)__ldg(&pk.row_word0[r]) * 32 + i0;
            // the first four keys of the cell in one round of loads (the tables are padded), the rest in a loop
            const double k0 = __ldg(k), k1 = __ldg(k + 1), k2 = __ldg(k + 2), k3 = __ldg(k + 3);
            const int c = i1 - i0;
            L = i0 + ((c > 0 && k0 < p0) ? 1 : 0) + ((c > 1 && k1 < p0) ? 1 : 0) + ((c > 2 && k2 < p0) ? 1 : 0) +
                ((c > 3 && k3 < p0) ? 1 : 0);
            U = i0 + ((c > 0 && k0 <= p0) ? 1 : 0) + ((c > 1 && k1 <= p0) ? 1 : 0) + ((c > 2 && k2 <= p0) ? 1 : 0) +
                ((c > 3 && k3 <= p0) ? 1 : 0);
            for (int i = 4; i < c; ++i) {
                const double x = __ldg(&k[i]);
                L += (x < p0) ? 1 : 0;
                U += (x <= p0) ? 1 : 0;
            }
        }
        ws.rowL[r] = L;
        ws.rowU[r] = U;
    }
    __syncwarp();
}

// The TCP's row of the texel layout (-1 / n_rows when it lies below / above all rows).
__device__ __forceinline__ int pose_row(const DevPack &pk, double p1) {
    const double f1 = floor((p1 - pk.row_o1) * pk.row_inv);
    return !(f1 >= 0.0) ? -1 : (f1 >= (double)pk.n_rows ? pk.n_rows : (int)f1);
}

// 4-sector observation (bullet_paint_wrapper.py:1033-1061): for every front texel, rx / ry = texel
// position - TCP position along the principal axes; skipped if both are 0; sector 0 if rx>0,ry>0,
// 1 if rx<0,ry>0, 2 if rx<0,ry<0, else 3; obs[s] = #(status != 255) / #texels of the sector.
template <typename WS, typename BITS>
__device__ __forceinline__ void section4_counts(const DevPack &pk, const Ax &ax, const BITS &bits, const Vec3 &pose, int lane, WS &ws,
                                                int tot[4], int open[4], bool ranks_ready PAINTRL_PROF_PARAM) {
    const double p0 = comp(pose, ax.a0), p1 = comp(pose, ax.a1);
    PAINTRL_PROF(21, lane == 0);
    if (!ranks_ready) row_ranks(pk, ax, p0, lane, ws);
    PAINTRL_PROF(22, lane == 0);
    const int prow = pose_row(pk, p1);
    const bool init_painted = (pk.status_init == kPainted);
    const unsigned flip = init_painted ? 0u : 0xffffffffu;   // open = bits ^ flip

    // ---- rows above / below the TCP's row, one row per lane: texels left of the TCP are the first L
    // slots of the row, texels right of it the slots from U on, so the sector counts are popcounts of
    // prefix masks of the row's words (totals are static: L, U - L, n - U)
    int t0 = 0, t1 = 0, t2 = 0, t3 = 0;
    int o0 = 0, o1 = 0, o2 = 0, o3 = 0;
    for (int r = lane; r < pk.n_rows; r += 32) {
        if (r == prow) continue;
        const int n = __ldg(&pk.row_count[r]), L = ws.rowL[r], U = ws.rowU[r];
        const int w0 = __ldg(&pk.row_word0[r]), nw = (n + 31) >> 5;
        const int kL = L >> 5, kU = U >> 5;
        const unsigned last = lowmask(n - ((nw - 1) << 5));
        int cL = 0, cU = 0, cA = 0;   // open texels among the first L / first U / all n slots
        for (int wi = 0; wi < nw; ++wi) {   // whole words
            unsigned o = bits.ld(w0 + wi) ^ flip;
            if (wi == nw - 1) o &= last;
            const int c = __popc(o);
            cA += c;
            cL += wi < kL ? c : 0;
            cU += wi < kU ? c : 0;
        }
        if (kL < nw) cL += __popc((bits.ld(w0 + kL) ^ flip) & lowmask(L & 31) & (kL == nw - 1 ? last : 0xffffffffu));
        if (kU < nw) cU += __popc((bits.ld(w0 + kU) ^ flip) & lowmask(U & 31) & (kU == nw - 1 ? last : 0xffffffffu));
        if (r > prow) { t1 += L; t0 += n - U; t3 += U - L; o1 += cL; o0 += cA - cU; o3 += cU - cL; }
        else { t2 += L; t3 += n - L; o2 += cL; o3 += cA - cL; }
    }
    PAINTRL_PROF(23, lane == 0);
    // ---- the TCP's own row, texel by texel along axis1 (lane = slot): ballots of y > p1 / y < p1
    // against the row's prefix masks; every lane holds the same counts, lane 0 contributes them
    if (prow >= 0 && prow < pk.n_rows) {
        const int w0 = __ldg(&pk.row_word0[prow]), w1 = __ldg(&pk.row_word0[prow + 1]);
        const int n = __ldg(&pk.row_count[prow]), L = ws.rowL[prow], U = ws.rowU[prow];
        const double *ky = axis_table(pk, ax.a1) + (size_t)w0 * 32 + lane;
        int u0 = 0, u1 = 0, u2 = 0, u3 = 0, v0 = 0, v1 = 0, v2 = 0, v3 = 0;
#pragma unroll 2
        for (int wi = 0; wi < w1 - w0; ++wi) {
            const double y = __ldg(ky + (size_t)wi * 32);
            const unsigned mV = lowmask(clamp32(n - (wi << 5)));
            const unsigned gy = __ballot_sync(kFull, y > p1) & mV, ly = __ballot_sync(kFull, y < p1) & mV;
            const unsigned mL = lowmask(clamp32(L - (wi << 5))), mU = lowmask(clamp32(U - (wi << 5)));
            const unsigned o = bits.ld(w0 + wi) ^ flip;
            const unsigned q0 = gy & ~mU, q1 = gy & mL, q2 = ly & mL;
            const unsigned skip = mV & ~gy & ~ly & mU & ~mL;              // rx == 0 and ry == 0
            const unsigned q3 = mV & ~(q0 | q1 | q2 | skip);
            u0 += __popc(q0); u1 += __popc(q1); u2 += __popc(q2); u3 += __popc(q3);
            v0 += __popc(q0 & o); v1 += __popc(q1 & o); v2 += __popc(q2 & o); v3 += __popc(q3 & o);
        }
        if (lane == 0) { t0 += u0; t1 += u1; t2 += u2; t3 += u3; o0 += v0; o1 += v1; o2 += v2; o3 += v3; }
    }
    PAINTRL_PROF(24, lane == 0);
    tot[0] = __reduce_add_sync(kFull, t0); tot[1] = __reduce_add_sync(kFull, t1);
    tot[2] = __reduce_add_sync(kFull, t2); tot[3] = __reduce_add_sync(kFull, t3);
    open[0] = __reduce_add_sync(kFull, o0); open[1] = __reduce_add_sync(kFull, o1);
    open[2] = __reduce_add_sync(kFull, o2); open[3] = __reduce_add_sync(kFull, o3);
}

// Section observation with K != 4 sectors (atan2 path, bullet_paint_wrapper.py:1026-1031): full scan.
template <typename BITS>
__device__ __forceinline__ void sectionk_counts(const DevPack &pk, const Ax &ax, const BITS &bits, const Vec3 &pose, int section,
                                                int lane, int *hist /*[2*kMaxObs] smem*/) {
    for (int i = lane; i < 2 * kMaxObs; i += 32) hist[i] = 0;
    __syncwarp();
    const double p0 = comp(pose, ax.a0), p1 = comp(pose, ax.a1);
    const double *c0 = axis_table(pk, ax.a0), *c1 = axis_table(pk, ax.a1);
    const double basis = 2 * kPi / section;
    const bool init_painted = (pk.status_init == kPainted);
    for (int w = 0; w < pk.n_words; ++w) {
        const int j = w * 32 + lane;
        if (__ldg(&pk.slot_to_pack[j]) < 0) continue;
        const double rx = __ldg(&c0[j]) - p0, ry = __ldg(&c1[j]) - p1;
        if (rx == 0.0 && ry == 0.0) continue;
        double angle = atan2(ry, rx);
        if (angle < 0.0) angle = 2 * kPi + angle;
        int idx = (int)np_floor_divide(angle, basis);
        if (idx >= section) idx = section - 1;
        atomicAdd(&hist[idx], 1);
        const bool bit = (bits.ld(w) >> lane) & 1u;
        if (init_painted ? bit : !bit) atomicAdd(&hist[kMaxObs + idx], 1);
    }
    __syncwarp();
}

// robot_gym_env.py:306-319 _augmented_observation; every lane returns, lanes < obs_dim write.
template <typename WS, typename BITS>
__device__ __forceinline__ void write_observation(const DevPack &pk, const Ax &ax, const DevConfig &cfg, const BITS &bits,
                                                  const unsigned *grid_cnt, const Vec3 &pose, int lane, WS &ws,
                                                  double *obs_a, double *obs_b PAINTRL_PROF_PARAM) {
    double a1, a2;
    normalized_pose(pk, ax, pose, a1, a2);
    const int grad = cfg.obs_grad;
    if (cfg.obs_mode == 2) {   // simple
        if (lane < 2) {
            double v = lane == 0 ? a1 : a2;
            if (obs_a) obs_a[lane] = v;
            if (obs_b) obs_b[lane] = v;
        }
        return;
    }
    if (cfg.obs_mode == 1) {   // grid (bullet_paint_wrapper.py:1126-1139): painted texels per cell from the flip counters
        const int cells = grad * grad;
        const bool init_painted = (pk.status_init == kPainted);
        for (int c = lane; c < cells; c += 32) {
            const int total = __ldg(&pk.gtotal[c]);
            const int fl = (int)__ldcg(&grid_cnt[c]);
            const int painted = init_painted ? total - fl : fl;
            double v = total == 0 ? 0.0 : 1.0 - (double)painted / (double)total;
            if (obs_a) obs_a[c] = v;
            if (obs_b) obs_b[c] = v;
        }
        return;
    }
    // section / discrete
    if (grad == 4) {
        int tot[4], open[4];
        section4_counts(pk, ax, bits, pose, lane, ws, tot, open, false PAINTRL_PROF_PASS);
        if (lane < 4) {
            int t = lane == 0 ? tot[0] : (lane == 1 ? tot[1] : (lane == 2 ? tot[2] : tot[3]));
            int o = lane == 0 ? open[0] : (lane == 1 ? open[1] : (lane == 2 ? open[2] : open[3]));
            double v = t == 0 ? 0.0 : (double)o / (double)t;
            if (obs_a) obs_a[lane] = v;
            if (obs_b) obs_b[lane] = v;
        }
    } else {
        int *hist = ws.rowWa;   // rowWa / rowWn are contiguous and free once the stamp is done
        sectionk_counts(pk, ax, bits, pose, grad, lane, hist);
        for (int s = lane; s < grad; s += 32) {
            int t = hist[s], o = hist[kMaxObs + s];
            double v = t == 0 ? 0.0 : (double)o / (double)t;
            if (obs_a) obs_a[s] = v;
            if (obs_b) obs_b[s] = v;
        }
        __syncwarp();
    }
    if (lane == 0) {
        if (cfg.obs_mode == 3) {   // discrete: robot_gym_env.py:101-103, 314-318
            int position = (handle_pos(a1) + 1) * 22 + handle_pos(a2);
            double v = 1.0 / position;
            if (obs_a) obs_a[grad] = v;
            if (obs_b) obs_b[grad] = v;
        } else {
            if (obs_a) { obs_a[grad] = a1; obs_a[grad + 1] = a2; }
            if (obs_b) { obs_b[grad] = a1; obs_b[grad + 1] = a2; }
        }
    }
}

// ------------------------------------------------------------------------------ reset pieces
// Part.reset_part (bullet_paint_wrapper.py:706-708): restore the init colour, 128-bit stores.
// HSI thickness plane: a texel's flip bit is set exactly when its thickness has left the initial 255
// (values only decrease, bullet_paint_wrapper.py:429-431; set_status_kernel keeps the same invariant), so
// only the 32-texel words with a bit set are rewritten -- a short episode touches a few hundred of the
// part's ~14 k texels, and the plane is 30 KB per environment.  `bits` is the environment's current
// bit-plane (shared copy or global), `gbits` its global home.
template <typename BITS>
__device__ __forceinline__ void clear_planes(const DevPack &pk, const BITS &bits, unsigned *gbits, int16_t *thick, unsigned *grid_cnt,
                                             int lane) {
    const uint4 z = make_uint4(0, 0, 0, 0);
    if (thick) {
        const unsigned v2 = ((unsigned)(uint16_t)pk.status_init) * 0x10001u;
        const uint4 v = make_uint4(v2, v2, v2, v2);
        if (pk.status_init == kPainted) {
            for (int w = lane; w < pk.n_words; w += 32) {
                if (bits.ld(w) != 0u) {
                    uint4 *dst = reinterpret_cast<uint4 *>(thick + (size_t)w * 32);
                    dst[0] = v; dst[1] = v; dst[2] = v; dst[3] = v;
                }
            }
            __syncwarp();      // every lane has read its words before the plane is zeroed below
        } else {
            for (int j = lane * 8; j < pk.n_slots; j += 256) *reinterpret_cast<uint4 *>(thick + j) = v;
        }
    }
    for (int w = lane * 4; w < pk.n_words_pad; w += 128) *reinterpret_cast<uint4 *>(gbits + w) = z;
    if (grid_cnt)
        for (int w = lane * 4; w < pk.n_gcells_pad; w += 128) *reinterpret_cast<uint4 *>(grid_cnt + w) = z;
}

// Initial fill of the thickness planes (paintrl_create): from then on resets are incremental.
__global__ void fill_thickness_kernel(int16_t *thick, size_t n, int16_t value) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) thick[i] = value;
}

// Robot.reset(pose) (robot.py:366-372, 208-212)
__device__ __forceinline__ void robot_reset(EnvState &st, const double *pos, const double *normal) {
    Vec3 n = {normal[0], normal[1], normal[2]};
    quat_from_normal(n, st.quat);
    st.pose[0] = pos[0]; st.pose[1] = pos[1]; st.pose[2] = pos[2];
    st.flags = (st.flags & kFlagHasLast) | kFlagLastOnPart;   // terminate cleared, last_on_part = True
    st.term_counter = 0;
    st.last_angle = 0.0;
}

// PaintGymEnv.reset (robot_gym_env.py:370-387) minus the planes and the observation
__device__ __forceinline__ void state_reset(const DevPack &pk, EnvState &st, int start_index) {
    st.flags &= ~kFlagHasLast;                 // _last_painted_pixels = []
    st.step_counter = 0;
    st.total_return = 0.0;
    st.total_reward = 0.0;
    robot_reset(st, pk.start_pos + 3 * start_index, pk.start_normal + 3 * start_index);
    st.episode += 1;
}

__device__ __forceinline__ void load_state(const EnvState *g, EnvState &st) {
    const double2 *src = reinterpret_cast<const double2 *>(g);
    double2 *dst = reinterpret_cast<double2 *>(&st);
#pragma unroll
    for (int i = 0; i < 8; ++i) dst[i] = src[i];
}
__device__ __forceinline__ void store_state(EnvState *g, const EnvState &st, int lane) {
    // lanes 0..7 each write one 16-byte piece of the record (the record is warp-uniform)
    const double2 *src = reinterpret_cast<const double2 *>(&st);
    double2 v = src[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) if (lane == i) v = src[i];
    if (lane < 8) reinterpret_cast<double2 *>(g)[lane] = v;
}

__device__ __forceinline__ int auto_start_index(const DevPack &pk, const DevConfig &cfg, int env, int episode) {
    return (int)(splitmix64(cfg.seed ^ splitmix64(((unsigned long long)env << 32) | (unsigned)episode)) %
                 (unsigned long long)pk.n_starts);
}

// ------------------------------------------------------------------------------ stamp
// Part.fast_paint x 5 (bullet_paint_wrapper.py:568-577) + colour handlers (:352-434).
//
// The ball test `dx*dx + dy*dy + dz*dz <= r*r` (FP64, exactly the kd-tree's) is decided in FP32 on
// origin-relative coordinates whenever the FP32 value is further than kBallEps from r*r -- the FP32
// evaluation differs from the FP64 one by < 2e-8 for |d| <= 2r (checked per part by build_tables)
// -- and in FP64 otherwise.
constexpr float kBallEps = 1e-7f;
constexpr int NS = kPaintPerAction;

struct ShotsF { float x[NS + 1], y[NS + 1], z[NS + 1]; };

// exact centre of shot s (s == NS: the previous step's last shot)
template <typename WS>
__device__ __forceinline__ double cen(const WS &ws, int s, int k) {
    return s < NS ? ws.mv.centers[s][k] : ws.st.last_center[k];
}

// FP32 pre-test of slot j against the six balls: e[s] = |t - c_s|^2 - r^2 (negative inside);
// returns true when some |e[s]| <= kBallEps, i.e. FP32 cannot decide and the FP64 test must.
__device__ __forceinline__ bool ball_pretest_at(const ShotsF &c, float tx, float ty, float tz, float e[NS + 1]) {
    const float nr2f = -(float)(kPaintRadius * kPaintRadius);
    float m = INFINITY;
#pragma unroll
    for (int s = 0; s <= NS; ++s) {
        const float dx = tx - c.x[s], dy = ty - c.y[s], dz = tz - c.z[s];
        e[s] = fmaf(dz, dz, fmaf(dy, dy, fmaf(dx, dx, nr2f)));
        m = fminf(m, fabsf(e[s]));
    }
    return m <= kBallEps;
}
__device__ __forceinline__ bool ball_pretest(const DevPack &pk, const ShotsF &c, int j, float e[NS + 1]) {
    return ball_pretest_at(c, __ldg(&pk.fx[j]), __ldg(&pk.fy[j]), __ldg(&pk.fz[j]), e);
}

// the exact test `dx*dx + dy*dy + dz*dz <= r*r` of slot j against ball s (bullet_paint_wrapper.py:569)
template <typename WS>
__device__ __forceinline__ bool ball_exact(const WS &ws, double x, double y, double z, int s) {
    const double r2 = kPaintRadius * kPaintRadius;
    const double dx = x - cen(ws, s, 0), dy = y - cen(ws, s, 1), dz = z - cen(ws, s, 2);
    return (dx * dx + dy * dy + dz * dz) <= r2;
}

// which shots (bits 0..4) and the previous step's last shot (bit 5) contain slot j
template <typename WS>
__device__ __forceinline__ unsigned ball_mask(const DevPack &pk, const ShotsF &c, const WS &ws, int j, bool has_last) {
    float e[NS + 1];
    unsigned in = 0;
    if (ball_pretest(pk, c, j, e)) {
        const double x = __ldg(&pk.tx[j]), y = __ldg(&pk.ty[j]), z = __ldg(&pk.tz[j]);
#pragma unroll
        for (int s = 0; s <= NS; ++s) in |= (ball_exact(ws, x, y, z, s) ? 1u : 0u) << s;
    } else {
#pragma unroll
        for (int s = 0; s <= NS; ++s) in |= (e[s] <= 0.f ? 1u : 0u) << s;
    }
    if (!has_last) in &= (1u << NS) - 1u;
    return in;
}

// RGB stamp: is slot j inside some shot, and is it a "valid pixel" of some shot -- inside shot s but
// not inside the shot before it (bullet_paint_wrapper.py:575; the shot before shot 0 is the previous
// step's last one).  Predicate logic only, no per-shot bit mask.
template <typename WS>
__device__ __forceinline__ void ball_flags_at(const DevPack &pk, const ShotsF &c, const WS &ws, int j, float tx, float ty, float tz,
                                              bool has_last, bool &any_shot, bool &possible) {
    float e[NS + 1];
    bool in[NS + 1];
    if (ball_pretest_at(c, tx, ty, tz, e)) {
        const double x = __ldg(&pk.tx[j]), y = __ldg(&pk.ty[j]), z = __ldg(&pk.tz[j]);
#pragma unroll
        for (int s = 0; s <= NS; ++s) in[s] = ball_exact(ws, x, y, z, s);
    } else {
#pragma unroll
        for (int s = 0; s <= NS; ++s) in[s] = e[s] <= 0.f;
    }
    bool prev = has_last && in[NS];
    any_shot = false;
    possible = false;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        any_shot = any_shot || in[s];
        possible = possible || (in[s] && !prev);
        prev = in[s];
    }
}
template <typename WS>
__device__ __forceinline__ void ball_flags(const DevPack &pk, const ShotsF &c, const WS &ws, int j, bool has_last, bool &any_shot,
                                           bool &possible) {
    ball_flags_at(pk, c, ws, j, __ldg(&pk.fx[j]), __ldg(&pk.fy[j]), __ldg(&pk.fz[j]), has_last, any_shot, possible);
}

// Per row, the words whose texels can lie inside one of the step's shots: the row's axis1 interval
// against the shots' axis1 extent gives a half-width along axis0 (the ball projects to a disc of
// the same radius), the static cell table turns the axis0 interval into a slot range.  FP32 on
// origin-relative coordinates with margins: it only has to be conservative, every slot of a
// candidate word is tested exactly.  STAGED: the words are also flattened into ws.cand (returns
// their number).
template <bool STAGED, int COLOR, typename WS>
__device__ __forceinline__ int stamp_ranges(const DevPack &pk, float lo0, float hi0, float lo1, float hi1, int lane, WS &ws) {
    const float rr = (float)kPaintRadius + 4e-5f;
    int base = 0;
    for (int r0 = 0; r0 < pk.n_rows; r0 += 32) {
        const int r = r0 + lane;
        int wa = 0, wn = 0;
        if (r < pk.n_rows) {
            const float ylo = fmaf((float)r, pk.rel_row_h, pk.rel_row_o1) - 2e-5f, yhi = ylo + pk.rel_row_h + 4e-5f;
            const float dy = fmaxf(0.f, fmaxf(ylo - hi1, lo1 - yhi));
            if (dy <= rr) {
                const float hw = sqrtf(rr * rr - dy * dy) + 4e-5f;
                const float fa = floorf((lo0 - hw - pk.rel_cx_o0) * pk.rel_cx_inv) - 1.f;
                const float fb = floorf((hi0 + hw - pk.rel_cx_o0) * pk.rel_cx_inv) + 1.f;
                if (fb >= 0.f && fa < (float)pk.ncx) {
                    const int ca = (int)fmaxf(fa, 0.f), cb = (int)fminf(fb, (float)(pk.ncx - 1));
                    const int *cs = pk.cell_start + (size_t)r * (pk.ncx + 1);
                    const int i0 = __ldg(cs + ca), i1 = __ldg(cs + cb + 1);
                    if (i1 > i0) {
                        wa = __ldg(&pk.row_word0[r]) + (i0 >> 5);
                        wn = ((i1 - 1) >> 5) - (i0 >> 5) + 1;
                    }
                }
            }
            ws.rowWa[r] = wa;
            ws.rowWn[r] = wn;
        }
        if (STAGED) {
            int incl = wn;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += u;
            }
            const int at = base + incl - wn;
            for (int t = 0; t < wn; ++t) ws.cand[at + t] = (uint16_t)(wa + t);
            base += __shfl_sync(kFull, incl, 31);
        }
    }
    __syncwarp();
    return base;
}

// Calls body(w) warp-uniformly for every candidate word.
template <bool STAGED, typename WS, typename BodyFn>
__device__ __forceinline__ void for_each_stamp_word(const DevPack &pk, int lane, const WS &ws, int n_cand, BodyFn body) {
    if constexpr (STAGED) {
        for (int k = 0; k < n_cand; ++k) body((int)ws.cand[k]);
    } else {
        for (int r0 = 0; r0 < pk.n_rows; r0 += 32) {
            const int r = r0 + lane;
            const int wa = r < pk.n_rows ? ws.rowWa[r] : 0, wn = r < pk.n_rows ? ws.rowWn[r] : 0;
            unsigned m = __ballot_sync(kFull, wn > 0);
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const int a = __shfl_sync(kFull, wa, src), n = __shfl_sync(kFull, wn, src);
                for (int w = a; w < a + n; ++w) body(w);
            }
        }
    }
}

// Returns (warp-uniform) the newly painted count (RGB) / removed thickness units (HSI), the
// |union of valid pixels| of robot.py:425 and whether any flip bit changed.
template <int COLOR, bool STAGED, typename WS, typename BITS>
__device__ __forceinline__ void stamp(const DevPack &pk, const Ax &ax, const BITS &bits, int16_t *thick, unsigned *grid_cnt, bool has_last,
                                      int lane, WS &ws, int &n_new_out, int &n_possible_out, bool &dirty_out PAINTRL_PROF_PARAM) {
    ShotsF c;
#pragma unroll
    for (int s = 0; s <= NS; ++s) {
        c.x[s] = (float)(cen(ws, s, 0) - pk.org0);
        c.y[s] = (float)(cen(ws, s, 1) - pk.org1);
        c.z[s] = (float)(cen(ws, s, 2) - pk.org2);
    }
    float lo0 = INFINITY, hi0 = -INFINITY, lo1 = INFINITY, hi1 = -INFINITY;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const float c0 = ax.a0 == 0 ? c.x[s] : (ax.a0 == 1 ? c.y[s] : c.z[s]);
        const float c1 = ax.a1 == 0 ? c.x[s] : (ax.a1 == 1 ? c.y[s] : c.z[s]);
        lo0 = fminf(lo0, c0); hi0 = fmaxf(hi0, c0);
        lo1 = fminf(lo1, c1); hi1 = fmaxf(hi1, c1);
    }
    PAINTRL_PROF(17, lane == 0);
    const int n_cand = stamp_ranges<STAGED, COLOR>(pk, lo0, hi0, lo1, hi1, lane, ws);
    PAINTRL_PROF(18, lane == 0);

    double rmax[NS];
    if (COLOR == 1) {   // HSI: r = distances.max() per shot (bullet_paint_wrapper.py:423-424)
#pragma unroll
        for (int s = 0; s < NS; ++s) rmax[s] = -1.0;
        for_each_stamp_word<STAGED>(pk, lane, ws, n_cand, [&](int w) {
            const int j = w * 32 + lane;
            const unsigned in = ball_mask(pk, c, ws, j, false);
            if (in) {
                const double x = __ldg(&pk.tx[j]), y = __ldg(&pk.ty[j]), z = __ldg(&pk.tz[j]);
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    if (in & (1u << s)) {
                        const double dx = x - cen(ws, s, 0), dy = y - cen(ws, s, 1), dz = z - cen(ws, s, 2);
                        rmax[s] = fmax(rmax[s], dx * dx + dy * dy + dz * dz);
                    }
                }
            }
        });
#pragma unroll
        for (int s = 0; s < NS; ++s) rmax[s] = sqrt(warp_max(rmax[s]));   // sqrt is monotone
        if (lane < NS) {                     // r and 1 / r^2 of shot `lane` (one division per lane)
            double r = rmax[0];
#pragma unroll
            for (int s = 1; s < NS; ++s) r = lane == s ? rmax[s] : r;
            ws.hsi_r[lane] = r;
            ws.hsi_r[NS + lane] = r > 0.0 ? 1.0 / (r * r) : 0.0;
        }
        __syncwarp();
    }

    int n_new = 0, n_possible = 0;   // RGB: warp-uniform; HSI n_new: per-lane partial
    unsigned any = 0;
    if (COLOR == 0 && !STAGED) {
        // Large textures (bit-plane in global memory, hundreds of candidate words per step): a word at a time the
        // loop pays two dependent L2 round trips per word (the texels' coordinates, then the plane word; ncu at
        // C4: 6.1 warps per issue on the long scoreboard, 50 % of the samples on those two waits).  Four words per
        // iteration, all their loads issued before the first is tested.
        constexpr int kBatch = 4;
        for (int r0 = 0; r0 < pk.n_rows; r0 += 32) {
            const int r = r0 + lane;
            const int wa = r < pk.n_rows ? ws.rowWa[r] : 0, wn = r < pk.n_rows ? ws.rowWn[r] : 0;
            unsigned m = __ballot_sync(kFull, wn > 0);
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const int a = __shfl_sync(kFull, wa, src), n = __shfl_sync(kFull, wn, src);
                for (int w0 = a; w0 < a + n; w0 += kBatch) {
                    float tx[kBatch], ty[kBatch], tz[kBatch];
                    unsigned old[kBatch];
#pragma unroll
                    for (int q = 0; q < kBatch; ++q) {
                        const int w = min(w0 + q, a + n - 1);          // the tail repeats the last word (not processed twice)
                        const int j = w * 32 + lane;
                        tx[q] = __ldg(&pk.fx[j]); ty[q] = __ldg(&pk.fy[j]); tz[q] = __ldg(&pk.fz[j]);
                        old[q] = bits.ld(w);
                    }
#pragma unroll
                    for (int q = 0; q < kBatch; ++q) {
                        const int w = w0 + q;
                        if (w >= a + n) break;
                        const int j = w * 32 + lane;
                        bool any_shot, possible;
                        ball_flags_at(pk, c, ws, j, tx[q], ty[q], tz[q], has_last, any_shot, possible);
                        const unsigned uni = __ballot_sync(kFull, any_shot);
                        if (uni == 0u) continue;
                        n_possible += __popc(__ballot_sync(kFull, possible));
                        const unsigned flipped = uni & ~old[q];
                        if (flipped) {
                            n_new += __popc(flipped);
                            if (lane == 0) bits.st(w, old[q] | uni);
                            any |= flipped;
                            if (grid_cnt && ((flipped >> lane) & 1u)) atomicAdd(grid_cnt + __ldg(&pk.gcell[j]), 1u);
                        }
                    }
                }
            }
        }
    } else if (COLOR == 0) {                               // :358-365
        for_each_stamp_word<STAGED>(pk, lane, ws, n_cand, [&](int w) {
            const int j = w * 32 + lane;
            bool any_shot, possible;
            ball_flags(pk, c, ws, j, has_last, any_shot, possible);
            const unsigned uni = __ballot_sync(kFull, any_shot);
            if (uni == 0u) return;
            n_possible += __popc(__ballot_sync(kFull, possible));
            const unsigned old = bits.ld(w);
            __syncwarp();                                  // every lane has read the word before lane 0 rewrites it
            const unsigned flipped = uni & ~old;           // slots whose painted predicate changes
            if (flipped) {
                n_new += __popc(flipped);
                if (lane == 0) bits.st(w, old | uni);
                any |= flipped;
                if (grid_cnt && ((flipped >> lane) & 1u)) atomicAdd(grid_cnt + __ldg(&pk.gcell[j]), 1u);
            }
        });
    } else {                                               // :411-434
        for_each_stamp_word<STAGED>(pk, lane, ws, n_cand, [&](int w) {
            const int j = w * 32 + lane;
            const unsigned in = ball_mask(pk, c, ws, j, has_last);
            const unsigned shots = in & ((1u << NS) - 1u);
            const unsigned uni = __ballot_sync(kFull, shots != 0u);
            if (uni == 0u) return;
            // affected \ last_affected, shot by shot (:575): shot s counts if the previous shot missed the texel
            const unsigned prev = ((shots << 1) | (in >> NS)) & ((1u << NS) - 1u);
            n_possible += __popc(__ballot_sync(kFull, (shots & ~prev) != 0u));
            bool fl = false;
            if (shots) {
                const int sv0 = (int)__ldcg(&thick[j]);
                int sv = sv0;
                const double x = __ldg(&pk.tx[j]), y = __ldg(&pk.ty[j]), z = __ldg(&pk.tz[j]);
                // not unrolled: one copy of the FP64 square root and division in the instruction stream (unrolled
                // five times the kernel outgrew the instruction cache: "no instruction" was its top stall at C3)
#pragma unroll 1
                for (int s = 0; s < NS; ++s) {
                    if ((shots & (1u << s)) && sv > 0) {
                        const double dx = x - cen(ws, s, 0), dy = y - cen(ws, s, 1), dz = z - cen(ws, s, 2);
                        const double d2 = dx * dx + dy * dy + dz * dz;
                        // quantity = int(25 (1 - (d / r)^2)) + 1 (:429).  The reference's 25 (1 - ratio^2) (a square
                        // root, a division, four roundings) and the screening value 25 (1 - d2 / r^2) differ by
                        // < 1e-13, so when the latter is more than 1e-9 away from an integer both truncate to the same
                        // one; otherwise -- and for the farthest texel, where it is 0 -- the reference's own
                        // expression decides.
                        const double qa = kHsiTargetMax * (1.0 - d2 * ws.hsi_r[NS + s]);
                        const double qf = floor(qa);
                        int quantity = (int)qf + 1;
                        if (!(qa > 1e-9 && qa - qf > 1e-9 && (qf + 1.0) - qa > 1e-9)) {
                            const double ratio = sqrt(d2) / ws.hsi_r[s];
                            quantity = (int)(kHsiTargetMax * (1.0 - ratio * ratio)) + 1;
                        }
                        sv -= quantity;
                        n_new += quantity;
                    }
                }
                if (sv != sv0) {
                    __stcg(&thick[j], (int16_t)sv);
                    fl = (sv0 == kPainted);                // values only decrease: 255 is left once
                }
            }
            const unsigned flipped = __ballot_sync(kFull, fl);
            if (flipped) {
                if (lane == 0) bits.st(w, bits.ld(w) | flipped);
                any |= flipped;
                if (grid_cnt && ((flipped >> lane) & 1u)) atomicAdd(grid_cnt + __ldg(&pk.gcell[j]), 1u);
            }
        });
    }
    n_new_out = (COLOR == 0) ? n_new : __reduce_add_sync(kFull, n_new);
    n_possible_out = n_possible;
    dirty_out = any != 0u;
    __syncwarp();
}

// ------------------------------------------------------------------------------ stamp, normal paint method
// Robot._paint (robot.py:280-285) + Part.paint (bullet_paint_wrapper.py:562-566): per shot a fan of n_beams rays from
// the TCP (Robot._paint_plain in the TCP frame, robot.py:251-258), the hits on the hull, the texel nearest to every hit
// (cKDTree.query, k = 1) and the colour handlers on that list -- duplicates included.  One lane per beam.
//   * ray: the move cell under the beam's expected entry point supplies a short plane list; the entry point lying in
//     that cell's region proves the list sufficient (ray_test's argument (2a)); otherwise all planes are scanned.
//     Max / min over planes are order-independent, so the hit is the serial scan's bit for bit.
//   * nearest texel: the 3 x (2R + 1) block of texel rows / cells around the hit, exact FP64 squared distances,
//     accepted when the best beats the distance to the block's border (every other texel is farther); else a wider
//     block, else all slots.  Texels sharing one position resolve to the kd-tree's twin (nn_rep_slot).
constexpr int kMaxBeams = 512;

struct alignas(16) NormalScratch {
    double pos[kPaintPerAction][3];
    double quat[kPaintPerAction][4];
    unsigned shot_mask[kStageWords];       // texels the current shot touched
    unsigned possible[kStageWords];        // union over the step's shots of (affected \ last affected)
    uint16_t beam_slot[kMaxBeams];         // nearest texel (slot) per beam, 0xFFFF = the beam missed
    double beam_q[kMaxBeams];              // HSI: distance of that texel to the shot centre
};

__device__ __forceinline__ void slab_serial(const double2 *planes, int n, const Vec3 &frm, double d0, double d1, double d2, double &t_in,
                                            double &t_out, bool &outside) {
    t_in = -INFINITY; t_out = INFINITY; outside = false;
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        const double2 lo = __ldg(planes + 2 * i), hi2 = __ldg(planes + 2 * i + 1);
        const double den = (lo.x * d0 + lo.y * d1) + hi2.x * d2;
        const double num = hi2.y - ((lo.x * frm.x + lo.y * frm.y) + hi2.x * frm.z);
        if (den == 0.0) {
            if (num < 0.0) outside = true;
        } else {
            const double t = num / den;
            if (den < 0.0) t_in = fmax(t_in, t);
            else t_out = fmin(t_out, t);
        }
    }
}

// shim S1 rayTestBatch for one beam, by one lane, as far as the move cells' plane lists decide it: 0 miss, 1 hit, 2
// undecided (the caller scans all hull planes with the whole warp: one lane doing that alone held up the other 31)
__device__ __forceinline__ int beam_ray(const DevPack &pk, int a0, int a1, Vec3 frm, Vec3 to, Vec3 &hit) {
    const double d0 = to.x - frm.x, d1 = to.y - frm.y, d2 = to.z - frm.z;
    const int npax = 3 - a0 - a1;
    // the TCP hovers kHookDistance above the surface and the fan's plane lies 0.2 ahead: expect the entry half way
    Vec3 h = {frm.x + d0 * 0.5, frm.y + d1 * 0.5, frm.z + d2 * 0.5};
    double t_in, t_out;
    bool outside;
    int tried_cx = -1, tried_cy = -1;
    unsigned long long link = 0ull;
#pragma unroll 1
    for (int attempt = 0; attempt < kRayAttempts; ++attempt) {
        const double g0 = comp(h, a0), g1 = comp(h, a1);
        int cx = (int)floor((g0 - pk.mc_o0) * pk.mc_inv);
        int cy = (int)floor((g1 - pk.mc_o1) * pk.mc_inv);
        if (link == 0ull && (cx < 0 || cy < 0 || cx >= pk.mc_nx || cy >= pk.mc_ny)) break;
        uint2 entry;
        if (link != 0ull) {                              // a silhouette cell's deeper second blob follows its thin primary
            cx = tried_cx; cy = tried_cy;
            entry = make_uint2((unsigned)link, (unsigned)(link >> 32));
        } else {
            if (cx == tried_cx && cy == tried_cy) break;
            entry = __ldg(&pk.mc_entry[cy * pk.mc_nx + cx]);
        }
        tried_cx = cx; tried_cy = cy;
        const int n_planes = (int)(entry.y & 0xffffu);
        if (n_planes <= 0) break;
        const double2 *blob = pk.mc_blob + (size_t)entry.x * 2;
        const double2 abv = __ldg(blob), clv = __ldg(blob + 1), hpv = __ldg(blob + 2);
        link = (unsigned long long)__double_as_longlong(hpv.y);
        slab_serial(blob + 4, n_planes, frm, d0, d1, d2, t_in, t_out, outside);
        if (outside || t_in > t_out || t_in > 1.0 || t_out < 0.0) return 0;              // a miss proven by the subset
        if (!(t_in > -INFINITY)) { if (link != 0ull) continue; break; }
        h.x = frm.x + d0 * t_in; h.y = frm.y + d1 * t_in; h.z = frm.z + d2 * t_in;
        if (in_cell_region(pk, h, comp(h, a0), comp(h, a1), comp(h, npax), cx, cy, abv, clv, hpv)) {
            if (!(0.0 <= t_in)) return 0;
            hit = h;
            return 1;
        }
    }
    return 2;
}

// cKDTree.query(point, k = 1) over the front texel positions, by one lane: returns the slot.
// Block search over the nearest-texel grid that grows to what the best distance so far demands: every texel outside
// the block lies beyond the block's border in the principal plane, so the block's winner is the global one as soon as
// its (3-D) distance is below the border distance.  Hits lie on the hull, texels on the mesh: over the part's concave
// regions the nearest texel is centimetres away, and the block grows once to the radius the first winner sets.
__device__ __forceinline__ int nearest_texel(const DevPack &pk, int a0, int a1, Vec3 p) {
    const double q0 = comp(p, a0), q1 = comp(p, a1);
    const int c0 = min(max((int)floor((q0 - pk.nn_o0) * pk.nn_inv), 0), pk.nn_nx - 1);
    const int c1 = min(max((int)floor((q1 - pk.nn_o1) * pk.nn_inv), 0), pk.nn_ny - 1);
    int R = 1;
#pragma unroll 1
    for (int round = 0; round < 12; ++round) {
        const int xa = max(c0 - R, 0), xb = min(c0 + R, pk.nn_nx - 1);
        const int ya = max(c1 - R, 0), yb = min(c1 + R, pk.nn_ny - 1);
        double best = INFINITY;
        long long arg = -1;
        for (int y = ya; y <= yb; ++y) {
            const int i0 = __ldg(&pk.nn_start[y * pk.nn_nx + xa]), i1 = __ldg(&pk.nn_start[y * pk.nn_nx + xb + 1]);
            for (int i = i0; i < i1; ++i) {
                const double2 xy = __ldg(pk.nn_pos + 2 * i), zs = __ldg(pk.nn_pos + 2 * i + 1);
                const double dx = xy.x - p.x, dy = xy.y - p.y, dz = zs.x - p.z;
                const double d = dx * dx + dy * dy + dz * dz;
                const long long slot = __double_as_longlong(zs.y);
                if (d < best || (d == best && slot < arg)) { best = d; arg = slot; }
            }
        }
        double m = INFINITY;
        if (xa > 0) m = fmin(m, q0 - (pk.nn_o0 + xa * pk.nn_cell));
        if (xb < pk.nn_nx - 1) m = fmin(m, (pk.nn_o0 + (xb + 1) * pk.nn_cell) - q0);
        if (ya > 0) m = fmin(m, q1 - (pk.nn_o1 + ya * pk.nn_cell));
        if (yb < pk.nn_ny - 1) m = fmin(m, (pk.nn_o1 + (yb + 1) * pk.nn_cell) - q1);
        if (arg >= 0 && m == INFINITY) return __ldg(&pk.nn_rep_slot[(int)arg]);      // the block is the whole grid
        m -= 1e-9;
        if (arg >= 0 && m > 0.0 && best < m * m) return __ldg(&pk.nn_rep_slot[(int)arg]);
        if (m == INFINITY) return -1;                                                 // no texel at all
        R = arg < 0 ? 2 * R + 1 : max(R + 1, (int)((sqrt(best) + 2e-9) * pk.nn_inv) + 2);
    }
    // (not reached with a sane grid: 12 rounds of a radius that at least doubles cover 4096 cells) scan everything
    double best = INFINITY;
    long long arg = -1;
    const int total = __ldg(&pk.nn_start[pk.nn_nx * pk.nn_ny]);
    for (int i = 0; i < total; ++i) {
        const double2 xy = __ldg(pk.nn_pos + 2 * i), zs = __ldg(pk.nn_pos + 2 * i + 1);
        const double dx = xy.x - p.x, dy = xy.y - p.y, dz = zs.x - p.z;
        const double d = dx * dx + dy * dy + dz * dz;
        const long long slot = __double_as_longlong(zs.y);
        if (d < best || (d == best && slot < arg)) { best = d; arg = slot; }
    }
    return arg >= 0 ? __ldg(&pk.nn_rep_slot[(int)arg]) : -1;
}

// Returns (warp-uniform) like stamp(): newly painted texels (RGB) / thickness units removed (HSI), |union of valid
// pixels| over the five shots (robot.py:423-425), whether a flip bit changed.  `last` = the environment's mask of the
// previous shot's texels in global memory (read and rewritten word by word; an all-miss shot leaves it alone:
// Part.paint returns early, bullet_paint_wrapper.py:563-564).
template <int COLOR, typename WS, typename BITS>
__device__ __forceinline__ void stamp_normal(const DevPack &pk, const DevConfig &cfg, const Ax &ax, const BITS &bits, int16_t *thick,
                                             unsigned *grid_cnt, unsigned *last, int lane, WS &ws, NormalScratch &ns, int &n_new_out,
                                             int &n_possible_out, bool &dirty_out) {
    const int nw = pk.n_words;
    for (int w = lane; w < nw; w += 32) ns.possible[w] = 0u;
    int n_new = 0;
    unsigned any = 0;
    const bool init_painted = (pk.status_init == kPainted);
#pragma unroll 1
    for (int s = 0; s < NS; ++s) {
        for (int w = lane; w < nw; w += 32) ns.shot_mask[w] = 0u;
        __syncwarp();
        const Vec3 pose = {ns.pos[s][0], ns.pos[s][1], ns.pos[s][2]};
        const Vec3 center = {ws.mv.centers[s][0], ws.mv.centers[s][1], ws.mv.centers[s][2]};
        int hits = 0;
        for (int b0 = 0; b0 < cfg.n_beams; b0 += 32) {
            const int b = b0 + lane;
            const bool live = b < cfg.n_beams;
            Vec3 dst = pose, hit = pose;
            int code = 0;
            if (live) {
                dst = transform_point(pose, ns.quat[s], __ldg(&cfg.beam_plain[3 * b]), __ldg(&cfg.beam_plain[3 * b + 1]),
                                      __ldg(&cfg.beam_plain[3 * b + 2]));
                code = beam_ray(pk, ax.a0, ax.a1, pose, dst, hit);
            }
            // beams no plane list decided: the serial slab test over all hull planes, the whole warp on one beam at a time
            unsigned undecided = __ballot_sync(kFull, code == 2);
            while (undecided) {
                const int src = __ffs(undecided) - 1;
                undecided &= undecided - 1;
                const double d0 = __shfl_sync(kFull, dst.x, src) - pose.x, d1 = __shfl_sync(kFull, dst.y, src) - pose.y,
                             d2 = __shfl_sync(kFull, dst.z, src) - pose.z;
                unsigned args;
                const SlabResult r = slab_pass_all<32>(reinterpret_cast<const double2 *>(pk.planes), pk.n_planes, pose, d0, d1, d2,
                                                       make_grp<32>(lane), &args);
                if (lane == src) {
                    code = (r.outside || !(r.t_in <= r.t_out && 0.0 <= r.t_in && r.t_in <= 1.0)) ? 0 : 1;
                    hit.x = pose.x + d0 * r.t_in; hit.y = pose.y + d1 * r.t_in; hit.z = pose.z + d2 * r.t_in;
                }
            }
            if (!live) continue;
            int slot = -1;
            if (code == 1) slot = nearest_texel(pk, ax.a0, ax.a1, hit);
            ns.beam_slot[b] = slot >= 0 ? (uint16_t)slot : (uint16_t)0xFFFF;
            if (slot >= 0) {
                hits++;
                atomicOr(&ns.shot_mask[slot >> 5], 1u << (slot & 31));
                if (COLOR == 1) {     // minkowski_distance(texel, centre) (bullet_paint_wrapper.py:421-423)
                    const double ex = fabs(center.x - __ldg(&pk.tx[slot])), ey = fabs(center.y - __ldg(&pk.ty[slot])),
                                 ez = fabs(center.z - __ldg(&pk.tz[slot]));
                    ns.beam_q[b] = sqrt((ex * ex + ey * ey) + ez * ez);
                }
            }
        }
        hits = __reduce_add_sync(kFull, hits);
        __syncwarp();
        if (hits == 0) continue;                       // `if not points: return [], 0`
        double rmax = 0.0;
        if (COLOR == 1) {
            double m = -1.0;
            for (int b = lane; b < cfg.n_beams; b += 32)
                if (ns.beam_slot[b] != 0xFFFF) m = fmax(m, ns.beam_q[b]);
            rmax = warp_max(m);
        }
        for (int w = lane; w < nw; w += 32) {
            const unsigned m = ns.shot_mask[w];
            const unsigned prev = last[w];
            last[w] = m;                               // _last_painted_pixels = affected_pixels (:576)
            ns.possible[w] |= m & ~prev;               // valid_pixels (:575)
            if (m == 0u) continue;
            const unsigned old = bits.ld(w);
            unsigned flipped = 0u;
            if (COLOR == 0) {                          // RGBColorHandler.change_pixels (:367-375): repaints count 0
                const unsigned painted_before = init_painted ? ~old : old;
                flipped = m & ~painted_before;
                n_new += __popc(flipped);
            } else {                                   // HSIColorHandler.change_pixels (:420-434), once per beam hit
                unsigned mm = m;
                while (mm) {
                    const int bit = __ffs(mm) - 1;
                    mm &= mm - 1;
                    const int slot = w * 32 + bit;
                    int times = 0;
                    double dist = 0.0;
                    for (int b = 0; b < cfg.n_beams; ++b)
                        if (ns.beam_slot[b] == (uint16_t)slot) { times++; dist = ns.beam_q[b]; }
                    const double ratio = dist / rmax;
                    const int quantity = (int)(kHsiTargetMax * (1.0 - ratio * ratio)) + 1;
                    const int v0 = (int)__ldcg(&thick[slot]);
                    int v = v0;
                    for (int k = 0; k < times && v > 0; ++k) { v -= quantity; n_new += quantity; }
                    if (v != v0) {
                        __stcg(&thick[slot], (int16_t)v);
                        if (v0 == kPainted) flipped |= 1u << bit;     // values only decrease: 255 is left once
                    }
                }
            }
            if (flipped) {
                bits.st(w, old | flipped);
                any |= flipped;
                if (grid_cnt) {
                    unsigned f = flipped;
                    while (f) {
                        const int bit = __ffs(f) - 1;
                        f &= f - 1;
                        atomicAdd(grid_cnt + __ldg(&pk.gcell[w * 32 + bit]), 1u);
                    }
                }
            }
        }
        __syncwarp();
    }
    int n_possible = 0;
    for (int w = lane; w < nw; w += 32) n_possible += __popc(ns.possible[w]);
    n_new_out = __reduce_add_sync(kFull, n_new);
    n_possible_out = __reduce_add_sync(kFull, n_possible);
    dirty_out = __any_sync(kFull, any != 0u);
    __syncwarp();
}

// ------------------------------------------------------------------------------ kernels
// Robot._get_actions (robot.py:302-329): action -> direction, five guided sub-steps.
// G lanes per environment (the plane / vertex / triangle lists of a sub-step are short).
template <int G, bool AX12>
__device__ __forceinline__ void move_body(const DevPack &pk, const DevConfig &cfg, const EnvArrays &ea, int env, int row, const void *actions) {
    const Ax ax = make_ax<AX12>(pk.axis0, pk.axis1);
    const int lane = threadIdx.x & 31;
    const Grp grp = make_grp<G>(lane);
    PAINTRL_PROF_BEGIN(env, 0, 15)
    PAINTRL_TRACE_MARK(env, 0, grp.gl == 0);
    PAINTRL_TRACE_SM(env, 6, grp.gl == 0);
    // the fields of the record this phase reads: pose, quaternion, turning angle, off-part state
    EnvState *gst = &ea.states[env];
    const double2 s0 = reinterpret_cast<const double2 *>(gst)[0], s1 = reinterpret_cast<const double2 *>(gst)[1],
                  s2 = reinterpret_cast<const double2 *>(gst)[2];
    const double quat_w = gst->quat[3], last_angle = gst->last_angle;
    int term_counter = gst->term_counter, flags = gst->flags;

    // ---- action -> direction (robot_gym_env.py:342-347, robot.py:390-398, 352-358)
    double u1, u2, new_angle;
    if (cfg.action_mode == 0) {
        long long a = reinterpret_cast<const long long *>(actions)[row];
        int ai = (int)min(max(a, 0ll), (long long)cfg.discrete_granularity);   // out-of-range actions are clipped, not rejected (robot.py:390-393)
        u1 = __ldg(&cfg.discrete_table[3 * ai]);
        u2 = __ldg(&cfg.discrete_table[3 * ai + 1]);
        new_angle = __ldg(&cfg.discrete_table[3 * ai + 2]);
    } else {
        const double *a = reinterpret_cast<const double *>(actions) + (size_t)row * cfg.action_shape;
        double a0 = a[0];
        if (!(-1.0 <= a0 && a0 <= 1.0)) a0 = a0 < -1.0 ? -1.0 : 1.0;   // robot.py:391-393 (a NaN ends up at 1 there too)
        if (cfg.action_shape == 1) {
            double phi = (a0 + 1.0) * kPi;
            u1 = cos(phi);
            u2 = sin(phi);
        } else {
            double a1v = a[1];
            if (!(-1.0 <= a1v && a1v <= 1.0)) a1v = a1v < -1.0 ? -1.0 : 1.0;
            double phi = atan2(a1v, a0);
            double x = fabs(a0), y = fabs(a1v);
            if (x == 0.0 && y == 0.0) { u1 = x; u2 = y; }
            else { double m = fmax(x, y); u1 = m * cos(phi); u2 = m * sin(phi); }
        }
        double da1 = u1 * kStepSize, da2 = u2 * kStepSize;
        new_angle = (da1 != 0.0) ? atan(fabs(da2 / da1)) : kPi / 2;
    }
    const double delta_axis1 = u1 * kStepSize, delta_axis2 = u2 * kStepSize;
    const double angle_diff = fabs(new_angle - last_angle);
    const int counter_before = term_counter;

    // ---- Robot._get_actions: 5 guided sub-steps (robot.py:302-329, bullet_paint_wrapper.py:865-880)
    Vec3 cur_p = {s0.x, s0.y, s1.x};
    double quat[4] = {s1.y, s2.x, s2.y, quat_w};
    Vec3 cur_n = tcp_orn_norm(cur_p, quat);
    const double delta1 = delta_axis1 / kPaintPerAction, delta2 = delta_axis2 / kPaintPerAction;
    const double delta2_scaled = delta2 * pk.lwr;
    int counts = 0;                                  // bits 8..15 full plane scans, 16..23 verify passes
    unsigned miss_cache = ea.moves[env].miss_cache;
    bool miss_quat_valid = false;   // quat == quat_from_normal(cur_n) from an earlier miss of this step
    double *centers = &ea.moves[env].centers[0][0];
#pragma unroll 1
    for (int s = 0; s < kPaintPerAction; ++s) {
        Vec3 p = cur_p;
        add_comp(p, ax.a0, delta1);
        add_comp(p, ax.a1, delta2_scaled);
        Vec3 end = {p.x + cur_n.x, p.y + cur_n.y, p.z + cur_n.z};
        Vec3 hit, pos, center;
        CellRef ref;
        double2 vc0 = make_double2(0.0, 0.0), vc1 = vc0;
        const double *rec = nullptr;
        PAINTRL_PROF(s == 0 ? 0 : 1, grp.gl == 0);
        if (ray_test<G>(pk, ax, p, end, grp, hit, ref, vc0, vc1, counts, miss_cache, delta1, delta2_scaled,
                        s + 1 < kPaintPerAction PAINTRL_PROF_PASS))
            rec = hook_triangle<G>(pk, ax, hit, ref, vc0, vc1, grp PAINTRL_PROF_PASS);
        PAINTRL_PROF(11, grp.gl == 0);
        if (rec) {
            // pose = hit + 0.1 n, orn = -n (bullet_paint_wrapper.py:529-530); quaternion and shot-centre
            // offset of -n come from the record (computed by the host with these same operations)
            const double2 *t = reinterpret_cast<const double2 *>(rec + 12);   // [12] inv, [13..15] n, [16..19] q, [20..22] off
            const double2 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2), t3 = __ldg(t + 3), t4 = __ldg(t + 4),
                          t5 = __ldg(t + 5);
            const double nx = t0.y, ny = t1.x, nz = t1.y;
            pos.x = hit.x + nx * kHookDistance;
            pos.y = hit.y + ny * kHookDistance;
            pos.z = hit.z + nz * kHookDistance;
            quat[0] = t2.x; quat[1] = t2.y; quat[2] = t3.x; quat[3] = t3.y;
            center.x = t4.x + pos.x; center.y = t4.y + pos.y; center.z = t5.x + pos.z;   // robot.py:277-278
            cur_n.x = -nx; cur_n.y = -ny; cur_n.z = -nz;
            flags |= kFlagLastOnPart;
            miss_quat_valid = false;
        } else {
            if (!miss_quat_valid) { quat_from_normal(cur_n, quat); miss_quat_valid = true; }
            pos = transform_point(cur_p, quat, delta2, delta1, 0.0);   // robot.py:317 (sic)
            center = transform_point(pos, quat, 0.0, 0.0, 0.1);        // robot.py:277-278
            if (flags & kFlagLastOnPart) {                              // robot.py:292-300
                flags &= ~kFlagLastOnPart;
            } else {
                term_counter += 1;
                if (term_counter > kNotOnPartTerminateSteps) flags |= kFlagTerminate;
            }
        }
        if (grp.gl == 0) { centers[3 * s] = center.x; centers[3 * s + 1] = center.y; centers[3 * s + 2] = center.z; }
        if (ea.shots && grp.gl == 0) {      // normal paint method: the beam fan of shot s is cast from this pose
            ShotPoses *sp = &ea.shots[env];
            sp->pos[s][0] = pos.x; sp->pos[s][1] = pos.y; sp->pos[s][2] = pos.z;
            sp->quat[s][0] = quat[0]; sp->quat[s][1] = quat[1]; sp->quat[s][2] = quat[2]; sp->quat[s][3] = quat[3];
        }
        cur_p = pos;
        PAINTRL_PROF(12, grp.gl == 0);
    }
    if (grp.gl == 0) {
        reinterpret_cast<double2 *>(gst)[0] = make_double2(cur_p.x, cur_p.y);
        reinterpret_cast<double2 *>(gst)[1] = make_double2(cur_p.z, quat[0]);
        reinterpret_cast<double2 *>(gst)[2] = make_double2(quat[1], quat[2]);
        gst->quat[3] = quat[3];
        reinterpret_cast<double2 *>(&gst->last_angle)[0] = make_double2(new_angle, angle_diff);
        gst->term_counter = term_counter;
        gst->flags = flags;
        ea.moves[env].counts = counts | (term_counter - counter_before);
        ea.moves[env].miss_cache = miss_cache;
        // publish: this lane wrote the record and the move output; the paint kernel's warp for this
        // environment acquires the flag instead of waiting for the whole grid
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ea.ready + env), "r"(1u) : "memory");
    }
    PAINTRL_PROF(13, grp.gl == 0);
#ifdef PAINTRL_PROFILE
    if (lane == 0) prof_row[14] = (unsigned)(counts | (term_counter - counter_before));
#endif
    PAINTRL_TRACE_MARK(env, 1, grp.gl == 0);
#ifdef PAINTRL_TRACE
    if (grp.gl == 0 && env < 65536) g_trace[env][6] |= (unsigned long long)(unsigned)(counts | (term_counter - counter_before)) << 16;
#endif
}

template <int G, int MINB, bool AX12, bool SUBSET = false>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, MINB)
move_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, const void *actions, EnvSel sel) {
    // programmatic dependent launch: let the paint kernel's CTAs be scheduled as this grid drains
    asm volatile("griddepcontrol.launch_dependents;");
    const int k = (blockIdx.x * blockDim.x + threadIdx.x) / G;   // launched with 32, 64 or 128 threads per block
    int env;
    if (!step_env<SUBSET>(sel, k, num_envs, env)) return;
    move_body<G, AX12>(pk, cfg, ea, env, k, actions);
}

// ------------------------------------------------------------------------------ move, fast path
// The move phase as the batch overwhelmingly runs it: every ray is decided by its move cell's own plane list
// -- a miss proven by the list (1), or an entry point inside the cell's region (2a) -- within kRayAttempts
// cells, and the nearest vertex comes from the cell's candidates.  Everything else of ray_test / hook_triangle
// (the verify pass (2b), the full plane scan (3), the miss-cache pair, the vertex-grid search) is NOT compiled
// into this kernel: an environment that needs any of it leaves without having written anything and raises its
// hand-off flag to kReadyBailed; the paint warp of that environment then runs the generic move_body itself
// before it paints.  Same arithmetic, same order, same results as move_body on the path both share -- but
// without the cold paths' live ranges the kernel fits the register budget of ONE wave at 4096 environments
// (28 warps per SM), which the generic kernel (128 registers, 1.73 waves) does not.
constexpr unsigned kReadyMoved = 1u, kReadyBailed = 2u;

template <int G>
__device__ __forceinline__ const double *hook_triangle_cell(const DevPack &pk, const Ax &ax, const Vec3 &point, const CellRef &ref, double2 vc0,
                                                            double2 vc1, const Grp &g) {
    // the hit's move cell lists every vertex that can be nearest; a hit outside every cell region (rare: accepted by
    // the verify pass or found by the full scan) searches the vertex grid
    const unsigned rec = ref.blob ? nearest_vertex_cell<G>(point, ref, vc0, vc1, g)
                                  : nearest_vertex_grid_call<G>(vertex_grid_args(pk), ax.a0, ax.a1, point, g);
    if (rec == 0xFFFFFFFFu) return nullptr;
    const int deg = (int)(rec & 0xffu);
    const double *base = pk.trirec + (size_t)(rec >> 8) * kTriRec;
    if (deg <= 0) return nullptr;
    int pick = -1;
    double run_max = -INFINITY;
    int run_arg = -1;
    for (int b0 = 0; b0 < deg; b0 += G) {
        const int k = b0 + g.gl;
        bool inside = false;
        double m = -INFINITY;
        if (k < deg) {
            const double2 *t = reinterpret_cast<const double2 *>(base + (size_t)k * kTriRec);
            // the tail of the record (normal, quaternion, shot-centre offset) is read right after the pick:
            // bring its sectors in with the head's
            prefetch_l1(reinterpret_cast<const char *>(t) + 128);
            const double2 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2), t3 = __ldg(t + 3), t4 = __ldg(t + 4),
                          t5 = __ldg(t + 5), t6 = __ldg(t + 6);
            const double v2x = point.x - t0.x, v2y = point.y - t0.y, v2z = point.z - t1.x;
            const double d20 = npdot3(v2x, v2y, v2z, t1.y, t2.x, t2.y);
            const double d21 = npdot3(v2x, v2y, v2z, t3.x, t3.y, t4.x);
            const double d00 = t4.y, d01 = t5.x, d11 = t5.y, inv = t6.x;
            double bv = (d11 * d20 - d01 * d21) * inv;
            double bw = (d00 * d21 - d01 * d20) * inv;
            double bu = 1.0 - bv - bw;
            if (inv == 0.0) { bu = -1.0; bv = -1.0; bw = -1.0; }
            inside = (0.0 <= bu && bu <= 1.0 && 0.0 <= bv && bv <= 1.0 && 0.0 <= bw && bw <= 1.0);
            m = fmin(fmin(bu, bv), bw);
        }
        const unsigned in_mask = grp_ballot<G>(inside, g);
        if (in_mask) { pick = b0 + __ffs(in_mask) - 1; break; }
        const double cm = grp_max<G>(m, g);
        if (cm >= run_max) {   // `>=`: a later triangle wins ties (bullet_paint_wrapper.py:520)
            const unsigned eq = grp_ballot<G>(k < deg && m == cm, g);
            run_max = cm;
            run_arg = b0 + 31 - __clz(eq);
        }
    }
    if (pick < 0) pick = (run_max >= -1.0) ? run_arg : 0;
    return base + (size_t)pick * kTriRec;
}

// 0 miss, 1 hit (hit / ref / vc0 / vc1 set), 2 leave the fast path.  `miss_cache_ptr`: the environment's pair of hull
// planes that decided its last full plane scan (MoveOut::miss_cache, maintained by the generic path): a ray no move
// cell can decide -- the TCP has wandered off the part, its rays start outside the grid -- is usually proven a miss
// by that pair (any subset of the planes may prove a miss), so such environments stay on the fast path too.
#ifdef PAINTRL_PROFILE
__device__ unsigned long long g_fast_reasons[8];   // why rays left the fast path: 1 outside the grid, 2 empty cell, 3 no entering plane, 4 attempts used up, 5 no vertex candidates
#define PAINTRL_FAST_REASON(k) do { if (grp.gl == 0) atomicAdd(&g_fast_reasons[k], 1ull); } while (0)
#else
#define PAINTRL_FAST_REASON(k) do {} while (0)
#endif
template <int G>
__device__ __forceinline__ int ray_fast(const DevPack &pk, const Ax &ax, const Vec3 &frm, const Vec3 &to, const Grp &grp, Vec3 &hit,
                                        CellRef &ref, double2 &vc0, double2 &vc1, double pf0, double pf1, bool do_prefetch,
                                        const unsigned *miss_cache_ptr, int &path_counts, int &path_sizes) {
    // path_counts (read by the trace build only): bits 0..7 off-part sub-steps, 8..15 misses proven by the cached plane
    // pair, 16..23 verify passes, 24..30 cell attempts
    const double d0 = to.x - frm.x, d1 = to.y - frm.y, d2 = to.z - frm.z;
    const int npax = 3 - ax.a0 - ax.a1;
    Vec3 h = {frm.x + d0 * kHookDistance, frm.y + d1 * kHookDistance, frm.z + d2 * kHookDistance};
    SlabResult r;
    r.t_in = -INFINITY; r.t_out = INFINITY; r.outside = false;
    bool candidate = false;
    int why = 4;
    const double2 *sub = nullptr;      // the plane list of the last cell tried
    int n_sub = 0;
    int tried = -1;                    // index of the cell just tried (one register instead of two coordinates)
    unsigned long long link = 0ull;    // fallback blob of the cell just tried (offset | counts << 32), 0: none
#pragma unroll 1
    for (int attempt = 0; attempt < kRayAttempts; ++attempt) {
        path_counts += 1 << 24;
        const double g0 = comp(h, ax.a0), g1 = comp(h, ax.a1);
        int cell = tried;
        uint2 entry;
        if (link != 0ull) {
            // the cell just tried is a silhouette cell whose thin primary slab did not hold the entry point: its second
            // blob (deep slab, build_move_cells) comes next, whichever cell the provisional entry point fell into
            entry = make_uint2((unsigned)link, (unsigned)(link >> 32));
        } else {
            const int cx = (int)floor((g0 - pk.mc_o0) * pk.mc_inv);
            const int cy = (int)floor((g1 - pk.mc_o1) * pk.mc_inv);
            if (cx < 0 || cy < 0 || cx >= pk.mc_nx || cy >= pk.mc_ny) { why = 1; break; }
            cell = cy * pk.mc_nx + cx;
            if (cell == tried) break;                        // the same cell again: same list, same result
            entry = __ldg(&pk.mc_entry[cell]);
        }
        tried = cell;
        const int n_planes = (int)(entry.y & 0xffffu), n_verts = (int)(entry.y >> 16);
        if (n_planes <= 0) { why = 2; break; }
#ifdef PAINTRL_TRACE
        path_sizes = max(path_sizes & 0xff, min(n_planes, 255)) | (max(path_sizes >> 8, min(n_verts, 255)) << 8);
#endif
        const double2 *blob = pk.mc_blob + (size_t)entry.x * 2;
        sub = blob + 4; n_sub = n_planes;
        const double2 abv = __ldg(blob), clv = __ldg(blob + 1), hpv = __ldg(blob + 2);
        link = (unsigned long long)__double_as_longlong(hpv.y);
        if (grp.gl < n_verts) {
            vc0 = __ldg(blob + 2 * (2 + n_planes + grp.gl));
            vc1 = __ldg(blob + 2 * (2 + n_planes + grp.gl) + 1);
        }
        if (do_prefetch && attempt == 0) {
            const int px = (int)floor((g0 + pf0 - pk.mc_o0) * pk.mc_inv);
            const int py = (int)floor((g1 + pf1 - pk.mc_o1) * pk.mc_inv);
            if (px >= 0 && py >= 0 && px < pk.mc_nx && py < pk.mc_ny && py * pk.mc_nx + px != cell) {
                const uint2 pe = __ldg(&pk.mc_entry[py * pk.mc_nx + px]);
                const int sectors = 2 + (int)(pe.y & 0xffffu) + (int)(pe.y >> 16);
                const char *pb = reinterpret_cast<const char *>(pk.mc_blob + (size_t)pe.x * 2);
                if (G == 32) { if (grp.gl * 128 < sectors * 32) prefetch_l1(pb + grp.gl * 128); }
                else for (int o = grp.gl * 128; o < sectors * 32; o += G * 128) prefetch_l1(pb + o);
            }
        }
        r = slab_pass<G>(blob + 4, n_planes, frm, d0, d1, d2, grp);
        if (r.outside || r.t_in > r.t_out || r.t_in > 1.0 || r.t_out < 0.0) return 0;   // (1)
        candidate = false;
        if (!(r.t_in > -INFINITY)) { if (link != 0ull) continue; why = 3; break; }
        candidate = true;
        h.x = frm.x + d0 * r.t_in; h.y = frm.y + d1 * r.t_in; h.z = frm.z + d2 * r.t_in;
        if (in_cell_region_idx(pk, comp(h, ax.a0), comp(h, ax.a1), comp(h, npax), cell, abv, clv, hpv)) {   // (2a)
            if (!(0.0 <= r.t_in)) return 0;        // with (1) passed this is the serial scan's hit test
            if (n_verts <= 0) { PAINTRL_FAST_REASON(5); return 2; }
            ref.blob = blob; ref.n_planes = n_planes; ref.n_verts = n_verts;
            hit = h;
            return 1;
        }
    }
    // (1) again with the pair of planes that decided this environment's last full scan, as ray_test does
    path_counts += 1 << 8;
    if (pair_proves_miss(pk, *miss_cache_ptr, r, candidate, frm, d0, d1, d2)) return 0;
    if (candidate) {
        path_counts += 1 << 16;
        // (2b) the entry point of the last list lies in the region of none of the cells tried (a ray grazing a sharp
        // feature of the hull): one division-free pass over all hull planes decides whether that list was enough.
        // Out-of-line, rolled: a handful of rays in a million come here, but a step is as slow as its slowest environment.
        if (near_violations_rolled<G>(reinterpret_cast<const double2 *>(pk.planes), pk.n_planes, h, grp) ==
            near_violations_rolled<G>(sub, n_sub, h, grp)) {
            if (!(r.t_in <= r.t_out && 0.0 <= r.t_in && r.t_in <= 1.0)) return 0;
            ref.blob = nullptr;          // the hit lies outside every cell region: its nearest vertex comes from the vertex grid
            hit = h;
            return 1;
        }
        why = 6;
    }
    PAINTRL_FAST_REASON(why);
    (void)why;
    return 2;
}

// FUSED (G == 32, called by the fused step kernel's warp): the record is read from and written to the warp's shared
// scratch `sst` / `smv` instead of global memory and no flag is published; returns true when the environment left
// the fast path (then nothing of `sst` has been changed).
template <int G, bool AX12, bool DISCRETE, bool FUSED>
__device__ __forceinline__ bool move_fast_body(const DevPack &pk, const DevConfig &cfg, const EnvArrays &ea, int env, int row, const void *actions,
                                               EnvState *sst, MoveOut *smv) {
    const Ax ax = make_ax<AX12>(pk.axis0, pk.axis1);
    const int lane = threadIdx.x & 31;
    const Grp grp = make_grp<G>(lane);
    PAINTRL_TRACE_MARK(env, 0, grp.gl == 0);
    PAINTRL_TRACE_SM(env, 6, grp.gl == 0);
    EnvState *gst = FUSED ? sst : &ea.states[env];
    Vec3 cur_p, cur_n;
    double last_angle;
    int term_counter = gst->term_counter, flags = gst->flags;
    {
        const double2 s0 = reinterpret_cast<const double2 *>(gst)[0], s1 = reinterpret_cast<const double2 *>(gst)[1],
                      s2 = reinterpret_cast<const double2 *>(gst)[2];
        const double q[4] = {s1.y, s2.x, s2.y, gst->quat[3]};
        last_angle = gst->last_angle;
        cur_p.x = s0.x; cur_p.y = s0.y; cur_p.z = s1.x;
        cur_n = tcp_orn_norm(cur_p, q);
    }
    // ---- action -> direction (robot_gym_env.py:342-347, robot.py:390-398, 352-358), as in move_body
    double u1, u2, new_angle;
    if (DISCRETE) {
        const long long a = reinterpret_cast<const long long *>(actions)[row];
        const int ai = (int)min(max(a, 0ll), (long long)cfg.discrete_granularity);
        u1 = __ldg(&cfg.discrete_table[3 * ai]);
        u2 = __ldg(&cfg.discrete_table[3 * ai + 1]);
        new_angle = __ldg(&cfg.discrete_table[3 * ai + 2]);
    } else {
        const double *a = reinterpret_cast<const double *>(actions) + (size_t)row * cfg.action_shape;
        double a0 = a[0];
        if (!(-1.0 <= a0 && a0 <= 1.0)) a0 = a0 < -1.0 ? -1.0 : 1.0;
        if (cfg.action_shape == 1) {
            const double phi = (a0 + 1.0) * kPi;
            u1 = cos(phi);
            u2 = sin(phi);
        } else {
            double a1v = a[1];
            if (!(-1.0 <= a1v && a1v <= 1.0)) a1v = a1v < -1.0 ? -1.0 : 1.0;
            const double phi = atan2(a1v, a0);
            const double x = fabs(a0), y = fabs(a1v);
            if (x == 0.0 && y == 0.0) { u1 = x; u2 = y; }
            else { const double m = fmax(x, y); u1 = m * cos(phi); u2 = m * sin(phi); }
        }
        const double da1 = u1 * kStepSize, da2 = u2 * kStepSize;
        new_angle = (da1 != 0.0) ? atan(fabs(da2 / da1)) : kPi / 2;
    }
    const double delta1 = (u1 * kStepSize) / kPaintPerAction, delta2 = (u2 * kStepSize) / kPaintPerAction;
    const int counter_before = term_counter;
    int path_counts = 0, path_sizes = 0;   // trace build: largest plane / vertex list met
    double quat[4];
    MoveOut *mv = FUSED ? smv : &ea.moves[env];
    double *centers = &mv->centers[0][0];
#pragma unroll 1
    for (int s = 0; s < kPaintPerAction; ++s) {
        const double delta2_scaled = delta2 * pk.lwr;
        Vec3 p = cur_p;
        add_comp(p, ax.a0, delta1);
        add_comp(p, ax.a1, delta2_scaled);
        const Vec3 end = {p.x + cur_n.x, p.y + cur_n.y, p.z + cur_n.z};
        Vec3 hit, pos, center;
        CellRef ref;
        double2 vc0 = make_double2(0.0, 0.0), vc1 = vc0;
        const double *rec = nullptr;
        const int code = ray_fast<G>(pk, ax, p, end, grp, hit, ref, vc0, vc1, delta1, delta2_scaled, s + 1 < kPaintPerAction,
                                     &ea.moves[env].miss_cache, path_counts, path_sizes);
        if (code == 2) {
            // not decidable on the fast path: nothing of this step has been published (the shot centres written so
            // far are rewritten by the generic pass); the environment's paint warp takes the move over
            if (!FUSED && grp.gl == 0)
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ea.ready + env), "r"(kReadyBailed) : "memory");
            PAINTRL_TRACE_MARK(env, 1, grp.gl == 0);
            return true;
        }
        if (code == 1) rec = hook_triangle_cell<G>(pk, ax, hit, ref, vc0, vc1, grp);
        if (rec) {
            const double2 *t = reinterpret_cast<const double2 *>(rec + 12);   // [12] inv, [13..15] n, [16..19] q, [20..22] off
            const double2 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2), t3 = __ldg(t + 3), t4 = __ldg(t + 4),
                          t5 = __ldg(t + 5);
            const double nx = t0.y, ny = t1.x, nz = t1.y;
            pos.x = hit.x + nx * kHookDistance;
            pos.y = hit.y + ny * kHookDistance;
            pos.z = hit.z + nz * kHookDistance;
            quat[0] = t2.x; quat[1] = t2.y; quat[2] = t3.x; quat[3] = t3.y;
            center.x = t4.x + pos.x; center.y = t4.y + pos.y; center.z = t5.x + pos.z;   // robot.py:277-278
            cur_n.x = -nx; cur_n.y = -ny; cur_n.z = -nz;
            flags |= kFlagLastOnPart;
        } else {
            path_counts += 1;
            quat_from_normal(cur_n, quat);                              // robot.py:313: the orientation of the kept normal
            pos = transform_point(cur_p, quat, delta2, delta1, 0.0);    // robot.py:317 (sic)
            center = transform_point(pos, quat, 0.0, 0.0, 0.1);         // robot.py:277-278
            if (flags & kFlagLastOnPart) {                              // robot.py:292-300
                flags &= ~kFlagLastOnPart;
            } else {
                term_counter += 1;
                if (term_counter > kNotOnPartTerminateSteps) flags |= kFlagTerminate;
            }
        }
        if (grp.gl == 0) { centers[3 * s] = center.x; centers[3 * s + 1] = center.y; centers[3 * s + 2] = center.z; }
        cur_p = pos;
    }
#ifdef PAINTRL_TRACE
    if (grp.gl == 0 && env < 65536) g_trace[env][6] |= ((unsigned long long)(unsigned)path_counts << 16) | ((unsigned long long)(unsigned)path_sizes << 48);
#endif
    (void)path_sizes;
    if (FUSED) __syncwarp();     // every lane read the record from the warp's shared scratch at the top; lane 0 rewrites it
    if (grp.gl == 0) {
        reinterpret_cast<double2 *>(gst)[0] = make_double2(cur_p.x, cur_p.y);
        reinterpret_cast<double2 *>(gst)[1] = make_double2(cur_p.z, quat[0]);
        reinterpret_cast<double2 *>(gst)[2] = make_double2(quat[1], quat[2]);
        gst->quat[3] = quat[3];
        reinterpret_cast<double2 *>(&gst->last_angle)[0] = make_double2(new_angle, fabs(new_angle - last_angle));
        gst->term_counter = term_counter;
        gst->flags = flags;
        mv->counts = term_counter - counter_before;
        if (!FUSED) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ea.ready + env), "r"(kReadyMoved) : "memory");
    }
    PAINTRL_TRACE_MARK(env, 1, grp.gl == 0);
    return false;
}

#ifndef PAINTRL_MOVE_FAST_MINB
#define PAINTRL_MOVE_FAST_MINB 7
#endif
template <int G, bool AX12, bool DISCRETE, bool SUBSET = false>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, PAINTRL_MOVE_FAST_MINB)
move_fast_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, const void *actions, EnvSel sel) {
    asm volatile("griddepcontrol.launch_dependents;");
    const int k = (blockIdx.x * blockDim.x + threadIdx.x) / G;
    int env;
    if (!step_env<SUBSET>(sel, k, num_envs, env)) return;
    if (cfg.debug_bail_mod > 0 && env % cfg.debug_bail_mod == 0) {      // tests: exercise the hand-over to the paint warp
        if ((threadIdx.x & (G - 1)) == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(ea.ready + env), "r"(kReadyBailed) : "memory");
        return;
    }
    move_fast_body<G, AX12, DISCRETE, false>(pk, cfg, ea, env, k, actions, nullptr, nullptr);
}

// The generic move of ONE environment, called by its paint warp when the fast move kernel bailed out.  Deliberately a
// real call (noinline) on a copy of the kernel arguments in global memory: the cold path's registers and spills stay
// out of the paint kernel's own allocation.  `row`: the environment's row of the actions.
struct ColdArgs { DevPack pk; DevConfig cfg; EnvArrays ea; };
__device__ __noinline__ void move_generic_cold(const ColdArgs *ca, int env, int row, const void *actions) {
    move_body<32, false>(ca->pk, ca->cfg, ca->ea, env, row, actions);
}

// Everything after the move: stamp, score, observe, auto-reset.  (STAGED) the environment's flip bits
// come in through a TMA bulk copy issued before the warp waits for its environment's hand-off flag and go
// back the same way; the record and the move kernel's output follow the flag with L2 loads.  State is indexed by
// `env`, the I/O buffers of `io` by `row` (the same in a whole-batch step).
template <int COLOR, bool STAGED, bool AX12, bool FUSED = false, bool DISCRETE = false, bool NORMAL = false>
__device__ __forceinline__ void paint_body(const DevPack &pk, const DevConfig &cfg, const EnvArrays &ea, int env, int row, const StepIO &io,
                                           WarpScratch<STAGED> &ws, const ColdArgs *cold, NormalScratch *ns = nullptr) {
    const Ax ax = make_ax<AX12>(pk.axis0, pk.axis1);
    typedef WarpScratch<STAGED> WS;
    const int lane = threadIdx.x & 31;
    PAINTRL_PROF_BEGIN(env, 15, 32)
    PAINTRL_TRACE_MARK(env, 2, lane == 0);
    PAINTRL_TRACE_SM(env, 7, lane == 0);
    unsigned *gbits = bits_of(pk, ea, env), *grid_cnt = grid_cnt_of(pk, ea, env);
    int16_t *thick = thick_of(pk, ea, env);
    const unsigned plane_bytes = (unsigned)pk.n_words_pad * 4u;
    // The bit-plane copy in, issued exactly once per step before mbar_wait.  One-kernel step with start_order: the
    // plane is not needed before the stamp, so its copy goes out after the move phase (before the generic move when
    // the fast one bails) instead of queueing in front of the record load and the move's first table lookups.
    const bool late_copy = FUSED && STAGED && !NORMAL && cfg.start_order;
    auto issue_copy = [&]() {
        if (STAGED && lane == 0) {
            mbar_init(&ws.bar, 1);
            mbar_expect_tx(&ws.bar, plane_bytes);
            bulk_g2s(ws.sbits, gbits, plane_bytes, &ws.bar);   // not written by the move phase
        }
    };
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
    if (FUSED && !cfg.start_order) l2_prefetch_tables(pk, tid, nthreads);
    if (!late_copy) issue_copy();
    // Launched with programmatic stream serialization: this grid's CTAs start as soon as every CTA of the
    // move kernel has started, and each warp waits only for ITS environment's move phase (acquire of the
    // flag the move warp released) -- not for the whole grid: a slow environment of the move phase delays
    // nobody else, and the paint phase fills the SMs the move kernel's last wave leaves idle.
    int bailed = 0;
    if (FUSED) {
        // One warp runs the whole step of its environment: the record comes into the scratch, the fast move phase
        // works on that copy (the bit-plane copy issued above lands meanwhile), the paint phase continues on it.
        if (lane < 8) reinterpret_cast<double2 *>(&ws.st)[lane] = __ldcg(reinterpret_cast<const double2 *>(&ea.states[env]) + lane);
        // start_order: the record load is every warp's first dependent load, so it goes out before the sweep's prefetches
        if (cfg.start_order) l2_prefetch_tables(pk, tid, nthreads);
        __syncwarp();
        if (cfg.debug_bail_mod > 0 && env % cfg.debug_bail_mod == 0) bailed = 1;      // tests: force the generic path
        else bailed = move_fast_body<32, AX12, DISCRETE, true>(pk, cfg, ea, env, row, io.actions, &ws.st, &ws.mv) ? 1 : 0;
        __syncwarp();
        // after the move, not inside it: a copy issued inside the sub-step loop keeps its operands live there (+40 / +96
        // bytes of spill stores / loads in the C2 kernel)
        if (late_copy) issue_copy();
    } else {
        // Launched with programmatic stream serialization: this grid's CTAs start as soon as every CTA of the
        // move kernel has started, and each warp waits only for ITS environment's move phase (acquire of the
        // flag the move warp released) -- not for the whole grid.
        if (lane == 0) {
            const unsigned *flag = ea.ready + env;
            unsigned v;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                if (v != 0u) break;
                __nanosleep(200);
            }
            // consume: the next step's move kernel (which starts after this grid has completed) raises it again.
            // No sequence number in the kernel arguments, so a captured step can be replayed from a CUDA graph.
            ea.ready[env] = 0u;
            bailed = (v == kReadyBailed);
        }
        bailed = __shfl_sync(kFull, bailed, 0);
    }
    if (bailed) {
        // the fast move phase could not decide one of this environment's rays from its move cell alone and wrote
        // nothing: run the generic move here (verify pass / full plane scan / vertex-grid search), then paint
        move_generic_cold(cold, env, row, io.actions);
        __threadfence();
        if (lane == 0) ea.ready[env] = 0u;      // move_body published 1: consumed
    }
    __syncwarp();
    PAINTRL_TRACE_MARK(env, 3, lane == 0);
    if (!FUSED || bailed) {
        // the record and the move output: L2 loads (another SM wrote them while this grid was already running)
        if (lane < 16) {
            const double2 *src = lane < 8 ? reinterpret_cast<const double2 *>(&ea.states[env]) + lane
                                          : reinterpret_cast<const double2 *>(&ea.moves[env]) + (lane - 8);
            double2 *dst = lane < 8 ? reinterpret_cast<double2 *>(&ws.st) + lane : reinterpret_cast<double2 *>(&ws.mv) + (lane - 8);
            *dst = __ldcg(src);
        }
        __syncwarp();
    }
    if (STAGED && !late_copy) mbar_wait(&ws.bar, 0);      // a late copy is waited for after the row ranks below
    PAINTRL_TRACE_MARK(env, 4, lane == 0);
    PAINTRL_PROF(16, lane == 0);
    const Bits<STAGED> bits = {gbits, ws.sbits};
    EnvState &st = ws.st;
    const Vec3 cur_p = {st.pose[0], st.pose[1], st.pose[2]};
    // 4-sector section / discrete observation: its per-row ranks only depend on the pose, so they are
    // looked up before the stamp and the TCP row's axis1 keys are prefetched into L1 meanwhile
    const bool fast4 = (cfg.obs_mode == 0 || cfg.obs_mode == 3) && cfg.obs_grad == 4;
    if (fast4) {
        row_ranks(pk, ax, comp(cur_p, ax.a0), lane, ws);
        const int prow = pose_row(pk, comp(cur_p, ax.a1));
        if (prow >= 0 && prow < pk.n_rows) {
            const int w0 = __ldg(&pk.row_word0[prow]), w1 = __ldg(&pk.row_word0[prow + 1]);
            const char *ky = reinterpret_cast<const char *>(axis_table(pk, ax.a1) + (size_t)w0 * 32);
            for (int k = lane; k < 2 * (w1 - w0); k += 32) prefetch_l1(ky + (size_t)k * 128);
        }
    }
    if (STAGED && late_copy) mbar_wait(&ws.bar, 0);
    PAINTRL_PROF(15, lane == 0);

    // ---- stamp the 5 shots (bullet_paint_wrapper.py:568-577)
    const bool has_last = (st.flags & kFlagHasLast) != 0;
    int n_new, n_possible;
    bool dirty;
    if (NORMAL) {
        // Robot.PAINT_METHOD == 'normal' (robot.py:414-417): the five beam fans instead of the five ball queries
        const double *src = reinterpret_cast<const double *>(&ea.shots[env]);
        for (int i = lane; i < kPaintPerAction * 7; i += 32) (&ns->pos[0][0])[i] = __ldcg(src + i);
        __syncwarp();
        stamp_normal<COLOR>(pk, cfg, ax, bits, thick, grid_cnt, ea.last_mask + (size_t)env * pk.n_words_pad, lane, ws, *ns, n_new, n_possible, dirty);
    } else {
        stamp<COLOR, STAGED>(pk, ax, bits, thick, grid_cnt, has_last, lane, ws, n_new, n_possible, dirty PAINTRL_PROF_PASS);
    }
    PAINTRL_PROF(19, lane == 0);

    // ---- robot.py:425-433, robot_gym_env.py:321-340 (every lane ends up with the same scalars).
    // The FP64 divisions of this block and of the normalised pose are independent of each other:
    // each is evaluated by one lane, all in the same instruction, and broadcast.
    int flags = st.flags | kFlagHasLast;
    const double succeeded = (COLOR == 0) ? (double)n_new : (double)n_new / 255.0;
    if ((ws.mv.counts & 0xf) >= kPaintPerAction && n_possible == 0) flags |= kFlagTerminate;
    const double radius = kPaintRadius;
    const double axis1_real = comp(cur_p, ax.a0), axis2_real = comp(cur_p, ax.a1);
    double rate, reward, turn, axis2_in, rel;
    {
        double num = succeeded, den = n_possible ? (double)n_possible : 1.0;    // lane 0: rate (robot.py:426)
        if (lane == 1) den = 100.0;                                             // reward (robot_gym_env.py:322)
        if (lane == 2) { num = st.angle_diff; den = kPi; }                      // turning penalty (:338)
        if (lane == 3) { num = axis2_real - pk.range1_min + radius; den = pk.range1_max - pk.range1_min + 2 * radius; }   // bullet_paint_wrapper.py:969
        if (lane == 4) { num = axis2_real - pk.range1_min; den = pk.range1_max - pk.range1_min; }                         // :845
        // 0 / den is +0 for these positive denominators; skipping it keeps the lanes whose numerator is 0
        // (nothing painted, no turn) out of the division's slow path
        double q = 0.0;
        if (num != 0.0) q = num / den;
        rate = n_possible ? __shfl_sync(kFull, q, 0) : 0.0;
        reward = __shfl_sync(kFull, q, 1);
        turn = __shfl_sync(kFull, q, 2);
        axis2_in = __shfl_sync(kFull, q, 3);
        rel = __shfl_sync(kFull, q, 4);
    }
    const double total_reward = st.total_reward + reward;
    double penalty = 0.2;
    if (cfg.overlap_penalty) penalty += 0.1 * (1 - rate);
    if (cfg.turning_penalty) penalty += 0.1 * turn;
    const double actual = reward - penalty;
    const int step_counter = st.step_counter + 1;
    // normalised pose, bullet_paint_wrapper.py:844-851, 965-978
    int gi;
    {
        const double scaled = rel * pk.grid_granularity;
        gi = !(scaled > -1.0) ? 0 : (scaled >= (double)pk.grid_granularity ? pk.grid_granularity - 1 : (int)scaled);
    }
    const double glo = __ldg(&pk.grid_lo[gi]), ghi = __ldg(&pk.grid_hi[gi]);
    PAINTRL_PROF(20, lane == 0);

    // ---- observation counts (robot_gym_env.py:358: computed even when done)
    int tot[4] = {0, 0, 0, 0}, open[4] = {0, 0, 0, 0};
    if (fast4) section4_counts(pk, ax, bits, cur_p, lane, ws, tot, open, true PAINTRL_PROF_PASS);

    // ---- second round of divisions: average reward (robot_gym_env.py:295), axis1 of the normalised pose, sector ratios
    double avg_reward, axis1_in, ratio;
    {
        double num = total_reward, den = (double)step_counter;
        if (lane == 1) { num = axis1_real - glo + radius; den = ghi - glo + 2 * radius; }
        int t = 1, o = 0;
        if (lane >= 2 && lane < 6) {
            t = lane == 2 ? tot[0] : (lane == 3 ? tot[1] : (lane == 4 ? tot[2] : tot[3]));
            o = lane == 2 ? open[0] : (lane == 3 ? open[1] : (lane == 4 ? open[2] : open[3]));
            num = (double)o; den = t ? (double)t : 1.0;
        }
        double q = 0.0;
        if (num != 0.0) q = num / den;
        ratio = t == 0 ? 0.0 : q;                        // lanes 2..5: sector s = lane - 2 (bullet_paint_wrapper.py:1057-1060)
        avg_reward = __shfl_sync(kFull, q, 0);
        axis1_in = (ghi - glo == 0.0) ? 0.0 : __shfl_sync(kFull, q, 1);
    }
    const double a1 = clip01(axis1_in), a2 = clip01(axis2_in);

    // ---- robot_gym_env.py:289-304 _termination
    const double max_pts = cfg.max_possible_point;
    const bool finished = !(max_pts > total_reward * 100);
    bool done, decided = false;
    if (avg_reward < cfg.expected_avg_reward && cfg.termination_mode != 0) {
        if (cfg.termination_mode == 1) { done = true; decided = true; }
        else if (total_reward < cfg.hybrid_threshold) { done = true; decided = true; }
    }
    if (!decided) done = finished || (flags & kFlagTerminate) || step_counter > cfg.episode_max_length - 1;

    // ---- write the observation (robot_gym_env.py:306-319)
    const bool resetting = done && cfg.auto_reset;
    double *obs = io.obs + (size_t)row * cfg.obs_dim;
    double *next_obs = io.next_obs ? io.next_obs + (size_t)row * cfg.obs_dim : nullptr;
    if (resetting) next_obs = nullptr;
    if (fast4) {
        if (lane >= 2 && lane < 6) {
            obs[lane - 2] = ratio;
            if (next_obs) next_obs[lane - 2] = ratio;
        }
        if (lane == 0) {
            if (cfg.obs_mode == 3) {   // discrete: robot_gym_env.py:101-103, 314-318
                const int position = (handle_pos(a1) + 1) * 22 + handle_pos(a2);
                const double v = 1.0 / position;
                obs[4] = v;
                if (next_obs) next_obs[4] = v;
            } else {
                obs[4] = a1; obs[5] = a2;
                if (next_obs) { next_obs[4] = a1; next_obs[5] = a2; }
            }
        }
    } else {
        write_observation(pk, ax, cfg, bits, grid_cnt, cur_p, lane, ws, obs, next_obs PAINTRL_PROF_PASS);
    }
    if (io.next_obs) next_obs = io.next_obs + (size_t)row * cfg.obs_dim;
    __syncwarp();
    PAINTRL_PROF(25, lane == 0);
    if (lane == 0) {
        io.reward[row] = reward;
        io.penalty[row] = penalty;
        io.actual[row] = actual;
        io.done[row] = done ? 1 : 0;
        if (io.new_texels) io.new_texels[row] = n_new;
        EnvStat *es = &ea.env_stats[env];       // no other thread touches this record: plain reductions, no return value
        if (done) atomicAdd(&es->episodes_ended, 1ull);
        if (n_possible) atomicAdd(&es->footprint_texels, (unsigned long long)n_possible);
        if (ws.mv.counts >> 8)   // full plane scans in the low half of the counter, verify passes in the high half
            atomicAdd(&es->full_scans, (unsigned long long)((ws.mv.counts >> 8) & 0xff) | ((unsigned long long)((ws.mv.counts >> 16) & 0xff) << 32));
        atomicAdd(&es->env_steps, 1ull);
        if (bailed) atomicAdd(&es->move_bailouts, 1ull);
        // the record
        st.last_center[0] = ws.mv.centers[NS - 1][0];
        st.last_center[1] = ws.mv.centers[NS - 1][1];
        st.last_center[2] = ws.mv.centers[NS - 1][2];
        st.flags = flags;
        st.total_reward = total_reward;
        st.step_counter = step_counter;
        if (!done) st.total_return += actual;
    }

    // ---- same-step auto-reset: `obs` keeps the terminal observation, `next_obs` gets reset()'s
    if (resetting) {
        int idx = io.reset_start_idx ? io.reset_start_idx[row] : auto_start_index(pk, cfg, env, st.episode);
        idx = min(max(idx, 0), pk.n_starts - 1);
        clear_planes(pk, bits, gbits, thick, grid_cnt, lane);
        if (ea.last_mask)
            for (int w = lane; w < pk.n_words_pad; w += 32) ea.last_mask[(size_t)env * pk.n_words_pad + w] = 0u;
        __syncwarp();
        if (lane == 0) state_reset(pk, st, idx);
        if (next_obs) {
            const double *src = pk.reset_obs + (size_t)idx * cfg.obs_dim;
            for (int i = lane; i < cfg.obs_dim; i += 32) next_obs[i] = __ldg(&src[i]);
        }
    } else if (STAGED && dirty) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) bulk_s2g(gbits, ws.sbits, plane_bytes);
    }
    __syncwarp();
    if (lane < 8) reinterpret_cast<double2 *>(&ea.states[env])[lane] = reinterpret_cast<const double2 *>(&st)[lane];
    if (STAGED && lane == 0) bulk_wait_read();
    PAINTRL_PROF(26, lane == 0);
    PAINTRL_TRACE_MARK(env, 5, lane == 0);
}

#ifndef PAINTRL_PAINT_OCC
#define PAINTRL_PAINT_OCC 28
#endif
template <int COLOR, bool STAGED, bool AX12, int WPB, bool SUBSET = false>
__global__ void __launch_bounds__(WPB * 32, (STAGED ? PAINTRL_PAINT_OCC : 16) / WPB)
paint_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, StepIO io, const ColdArgs *cold, EnvSel sel) {
    __shared__ WarpScratch<STAGED> scratch[WPB];
    const int warp = threadIdx.x >> 5;
    const int k = blockIdx.x * WPB + warp;
    int env;
    if (!step_env<SUBSET>(sel, k, num_envs, env)) return;
    paint_body<COLOR, STAGED, AX12>(pk, cfg, ea, env, k, io, scratch[warp], cold);
}

// Paint kernel of the normal paint method (staged plane, generic axes; one warp per block).
template <int COLOR, bool SUBSET = false>
__global__ void __launch_bounds__(32, 14)   // 15 KB of shared memory per warp: 14 warps per SM
paint_normal_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, StepIO io, const ColdArgs *cold, EnvSel sel) {
    __shared__ WarpScratch<true> scratch[1];
    __shared__ NormalScratch nscratch[1];
    const int k = blockIdx.x;
    int env;
    if (!step_env<SUBSET>(sel, k, num_envs, env)) return;
    paint_body<COLOR, true, false, false, false, true>(pk, cfg, ea, env, k, io, scratch[0], cold, &nscratch[0]);
}

// The whole step of one environment in one warp (batches that cannot fill the GPU twice over: the two-kernel step
// pays the move grid's drain before the paint grid's warps get their slots; here a warp goes straight on).
#ifndef PAINTRL_FUSED_WPB
#define PAINTRL_FUSED_WPB 1      // warps (= environments) per CTA of the one-kernel step
#endif
template <int COLOR, bool STAGED, bool AX12, bool DISCRETE, bool SUBSET = false>
__global__ void __launch_bounds__(32 * PAINTRL_FUSED_WPB, (STAGED ? PAINTRL_PAINT_OCC : 16) / PAINTRL_FUSED_WPB)
step_fused_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, StepIO io, const ColdArgs *cold, EnvSel sel) {
    __shared__ WarpScratch<STAGED> scratch[PAINTRL_FUSED_WPB];
    const int warp = threadIdx.x >> 5;
    const int k = blockIdx.x * PAINTRL_FUSED_WPB + warp;
    int env;
    if (!step_env<SUBSET>(sel, k, num_envs, env)) return;
    paint_body<COLOR, STAGED, AX12, true, DISCRETE>(pk, cfg, ea, env, k, io, scratch[warp], cold);   // sweeps the tables into L2
}

// PaintGymEnv.reset / Robot.reset(pose) for the listed environments, with their first observation.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
reset_kernel(DevPack pk, DevConfig cfg, EnvArrays ea, int num_envs, const int32_t *env_ids, int n, const int32_t *start_idx,
             const double *set_pos, const double *set_normal, double *obs_out, int mode /*0 reset, 1 set_pose*/) {
    const Ax ax = make_ax<false>(pk.axis0, pk.axis1);
    __shared__ WarpScratch<false> scratch[kWarpsPerBlock];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = blockIdx.x * kWarpsPerBlock + warp;
    if (k >= n) return;
    const int env = env_ids ? env_ids[k] : k;
    if ((unsigned)env >= (unsigned)num_envs) return;      // the host validates the list; never index out of bounds
    unsigned *gbits = bits_of(pk, ea, env), *grid_cnt = grid_cnt_of(pk, ea, env);
    int16_t *thick = thick_of(pk, ea, env);
    if (lane == 0) ea.ready[env] = 0u;                    // a hand-off flag left behind by a failed step launch
    EnvState st;
    load_state(&ea.states[env], st);
    if (mode == 0) {
        int idx = start_idx ? start_idx[k] : auto_start_index(pk, cfg, env, st.episode);
        idx = min(max(idx, 0), pk.n_starts - 1);
        clear_planes(pk, Bits<false>{gbits, nullptr}, gbits, thick, grid_cnt, lane);
        if (ea.last_mask)
            for (int w = lane; w < pk.n_words_pad; w += 32) ea.last_mask[(size_t)env * pk.n_words_pad + w] = 0u;
        state_reset(pk, st, idx);
    } else {
        robot_reset(st, set_pos + 3 * k, set_normal + 3 * k);
    }
    __syncwarp();
    const Bits<false> bits = {gbits, nullptr};
    Vec3 pose = {st.pose[0], st.pose[1], st.pose[2]};
    PAINTRL_PROF_BEGIN(65535, 0, 0)
    write_observation(pk, ax, cfg, bits, grid_cnt, pose, lane, scratch[warp], obs_out ? obs_out + (size_t)k * cfg.obs_dim : nullptr,
                      nullptr PAINTRL_PROF_PASS);
    store_state(&ea.states[env], st, lane);
}

// Observation of a fresh environment standing at each start point (paint_kernel's auto-reset
// copies it instead of scanning the cleared planes again).  `zero_bits` / `grid_cnt` are all-zero planes.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
reset_obs_kernel(DevPack pk, DevConfig cfg, unsigned *zero_bits, const unsigned *grid_cnt, double *table) {
    const Ax ax = make_ax<false>(pk.axis0, pk.axis1);
    __shared__ WarpScratch<false> scratch[kWarpsPerBlock];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = blockIdx.x * kWarpsPerBlock + warp;
    if (k >= pk.n_starts) return;
    const Bits<false> bits = {zero_bits, nullptr};
    Vec3 pose = {pk.start_pos[3 * k], pk.start_pos[3 * k + 1], pk.start_pos[3 * k + 2]};
    PAINTRL_PROF_BEGIN(65535, 0, 0)
    write_observation(pk, ax, cfg, bits, grid_cnt, pose, lane, scratch[warp], table + (size_t)k * cfg.obs_dim, nullptr PAINTRL_PROF_PASS);
}

// ------------------------------------------------------------------------------ state access
__global__ void get_state_kernel(DevPack pk, EnvArrays ea, int num_envs, const int32_t *env_ids, int n, int16_t *status_out,
                                 double *pose_out, double *quat_out, double *scalars_out) {
    const int k = blockIdx.y;
    const int env = env_ids ? env_ids[k] : k;
    if ((unsigned)env >= (unsigned)num_envs) return;
    if (status_out) {
        const unsigned *bits = bits_of(pk, ea, env);
        const int16_t *thick = thick_of(pk, ea, env);
        for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < pk.n_texels; p += gridDim.x * blockDim.x) {
            const int j = pk.pack_to_slot[p];
            int v;
            if (thick) v = thick[j];
            else v = ((bits[j >> 5] >> (j & 31)) & 1u) ? kPainted : pk.status_init;
            status_out[(size_t)k * pk.n_texels + p] = (int16_t)v;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const EnvState &st = ea.states[env];
        if (pose_out) for (int i = 0; i < 3; ++i) pose_out[3 * k + i] = st.pose[i];
        if (quat_out) for (int i = 0; i < 4; ++i) quat_out[4 * k + i] = st.quat[i];
        if (scalars_out) {
            double *o = scalars_out + kStateScalars * (size_t)k;
            o[0] = st.total_reward; o[1] = st.total_return; o[2] = st.step_counter; o[3] = st.term_counter;
            o[4] = (st.flags & kFlagLastOnPart) ? 1.0 : 0.0; o[5] = (st.flags & kFlagTerminate) ? 1.0 : 0.0;
            o[6] = st.last_angle; o[7] = st.angle_diff;
            // the overlap reference Part._last_painted_pixels (bullet_paint_wrapper.py:483, 575-576): the set is the
            // ball query of the last shot's centre, so the centre (and whether there is one) carries it exactly
            o[8] = (st.flags & kFlagHasLast) ? 1.0 : 0.0;
            o[9] = st.last_center[0]; o[10] = st.last_center[1]; o[11] = st.last_center[2];
        }
    }
}

// Scalars / pose of set_state (one thread per listed environment).
__global__ void set_scalars_kernel(EnvArrays ea, int num_envs, const int32_t *env_ids, int n, const double *pose_in, const double *quat_in,
                                   const double *scalars_in, int status_given) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int env = env_ids ? env_ids[k] : k;
    if ((unsigned)env >= (unsigned)num_envs) return;
    ea.ready[env] = 0u;
    EnvState &st = ea.states[env];
    if (pose_in) for (int i = 0; i < 3; ++i) st.pose[i] = pose_in[3 * k + i];
    if (quat_in) for (int i = 0; i < 4; ++i) st.quat[i] = quat_in[4 * k + i];
    if (scalars_in) {
        const double *o = scalars_in + kStateScalars * (size_t)k;
        st.total_reward = o[0]; st.total_return = o[1]; st.step_counter = (int)o[2]; st.term_counter = (int)o[3];
        int f = 0;
        if (o[4] != 0.0) f |= kFlagLastOnPart;
        if (o[5] != 0.0) f |= kFlagTerminate;
        if (o[8] != 0.0) f |= kFlagHasLast;               // the overlap reference travels with the scalars (ABI v2)
        st.flags = f;
        st.last_angle = o[6]; st.angle_diff = o[7];
        st.last_center[0] = o[9]; st.last_center[1] = o[10]; st.last_center[2] = o[11];
    } else if (status_given) {
        // a status plane without scalars: no overlap reference came with it -- clear it, as reset_part does
        // (bullet_paint_wrapper.py:708)
        st.flags &= ~kFlagHasLast;
    }
}

// Status planes of set_state: one warp per listed environment rebuilds the flip bits, the
// thickness plane (HSI) and the grid-cell counters.  In RGB mode a texel is painted (255) or not:
// any other value reads back as the fresh colour.
__global__ void set_status_kernel(DevPack pk, EnvArrays ea, int num_envs, const int32_t *env_ids, int n, const int16_t *status_in) {
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= n) return;
    const int env = env_ids ? env_ids[k] : k;
    if ((unsigned)env >= (unsigned)num_envs) return;
    unsigned *bits = bits_of(pk, ea, env), *grid_cnt = grid_cnt_of(pk, ea, env);
    int16_t *thick = thick_of(pk, ea, env);
    if (grid_cnt) for (int w = lane; w < pk.n_gcells_pad; w += 32) grid_cnt[w] = 0;
    // normal paint method: the previous shot's texel set is not part of the exported state -- start from none
    if (ea.last_mask) for (int w = lane; w < pk.n_words_pad; w += 32) ea.last_mask[(size_t)env * pk.n_words_pad + w] = 0u;
    __syncwarp();
    const bool init_painted = (pk.status_init == kPainted);
    const int16_t *src = status_in + (size_t)k * pk.n_texels;
    for (int w = 0; w < pk.n_words_pad; ++w) {
        bool fl = false;
        if (w < pk.n_words) {
            const int j = w * 32 + lane;
            const int p = pk.slot_to_pack[j];
            if (p >= 0) {
                const int v = src[p];
                fl = ((v == kPainted) != init_painted);
                if (thick) thick[j] = (int16_t)v;
                if (fl && grid_cnt) atomicAdd(grid_cnt + pk.gcell[j], 1u);
            } else if (thick) {
                thick[j] = (int16_t)pk.status_init;
            }
        }
        const unsigned m = __ballot_sync(kFull, fl);
        if (lane == 0) bits[w] = m;
    }
}

// get_job_status (bullet_paint_wrapper.py:727-732): painted front texels per env, one warp each
__global__ void job_status_kernel(DevPack pk, EnvArrays ea, int num_envs, int32_t *out) {
    const int lane = threadIdx.x & 31;
    const int env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= num_envs) return;
    const unsigned *bits = bits_of(pk, ea, env);
    int c = 0;
    for (int w = lane; w < pk.n_words; w += 32) c += __popc(bits[w]);
    c = __reduce_add_sync(kFull, c);
    if (lane == 0) out[env] = (pk.status_init == kPainted) ? pk.n_texels - c : c;
}

// paintrl_stats: sum of the per-environment counters.
__global__ void stats_kernel(const EnvStat *es, int num_envs, unsigned long long *out /*[5], zeroed*/) {
    unsigned long long a = 0, b = 0, c = 0, d = 0, f = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < num_envs; i += gridDim.x * blockDim.x) {
        a += es[i].episodes_ended; b += es[i].footprint_texels; c += es[i].full_scans; d += es[i].env_steps;
        f += es[i].move_bailouts;
    }
    atomicAdd(&out[0], a); atomicAdd(&out[1], b); atomicAdd(&out[2], c); atomicAdd(&out[3], d); atomicAdd(&out[4], f);
}

}  // namespace paintrl
