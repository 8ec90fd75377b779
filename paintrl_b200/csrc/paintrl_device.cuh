// paintrl_device.cuh -- device-side tables, state and FP64 geometry helpers of the batched paint step.
//
// Arithmetic contract (bit-exact against the oracle, see DESIGN.md "Arithmetic"):
//   * this translation unit is compiled with -fmad=false: every product and sum below is rounded
//     separately, in the written (= the reference's) order; FP64 division and sqrt are IEEE.
//   * np.dot / np.linalg.norm on 3-vectors (reference call sites: bullet_paint_wrapper.py:156-157,
//     robot.py:97, 269) are OpenBLAS ddot = fma(x2,y2, fma(x1,y1, x0*y0)); npdot3() is that chain,
//     written with explicit fma().
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace paintrl {

// Optional phase timing (build with -DPAINTRL_PROFILE; see profiles/README): cycles between
// PAINTRL_PROF marks, summed over environments into a 64-slot device array.
#ifdef PAINTRL_PROFILE
__device__ unsigned long long g_prof[64];
__device__ unsigned g_prof_env[65536][32];   // the same marks per environment, last step only (profiles/phase_profile.py --per-env)
#define PAINTRL_PROF_BEGIN(envidx, lo, hi)                                                \
    long long prof_t = clock64();                                                         \
    unsigned *prof_row = g_prof_env[(envidx) < 65536 ? (envidx) : 65535];                 \
    if ((threadIdx.x & 31) == 0) for (int prof_k = (lo); prof_k < (hi); ++prof_k) prof_row[prof_k] = 0;
#define PAINTRL_PROF(slot, leader)                                                        \
    do {                                                                                  \
        long long prof_now = clock64();                                                   \
        if (leader) {                                                                     \
            atomicAdd(&g_prof[slot], (unsigned long long)(prof_now - prof_t));            \
            if ((threadIdx.x & 31) == 0) prof_row[(slot) & 31] += (unsigned)(prof_now - prof_t); \
        }                                                                                 \
        prof_t = prof_now;                                                                \
    } while (0)
#define PAINTRL_PROF_PARAM , long long &prof_t, unsigned *prof_row
#define PAINTRL_PROF_PASS , prof_t, prof_row
#else
#define PAINTRL_PROF_BEGIN(envidx, lo, hi)
#define PAINTRL_PROF(slot, leader) do {} while (0)
#define PAINTRL_PROF_PARAM
#define PAINTRL_PROF_PASS
#endif

// Optional per-warp timeline (build with -DPAINTRL_TRACE; profiles/timeline.py): %globaltimer at the start and
// end of each environment's move and paint work plus the SM it ran on, last step only.
#ifdef PAINTRL_TRACE
__device__ unsigned long long g_trace[65536][8];
__device__ __forceinline__ unsigned long long trace_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned trace_smid() {
    unsigned s;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
    return s;
}
#define PAINTRL_TRACE_MARK(env, slot, leader) do { if ((leader) && (env) < 65536) g_trace[env][slot] = trace_now(); } while (0)
#define PAINTRL_TRACE_SM(env, slot, leader) do { if ((leader) && (env) < 65536) g_trace[env][slot] = trace_smid(); } while (0)
#else
#define PAINTRL_TRACE_MARK(env, slot, leader) do {} while (0)
#define PAINTRL_TRACE_SM(env, slot, leader) do {} while (0)
#endif

constexpr double kPaintRadius = 0.051;        // bullet_paint_wrapper.py:42
constexpr double kStepSize = kPaintRadius;    // bullet_paint_wrapper.py:43
constexpr int kPaintPerAction = 5;            // robot.py:165
constexpr int kNotOnPartTerminateSteps = 1000;  // robot.py:167
constexpr double kHookDistance = 0.1;         // bullet_paint_wrapper.py:443
constexpr int kHsiTargetMax = 25;             // bullet_paint_wrapper.py:388
constexpr int kPainted = 255;                 // bullet_paint_wrapper.py:354, 496
constexpr double kPi = 3.141592653589793;     // math.pi / np.pi
constexpr int kStateScalars = 12;             // doubles per environment in paintrl_get_state / set_state `scalars` (ABI v2)
constexpr int kMaxObs = 128;                  // largest observation vector (OBS_GRAD^2 or OBS_GRAD+2)
constexpr int kWarpsPerBlock = 4;
constexpr int kMaxRows = 128;                // rows of the texel layout
constexpr unsigned kFull = 0xffffffffu;

enum : int { kFlagLastOnPart = 1, kFlagTerminate = 2, kFlagHasLast = 4 };

// Per-environment record: one 128-byte line, read and written once per step.
// Robot._pose/_orn (robot.py:235-242), Part._last_painted_pixels (bullet_paint_wrapper.py:483,
// represented by the centre of the last shot: the set is the ball query of that centre),
// Robot turning/termination state (robot.py:201-218), PaintGymEnv counters (robot_gym_env.py:219-221).
struct alignas(128) EnvState {
    double pose[3];
    double quat[4];
    double last_center[3];
    double last_angle;
    double angle_diff;
    double total_reward;
    double total_return;
    int32_t step_counter;
    int32_t term_counter;
    int32_t flags;
    int32_t episode;
};
static_assert(sizeof(EnvState) == 128, "EnvState must be one 128-byte line");

// What the move kernel hands to the paint kernel: the five shot centres of the step
// (robot.py:277-278) and how many off-part sub-steps it counted (robot.py:427-430).
struct alignas(128) MoveOut {
    double centers[kPaintPerAction][3];
    int32_t counts;        // bits 0..3 off-part sub-steps added, 8..15 full plane scans, 16..23 verify passes
    uint32_t miss_cache;   // the entering | exiting << 16 hull planes that decided the env's last full plane scan
                           // (0xffff: none); kept from step to step, only ever used to prove misses
};
static_assert(sizeof(MoveOut) == 128, "MoveOut must be one 128-byte line");

// Normal paint method: what the move kernel hands over per shot besides the centre -- the TCP pose and orientation
// the beam fan is cast from (Robot._generate_paint_beams, robot.py:251-258).
struct alignas(32) ShotPoses {
    double pos[kPaintPerAction][3];
    double quat[kPaintPerAction][4];
    double pad;
};

// Per-environment counters behind paintrl_stats (summed on request; no atomics on the step path).
struct alignas(64) EnvStat {
    unsigned long long episodes_ended, footprint_texels, full_scans, env_steps;
    unsigned long long move_bailouts;   // steps whose move phase the fast kernel handed to the paint warp
    unsigned long long pad[3];
};

// Move grid over (axis0, axis1) (see build_move_cells in paintrl_capi.cu).  Every cell has an 8-byte
// entry (blob offset in 32-byte sectors, list lengths) and a contiguous blob
//   sector 0: a, b, c, rlo      sector 1: rhi, -, -, -
//   sectors 2 .. 2 + n_planes:  hull planes (nx, ny, nz, off), copied from the plane table
//   then n_verts sectors:       candidate nearest vertices (x, y, z, id | rec << 32)
// so that one table lookup is followed by one round of independent loads.
// Cells the hull's tool-side surface passes over carry a region hugging that surface: the cell's
// footprint x { depth : rlo <= depth - (a + b x0 + c x1) <= rhi } (depth = non-principal coordinate,
// the plane a + b x0 + c x1 is fitted to the surface over the cell), the hull planes that are not
// satisfied with margin everywhere in the region, and the front vertices that can be nearest to
// some point of it.  Other cells: rlo > rhi (never accepted), a short list of planes that usually
// proves a miss, no vertices.
struct CellRef {
    const double2 *blob;   // nullptr: none
    int n_planes, n_verts;
};

// Candidate nearest vertex: position, pack vertex index (tie-break), its incident-triangle
// records [rec_begin, rec_begin + deg) in `trirec`.
struct alignas(32) VertCand {
    double x, y, z;
    unsigned id;
    unsigned rec;                 // rec_begin << 8 | deg
};
static_assert(sizeof(VertCand) == 32, "VertCand is one 32-byte sector");

constexpr int kTriRec = 24;       // doubles per incident-triangle record:
// [0..2] a  [3..5] v0  [6..8] v1  [9] d00 [10] d01 [11] d11 [12] inv_denom   (BarycentricInterpolator, :123-146)
// [13..15] corrected normal n   [16..19] quat_from_normal(-n)   [20..22] R(quat)*(0,0,0.1)   [23] pad

// Constant per-part tables in device memory (shared by all environments, L1/L2 resident).
struct DevPack {
    int n_texels;
    int axis0, axis1;
    int status_init;
    // collision hull: (nx, ny, nz, off) per plane
    int n_planes;
    const double4 *planes;
    // move grid
    int mc_nx, mc_ny;
    double mc_o0, mc_o1, mc_inv;
    const uint2 *mc_entry;        // [mc_nx * mc_ny] x = blob sector offset, y = n_planes | n_verts << 16
    const double2 *mc_blob;       // 32-byte sectors (two double2 each)
    const double *trirec;         // [n_rec][kTriRec]
    // slow-path nearest-vertex grid over (axis0, axis1): front vertices sorted by cell
    int vg_nx, vg_ny;
    double vg_o0, vg_o1, vg_cs, vg_inv;
    const int *vg_start;          // [vg_nx*vg_ny + 1]
    const double *vx, *vy, *vz;   // sorted vertex coordinates
    const int *vid;               // sorted -> pack vertex index
    const unsigned *vrec;         // [n_vertices] rec_begin << 8 | deg per pack vertex
    // texel layout "rows and words" (see build_tables in paintrl_capi.cu): rows = strips along
    // axis1, texels of a row sorted by their axis0 coordinate and packed 32 to a word; every row
    // starts a new word.  A slot is (word, bit); pad slots hold far-away positions.
    int n_words, n_words_pad;     // n_words_pad: per-env bit-plane stride in words (multiple of 32)
    int n_slots;                  // n_words * 32
    int n_rows;                   // <= kMaxRows
    double row_o1, row_inv, row_h;   // row(y) = floor((y - row_o1) * row_inv)
    int ncx;                      // cells along axis0, cell(x) = floor((x - cx_o0) * cx_inv)
    double cx_o0, cx_inv;
    float rel_row_o1, rel_row_h, rel_cx_o0, rel_cx_inv;   // the two grids relative to the origin, FP32 (stamp_ranges)
    const int *row_word0;         // [n_rows + 1] first word of each row
    const int *row_count;         // [n_rows] texels in the row
    const int *cell_start;        // [n_rows][ncx + 1] index in the row of the first texel with cell >= c
    const unsigned *word_info;    // [n_words] row | valid slots << 8 | (word index within the row) << 14
    const float *fx, *fy, *fz;    // [n_slots] position - origin in FP32 (ball pre-test)
    double org0, org1, org2;
    const double *tx, *ty, *tz;   // [n_slots] exact texel positions (world x, y, z)
    const uint16_t *gcell;        // [n_slots] grid-observation cell (grid mode only)
    const int *slot_to_pack;      // [n_slots] part-pack texel index, -1 for pad slots
    const int *pack_to_slot;      // [n_texels]
    const int *nn_rep_slot;       // [n_slots] normal paint: the slot cKDTree.query reports among texels at this slot's exact position
    // normal paint: nearest-texel grid over the principal plane (square cells of two texel pitches)
    int nn_nx, nn_ny;
    double nn_o0, nn_o1, nn_inv, nn_cell;
    const int *nn_start;          // [nn_nx * nn_ny + 1]
    const double2 *nn_pos;        // per texel, grouped by cell: (x, y) (z, slot as int64 bits)
    // grid observation (bullet_paint_wrapper.py:1072-1112)
    int n_gcells, n_gcells_pad;
    const int *gtotal;            // [obs_grad^2]
    // normalised pose (bullet_paint_wrapper.py:965-978)
    int grid_granularity;
    const double *grid_lo, *grid_hi;
    double range0_min, range0_max, range1_min, range1_max, lwr;
    // start points
    int n_starts;
    const double *start_pos, *start_normal;
    const double *reset_obs;      // [n_starts][obs_dim] observation of a fresh environment at each start point
    // the read-only tables above live in a few slabs; the step kernels pull them into L2 at their start (l2_prefetch_tables)
    int pf_n;
    const char *pf_base[4];
    unsigned pf_lines[4];         // 128-byte lines per slab
};

// One strided pass of L2 prefetches over the static tables: thread `tid` of `nthreads`.  At 4096 environments the
// 11 MB of tables are 86 k lines, less than one per thread; the step then finds its table lookups (move cells,
// triangle records, texel coordinates: dependent loads, a handful per sub-step) in L2 even when other work has evicted
// them since the last step, instead of paying a DRAM round trip on each.
__device__ __forceinline__ void l2_prefetch_tables(const DevPack &pk, unsigned tid, unsigned nthreads) {
    for (int k = 0; k < pk.pf_n; ++k) {
        const char *base = pk.pf_base[k];
        for (unsigned i = tid; i < pk.pf_lines[k]; i += nthreads)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)i * 128));
    }
}

struct DevConfig {
    int action_mode, action_shape, discrete_granularity;
    const double *discrete_table;   // [n][3] u1, u2, angle
    int obs_mode, obs_grad, obs_dim;
    int color_mode, termination_mode;
    double switch_threshold;
    int expected_episode_length, episode_max_length;
    int turning_penalty, overlap_penalty;
    double max_possible_point;
    double expected_avg_reward;     // max_possible_point / (Expected_Episode_Length * 100)   (robot_gym_env.py:297)
    double hybrid_threshold;        // SWITCH_THRESHOLD * max_possible_point / 100            (robot_gym_env.py:302)
    int auto_reset;
    int paint_method;               // 0 fast (ball query per shot), 1 normal (beam fan per shot; robot.py:172, 414-417)
    int n_beams;
    const double *beam_plain;       // [n_beams][3] Robot._paint_plain, ray end points in the TCP frame
    int debug_bail_mod;             // PAINTRL_DEBUG_BAIL_MOD=n (tests): every n-th environment leaves the fast move kernel at once
    int start_order;                // PAINTRL_START_ORDER (default 1): the one-kernel step loads the record before the L2 sweep and
                                    // copies the bit-plane in after the move phase; 0: sweep, copy, record (results are the same)
    unsigned long long seed;
};

// ------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ double npdot3(double x0, double x1, double x2, double y0, double y1, double y2) {
    return fma(x2, y2, fma(x1, y1, x0 * y0));
}

struct Vec3 { double x, y, z; };

// Principal axes of the part.  Both reference parts use (1, 2): kernels instantiated with AX12 carry
// them as compile-time constants, so component selections fold away.
struct Ax { int a0, a1; };
template <bool AX12>
__device__ __forceinline__ Ax make_ax(int axis0, int axis1) {
    Ax ax;
    ax.a0 = AX12 ? 1 : axis0;
    ax.a1 = AX12 ? 2 : axis1;
    return ax;
}

__device__ __forceinline__ double comp(const Vec3 &v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }
__device__ __forceinline__ void add_comp(Vec3 &v, int a, double d) {
    if (a == 0) v.x += d; else if (a == 1) v.y += d; else v.z += d;
}

// oracle/shims/pybullet.py multiplyTransforms (Bullet btMatrix3x3::setRotation + btTransform())
__host__ __device__ __forceinline__ Vec3 transform_point(const Vec3 &pos, const double q[4], double v0, double v1, double v2) {
    double x = q[0], y = q[1], z = q[2], w = q[3];
    double d = x * x + y * y + z * z + w * w;
    double s = 2.0 / d;
    double xs = x * s, ys = y * s, zs = z * s;
    double wx = w * xs, wy = w * ys, wz = w * zs;
    double xx = x * xs, xy = x * ys, xz = x * zs;
    double yy = y * ys, yz = y * zs, zz = z * zs;
    Vec3 o;
    o.x = (((1.0 - (yy + zz)) * v0 + (xy - wz) * v1) + (xz + wy) * v2) + pos.x;
    o.y = (((xy + wz) * v0 + (1.0 - (xx + zz)) * v1) + (yz - wx) * v2) + pos.y;
    o.z = (((xz - wy) * v0 + (yz + wx) * v1) + (1.0 - (xx + yy)) * v2) + pos.z;
    return o;
}

// robot.py:93-100 get_pose_orn + bullet_paint_wrapper.py:32-37 normalize
__host__ __device__ __forceinline__ void quat_from_normal(const Vec3 &n, double q[4]) {
    double x = 0.0 * n.z - 1.0 * n.y;
    double y = 1.0 * n.x - 0.0 * n.z;
    double z = 0.0 * n.y - 0.0 * n.x;
    double w = 1.0 + npdot3(0.0, 0.0, 1.0, n.x, n.y, n.z);
    double mag2 = ((x * x + y * y) + z * z) + w * w;
    if (fabs(mag2 - 1.0) > 0.00001) {
        double mag = sqrt(mag2);
        x /= mag; y /= mag; z /= mag; w /= mag;
    }
    q[0] = x; q[1] = y; q[2] = z; q[3] = w;
}

// robot.py:266-271 _get_tcp_orn_norm
__device__ __forceinline__ Vec3 tcp_orn_norm(const Vec3 &pose, const double q[4]) {
    Vec3 along = transform_point(pose, q, 0.0, 0.0, 1.0);
    double vx = along.x - pose.x, vy = along.y - pose.y, vz = along.z - pose.z;
    double norm = sqrt(npdot3(vx, vy, vz, vx, vy, vz));
    Vec3 o = {vx / norm, vy / norm, vz / norm};
    return o;
}

// Warp max of doubles through two 32-bit REDUX steps on an order-preserving key (paint kernel).
__device__ __forceinline__ unsigned long long ordered_key(double v) {
    long long b = __double_as_longlong(v);
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000ull));
}
__device__ __forceinline__ double from_ordered_key(unsigned long long k) {
    long long b = (long long)k;
    b ^= ((~b) >> 63) | (long long)0x8000000000000000ull;
    return __longlong_as_double(b);
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long k) {
    unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
    unsigned mhi = __reduce_max_sync(kFull, hi);
    unsigned mlo = __reduce_max_sync(kFull, hi == mhi ? lo : 0u);
    return ((unsigned long long)mhi << 32) | mlo;
}
__device__ __forceinline__ double warp_max(double v) { return from_ordered_key(warp_max_u64(ordered_key(v))); }

// ------------------------------------------------------------------------------------------
// The move phase runs G lanes per environment (G = 8, 16 or 32; 32 / G environments per warp).
// `Grp` is a lane's view of its group: index within the group, the group's lane mask, its first lane.
struct Grp { int gl; unsigned mask; int base; };

template <int G>
__device__ __forceinline__ Grp make_grp(int lane) {
    Grp g;
    g.gl = lane & (G - 1);
    g.base = lane & ~(G - 1);
    g.mask = (G == 32) ? kFull : (((1u << G) - 1u) << g.base);
    return g;
}
// max / min / sum over the group.  A full warp uses the REDUX unit on an order-preserving integer
// key (two 32-bit steps per double); smaller groups use xor-shuffles.
__device__ __forceinline__ double warp_min(double v) { return from_ordered_key(~warp_max_u64(~ordered_key(v))); }

template <int G>
__device__ __forceinline__ double grp_max(double v, const Grp &g) {
    if constexpr (G == 32) {
        return warp_max(v);
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(g.mask, v, o));
        return v;
    }
}
template <int G>
__device__ __forceinline__ double grp_min(double v, const Grp &g) {
    if constexpr (G == 32) {
        return warp_min(v);
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(g.mask, v, o));
        return v;
    }
}
template <int G>
__device__ __forceinline__ int grp_sum(int v, const Grp &g) {
    if constexpr (G == 32) {
        return __reduce_add_sync(kFull, v);
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(g.mask, v, o);
        return v;
    }
}
template <int G>
__device__ __forceinline__ bool grp_any(bool p, const Grp &g) {
    return G == 32 ? __any_sync(kFull, p) : __any_sync(g.mask, p);
}
template <int G>
__device__ __forceinline__ unsigned grp_ballot(bool p, const Grp &g) {   // bit i = lane i of the group
    return G == 32 ? __ballot_sync(kFull, p) : ((__ballot_sync(g.mask, p) & g.mask) >> g.base);
}

// One pass of the slab test over a list of planes (`planes` = two double2 per plane: the plane table
// or a cell blob's copy of some of its entries), split across the group; max/min are
// order-independent so the result equals the serial one.
struct SlabResult { double t_in, t_out; bool outside; };

template <int G, bool TRACK = false>
__device__ __forceinline__ SlabResult slab_pass(const double2 *planes, int n, const Vec3 &frm, double d0, double d1, double d2,
                                                const Grp &g, unsigned *args = nullptr) {
    double t_in = -INFINITY, t_out = INFINITY;
    bool outside = false;
    int a_in = 0xffff, a_out = 0xffff;   // TRACK: list positions attaining this lane's t_in / t_out
    for (int i = g.gl; i < n; i += G) {
        const double2 lo = __ldg(planes + 2 * i), hi2 = __ldg(planes + 2 * i + 1);
        double den = (lo.x * d0 + lo.y * d1) + hi2.x * d2;
        double num = hi2.y - ((lo.x * frm.x + lo.y * frm.y) + hi2.x * frm.z);
        if (den == 0.0) {
            if (num < 0.0) outside = true;
        } else {
            double t = num / den;
            if (den < 0.0) { if (TRACK && t > t_in) a_in = i; t_in = fmax(t_in, t); }
            else { if (TRACK && t < t_out) a_out = i; t_out = fmin(t_out, t); }
        }
    }
    SlabResult r;
    r.t_in = grp_max<G>(t_in, g);
    r.t_out = grp_min<G>(t_out, g);
    r.outside = grp_any<G>(outside, g);
    if (TRACK) {
        const unsigned m_in = grp_ballot<G>(t_in == r.t_in && a_in != 0xffff, g), m_out = grp_ballot<G>(t_out == r.t_out && a_out != 0xffff, g);
        const int w_in = m_in ? __shfl_sync(g.mask, a_in, g.base + __ffs(m_in) - 1) : 0xffff;
        const int w_out = m_out ? __shfl_sync(g.mask, a_out, g.base + __ffs(m_out) - 1) : 0xffff;
        *args = (unsigned)min(w_in, 0xffff) | ((unsigned)min(w_out, 0xffff) << 16);
    }
    return r;
}

// Does the pair of hull planes `cache` (entering | exiting << 16), together with the bounds of a
// subset already scanned, prove that the ray misses the hull?  (Any subset may be used for that.)
__device__ __forceinline__ bool pair_proves_miss(const DevPack &pk, unsigned cache, const SlabResult &r0, bool have_r0, const Vec3 &frm,
                                                 double d0, double d1, double d2) {
    double t_in = have_r0 ? r0.t_in : -INFINITY, t_out = have_r0 ? r0.t_out : INFINITY;
    bool outside = false;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int pi = (int)((cache >> (16 * k)) & 0xffffu);
        if (pi >= pk.n_planes) continue;
        const double2 *p2 = reinterpret_cast<const double2 *>(pk.planes) + 2 * pi;
        const double2 lo = __ldg(p2), hi2 = __ldg(p2 + 1);
        double den = (lo.x * d0 + lo.y * d1) + hi2.x * d2;
        double num = hi2.y - ((lo.x * frm.x + lo.y * frm.y) + hi2.x * frm.z);
        if (den == 0.0) {
            if (num < 0.0) outside = true;
        } else {
            double t = num / den;
            if (den < 0.0) t_in = fmax(t_in, t);
            else t_out = fmin(t_out, t);
        }
    }
    return outside || t_in > t_out || t_in > 1.0 || t_out < 0.0;
}

// Number of listed planes the point h does not satisfy with margin (n.h - off > -kVerifyMargin).
// The value per plane depends only on the plane's four doubles, so equal counts over the full
// plane table and over a list of copies of some of its entries mean that every plane outside the
// list is satisfied with margin.
constexpr double kVerifyMargin = 1e-9;
template <int G>
__device__ __forceinline__ int near_violations(const double2 *planes, int n, const Vec3 &h, const Grp &g) {
    int c = 0;
    int i = g.gl;
    // long lists (the whole plane table): four planes per lane in flight, their loads issued together
    for (; i + 3 * G < n; i += 4 * G) {
        double2 lo[4], hi[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { lo[k] = __ldg(planes + 2 * (i + k * G)); hi[k] = __ldg(planes + 2 * (i + k * G) + 1); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double sd = fma(hi[k].x, h.z, fma(lo[k].y, h.y, lo[k].x * h.x)) - hi[k].y;
            c += (sd > -kVerifyMargin) ? 1 : 0;
        }
    }
    for (; i < n; i += G) {
        const double2 lo = __ldg(planes + 2 * i), hi2 = __ldg(planes + 2 * i + 1);
        double sd = fma(hi2.x, h.z, fma(lo.y, h.y, lo.x * h.x)) - hi2.y;
        c += (sd > -kVerifyMargin) ? 1 : 0;
    }
    return grp_sum<G>(c, g);
}

// The same count with a plain loop (the fast move path's copy of the verify pass: rare there, and its registers must
// not add to that kernel's budget).  Per plane the same expression as near_violations, so counts are comparable.
template <int G>
__device__ __noinline__ int near_violations_rolled(const double2 *planes, int n, Vec3 h, Grp g) {
    int c = 0;
#pragma unroll 1
    for (int i = g.gl; i < n; i += G) {
        const double2 lo = __ldg(planes + 2 * i), hi2 = __ldg(planes + 2 * i + 1);
        const double sd = fma(hi2.x, h.z, fma(lo.y, h.y, lo.x * h.x)) - hi2.y;
        c += (sd > -kVerifyMargin) ? 1 : 0;
    }
    return grp_sum<G>(c, g);
}

// The slab test over the WHOLE plane table (the slow path of ray_test), tracking the planes that attain
// t_in / t_out.  Same per-plane arithmetic as slab_pass; two planes per lane in flight and a branch-free
// body, so the loads and the two FP64 divisions of an iteration overlap.
template <int G>
__device__ __forceinline__ SlabResult slab_pass_all(const double2 *planes, int n, const Vec3 &frm, double d0, double d1, double d2,
                                                    const Grp &g, unsigned *args) {
    double t_in = -INFINITY, t_out = INFINITY;
    bool outside = false;
    int a_in = 0xffff, a_out = 0xffff;
    auto one = [&](int i, const double2 &lo, const double2 &hi2) {
        const double den = (lo.x * d0 + lo.y * d1) + hi2.x * d2;
        const double num = hi2.y - ((lo.x * frm.x + lo.y * frm.y) + hi2.x * frm.z);
        const double t = num / (den == 0.0 ? 1.0 : den);
        outside |= (den == 0.0 && num < 0.0);
        const bool ent = den < 0.0, ext = den > 0.0;
        if (ent && t > t_in) a_in = i;
        if (ext && t < t_out) a_out = i;
        t_in = ent ? fmax(t_in, t) : t_in;
        t_out = ext ? fmin(t_out, t) : t_out;
    };
    int i = g.gl;
    for (; i + G < n; i += 2 * G) {
        const double2 lo0 = __ldg(planes + 2 * i), hi0 = __ldg(planes + 2 * i + 1);
        const double2 lo1 = __ldg(planes + 2 * (i + G)), hi1 = __ldg(planes + 2 * (i + G) + 1);
        one(i, lo0, hi0);
        one(i + G, lo1, hi1);
    }
    if (i < n) one(i, __ldg(planes + 2 * i), __ldg(planes + 2 * i + 1));
    SlabResult r;
    r.t_in = grp_max<G>(t_in, g);
    r.t_out = grp_min<G>(t_out, g);
    r.outside = grp_any<G>(outside, g);
    const unsigned m_in = grp_ballot<G>(t_in == r.t_in && a_in != 0xffff, g), m_out = grp_ballot<G>(t_out == r.t_out && a_out != 0xffff, g);
    const int w_in = m_in ? __shfl_sync(g.mask, a_in, g.base + __ffs(m_in) - 1) : 0xffff;
    const int w_out = m_out ? __shfl_sync(g.mask, a_out, g.base + __ffs(m_out) - 1) : 0xffff;
    *args = (unsigned)min(w_in, 0xffff) | ((unsigned)min(w_out, 0xffff) << 16);
    return r;
}

__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// debug (instrumented build only): rays that left the fast path, for offline analysis of the move cells
#ifdef PAINTRL_PROFILE
__device__ unsigned long long g_dbg_counts[4];   // [0] grid searches  [1] rays logged
__device__ double g_dbg_rays[4096][8];           // frm.xyz, d.xyz, kind (1 verify ok, 2 full scan), hit flag
#endif
__device__ __forceinline__ void g_dbg_grid_searches_inc() {
#ifdef PAINTRL_PROFILE
    atomicAdd(&g_dbg_counts[0], 1ull);
#endif
}
__device__ __forceinline__ void g_dbg_log_ray(const Vec3 &frm, double d0, double d1, double d2, int kind, bool hit, bool leader) {
#ifdef PAINTRL_PROFILE
    if (leader) {
        unsigned long long i = atomicAdd(&g_dbg_counts[1], 1ull);
        if (i < 4096) {
            double *o = g_dbg_rays[i];
            o[0] = frm.x; o[1] = frm.y; o[2] = frm.z; o[3] = d0; o[4] = d1; o[5] = d2; o[6] = kind; o[7] = hit ? 1.0 : 0.0;
        }
    }
#endif
}

// Exact slab test of the ray frm -> to against the hull half-spaces (shim S1).
//
// For any subset S of the planes t_in(S) <= t_in and t_out(S) >= t_out, so
//   (1) a miss is proven by S alone when outside(S), t_in(S) > t_out(S), t_in(S) > 1 or t_out(S) < 0;
//   (2) if every plane outside S is satisfied with margin at the entry point h* = frm + d t_in(S),
//       i.e. n_j.h* < off_j - margin, then t_j < t* for an entering plane j and t_j > t* for an
//       exiting one: t* is the global t_in bit for bit and the hit / miss decision over S equals the
//       one over all planes.  This holds by construction when S is a move cell's list and h* lies in
//       that cell's region (2a), and otherwise it is checked directly with one division-free pass
//       over the plane table (2b).
// Otherwise the full plane list is scanned.  Either way the result is the serial slab test's.
// On a hit accepted through (2a) `ref` is the move cell holding the hit point (for the vertex
// candidates; `vc0` / `vc1` hold this lane's first candidate), else ref.blob == nullptr.
// (pf0, pf1): expected displacement of the next ray along the principal axes -- its cell's blob is
// prefetched into L1 while this ray is being tested (do_prefetch).
constexpr int kRayAttempts = 5;   // two tiers per silhouette cell: a ray may need (cell A, its fallback, cell B, its fallback)

// Region test of a move cell: does the point h (principal coordinates h0, h1) lie in the cell
// (cx, cy) and within the slab around its fitted surface plane?
__device__ __forceinline__ bool in_cell_region(const DevPack &pk, const Vec3 &h, double h0, double h1, double depth, int cx, int cy,
                                               const double2 &abv, const double2 &clv, const double2 &hpv) {
    const int hx = (int)floor((h0 - pk.mc_o0) * pk.mc_inv);
    const int hy = (int)floor((h1 - pk.mc_o1) * pk.mc_inv);
    const double resid = depth - (abv.x + abv.y * h0 + clv.x * h1);
    return hx == cx && hy == cy && resid >= clv.y && resid <= hpv.x;
}

// The same test against the cell's index cy * mc_nx + cx.
__device__ __forceinline__ bool in_cell_region_idx(const DevPack &pk, double h0, double h1, double depth, int cell, const double2 &abv,
                                                   const double2 &clv, const double2 &hpv) {
    const int hx = (int)floor((h0 - pk.mc_o0) * pk.mc_inv);
    const int hy = (int)floor((h1 - pk.mc_o1) * pk.mc_inv);
    const double resid = depth - (abv.x + abv.y * h0 + clv.x * h1);
    return hx >= 0 && hx < pk.mc_nx && hy * pk.mc_nx + hx == cell && resid >= clv.y && resid <= hpv.x;
}

template <int G>
__device__ __forceinline__ bool ray_test(const DevPack &pk, const Ax &ax, const Vec3 &frm, const Vec3 &to, const Grp &grp, Vec3 &hit,
                                         CellRef &ref, double2 &vc0, double2 &vc1, int &counts, unsigned &miss_cache, double pf0,
                                         double pf1, bool do_prefetch PAINTRL_PROF_PARAM) {
    double d0 = to.x - frm.x, d1 = to.y - frm.y, d2 = to.z - frm.z;
    SlabResult r;
    bool accepted = false, candidate = false;
    const double2 *sub = nullptr;
    int n_sub = 0;
    ref.blob = nullptr;
    const int npax = 3 - ax.a0 - ax.a1;
    // the TCP hovers kHookDistance above the surface: first guess = the point that far along the ray;
    // later guesses = the entry point of the previous cell's list
    Vec3 h = {frm.x + d0 * kHookDistance, frm.y + d1 * kHookDistance, frm.z + d2 * kHookDistance};
#ifdef PAINTRL_PROFILE
    int why = 0;   // why the last attempt did not accept: 1 outside the grid, 2 empty cell, 3 no entering plane, 4 other cell, 5 below, 6 above the slab
#define PAINTRL_WHY(v) why = (v)
#else
#define PAINTRL_WHY(v)
#endif
    int tried_cx = -1, tried_cy = -1;
    unsigned long long link = 0ull;    // fallback blob of the cell just tried (offset | counts << 32), 0: none
#pragma unroll 1
    for (int attempt = 0; attempt < kRayAttempts; ++attempt) {
        const double g0 = comp(h, ax.a0), g1 = comp(h, ax.a1);
        int cx = (int)floor((g0 - pk.mc_o0) * pk.mc_inv);
        int cy = (int)floor((g1 - pk.mc_o1) * pk.mc_inv);
        if (link == 0ull && (cx < 0 || cy < 0 || cx >= pk.mc_nx || cy >= pk.mc_ny)) { PAINTRL_WHY(1); break; }
#if defined(PAINTRL_TRACE) || defined(PAINTRL_PROFILE)
        counts += 1 << 24;   // cell attempts of the step (diagnostic builds only)
#endif
        uint2 entry;
        if (link != 0ull) {
            // the cell just tried is a silhouette cell whose thin primary slab did not hold the entry point: its second
            // blob (deep slab, build_move_cells) comes next, whichever cell the provisional entry point fell into
            cx = tried_cx; cy = tried_cy;
            entry = make_uint2((unsigned)link, (unsigned)(link >> 32));
        } else {
            if (cx == tried_cx && cy == tried_cy) break;     // the same cell again: same list, same result
            entry = __ldg(&pk.mc_entry[cy * pk.mc_nx + cx]);
        }
        tried_cx = cx; tried_cy = cy;
        const int n_planes = (int)(entry.y & 0xffffu), n_verts = (int)(entry.y >> 16);
        if (n_planes <= 0) { PAINTRL_WHY(2); break; }
        const double2 *blob = pk.mc_blob + (size_t)entry.x * 2;
        // one round of independent loads: region, this lane's plane(s) (in slab_pass), first vertex candidate
        const double2 abv = __ldg(blob), clv = __ldg(blob + 1), hpv = __ldg(blob + 2);   // (a, b) (c, rlo) (rhi, link)
        link = (unsigned long long)__double_as_longlong(hpv.y);
        if (grp.gl < n_verts) {
            vc0 = __ldg(blob + 2 * (2 + n_planes + grp.gl));
            vc1 = __ldg(blob + 2 * (2 + n_planes + grp.gl) + 1);
        }
        if (do_prefetch && attempt == 0) {
            int px = (int)floor((g0 + pf0 - pk.mc_o0) * pk.mc_inv);
            int py = (int)floor((g1 + pf1 - pk.mc_o1) * pk.mc_inv);
            if (px >= 0 && py >= 0 && px < pk.mc_nx && py < pk.mc_ny && (px != cx || py != cy)) {
                const uint2 pe = __ldg(&pk.mc_entry[py * pk.mc_nx + px]);
                const int sectors = 2 + (int)(pe.y & 0xffffu) + (int)(pe.y >> 16);
                const char *pb = reinterpret_cast<const char *>(pk.mc_blob + (size_t)pe.x * 2);
                if (G == 32) { if (grp.gl * 128 < sectors * 32) prefetch_l1(pb + grp.gl * 128); }
                else for (int o = grp.gl * 128; o < sectors * 32; o += G * 128) prefetch_l1(pb + o);
            }
        }
        PAINTRL_PROF(6, grp.gl == 0);
        r = slab_pass<G>(blob + 4, n_planes, frm, d0, d1, d2, grp);
        PAINTRL_PROF(7, grp.gl == 0);
        if (r.outside || r.t_in > r.t_out || r.t_in > 1.0 || r.t_out < 0.0) return false;   // (1)
        candidate = false;
        if (!(r.t_in > -INFINITY)) { if (link != 0ull) continue; PAINTRL_WHY(3); break; }
        candidate = true;
        sub = blob + 4; n_sub = n_planes;
        h.x = frm.x + d0 * r.t_in; h.y = frm.y + d1 * r.t_in; h.z = frm.z + d2 * r.t_in;
        if (in_cell_region(pk, h, comp(h, ax.a0), comp(h, ax.a1), comp(h, npax), cx, cy, abv, clv, hpv)) {   // (2a)
            accepted = true;
            ref.blob = blob; ref.n_planes = n_planes; ref.n_verts = n_verts;
            break;
        }
#ifdef PAINTRL_PROFILE
        {
            const double h0 = comp(h, ax.a0), h1 = comp(h, ax.a1);
            const int hx = (int)floor((h0 - pk.mc_o0) * pk.mc_inv), hy = (int)floor((h1 - pk.mc_o1) * pk.mc_inv);
            const double resid = comp(h, npax) - (abv.x + abv.y * h0 + clv.x * h1);
            why = (hx != cx || hy != cy) ? 4 : (resid < clv.y ? 5 : 6);
            if (why >= 5) why += 10 * (n_verts > 0 ? 1 : 0) + 100 * min(99, (int)(fabs(resid - (resid < clv.y ? clv.y : hpv.x)) * 1e4));
        }
#endif
    }
    PAINTRL_PROF(8, grp.gl == 0);
    if (!accepted) {
        // (1) again with the pair of planes that decided this environment's last full scan
        if (pair_proves_miss(pk, miss_cache, r, candidate, frm, d0, d1, d2)) return false;
    }
    if (!accepted && candidate) {                                                           // (2b)
        counts += 1 << 16;
        const int c_all = near_violations<G>(reinterpret_cast<const double2 *>(pk.planes), pk.n_planes, h, grp);
        const int c_sub = near_violations<G>(sub, n_sub, h, grp);
        accepted = (c_all == c_sub);
        if (accepted && r.t_in <= r.t_out && 0.0 <= r.t_in && r.t_in <= 1.0) {
            // a hit: if it lies in the region of its own cell, that cell's vertex candidates apply
            const double h0 = comp(h, ax.a0), h1 = comp(h, ax.a1);
            const int cx = (int)floor((h0 - pk.mc_o0) * pk.mc_inv), cy = (int)floor((h1 - pk.mc_o1) * pk.mc_inv);
            if (cx >= 0 && cy >= 0 && cx < pk.mc_nx && cy < pk.mc_ny) {
                const uint2 entry = __ldg(&pk.mc_entry[cy * pk.mc_nx + cx]);
                const int n_planes = (int)(entry.y & 0xffffu), n_verts = (int)(entry.y >> 16);
                const double2 *blob = pk.mc_blob + (size_t)entry.x * 2;
                const double2 abv = __ldg(blob), clv = __ldg(blob + 1), hpv = __ldg(blob + 2);
                if (n_verts > 0 && in_cell_region(pk, h, h0, h1, comp(h, npax), cx, cy, abv, clv, hpv)) {
                    ref.blob = blob; ref.n_planes = n_planes; ref.n_verts = n_verts;
                    if (grp.gl < n_verts) {
                        vc0 = __ldg(blob + 2 * (2 + n_planes + grp.gl));
                        vc1 = __ldg(blob + 2 * (2 + n_planes + grp.gl) + 1);
                    }
                }
            }
        }
    }
    if (!accepted) {
        unsigned args = 0xffffffffu;
        r = slab_pass_all<G>(reinterpret_cast<const double2 *>(pk.planes), pk.n_planes, frm, d0, d1, d2, grp, &args);
        miss_cache = args;
        counts += 1 << 8;
    }
    const bool is_hit = !(r.outside || !(r.t_in <= r.t_out && 0.0 <= r.t_in && r.t_in <= 1.0));
#ifdef PAINTRL_PROFILE
    if (!ref.blob) g_dbg_log_ray(frm, d0, d1, d2, (accepted ? 1 : 2) + 10 * why, is_hit, grp.gl == 0);
#endif
    if (!is_hit) return false;
    hit.x = frm.x + d0 * r.t_in;
    hit.y = frm.y + d1 * r.t_in;
    hit.z = frm.z + d2 * r.t_in;
    PAINTRL_PROF(9, grp.gl == 0);
    return true;
}

// Lexicographic arg-min of (squared distance, vertex id) over the group; `rec` travels with it.
// d >= 0, so its raw bits order like its value.
template <int G>
__device__ __forceinline__ void grp_argmin(double &d, unsigned &id, unsigned &rec, const Grp &g) {
    if constexpr (G == 32) {
        const unsigned long long k = (unsigned long long)__double_as_longlong(d);
        const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
        const unsigned mhi = __reduce_min_sync(kFull, hi);
        const unsigned mlo = __reduce_min_sync(kFull, hi == mhi ? lo : 0xffffffffu);
        const bool best = (hi == mhi && lo == mlo);
        const unsigned mid = __reduce_min_sync(kFull, best ? id : 0xffffffffu);
        const int src = __ffs(__ballot_sync(kFull, best && id == mid)) - 1;
        rec = __shfl_sync(kFull, rec, src);
        id = mid;
        d = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(g.mask, d, o);
            const unsigned oi = __shfl_xor_sync(g.mask, id, o), orc = __shfl_xor_sync(g.mask, rec, o);
            if (od < d || (od == d && oi < id)) { d = od; id = oi; rec = orc; }
        }
    }
}

// cKDTree.query(point, k=1) over the side-masked vertices (bullet_paint_wrapper.py:526): exact
// FP64 squared distances, lowest pack index on ties.  Returns the vertex's record word
// (rec_begin << 8 | deg), or 0xFFFFFFFF if there is none.
//
// Fast path: the move cell that holds the point lists every vertex that can be nearest to a
// point of its region, so the arg-min over that list is the arg-min over all vertices.
// (vc0, vc1) = this lane's first candidate, loaded by ray_test.
template <int G>
__device__ __forceinline__ unsigned nearest_vertex_cell(const Vec3 &p, const CellRef &ref, double2 vc0, double2 vc1, const Grp &g) {
    double best = INFINITY;
    unsigned bid = 0xFFFFFFFFu, brec = 0xFFFFFFFFu;
    const double2 *vc = ref.blob + 2 * (2 + ref.n_planes);
    for (int i = g.gl; i < ref.n_verts; i += G) {
        if (i >= G) { vc0 = __ldg(vc + 2 * i); vc1 = __ldg(vc + 2 * i + 1); }
        double dx = vc0.x - p.x, dy = vc0.y - p.y, dz = vc1.x - p.z;
        double d = dx * dx + dy * dy + dz * dz;
        unsigned long long meta = (unsigned long long)__double_as_longlong(vc1.y);
        unsigned id = (unsigned)meta, rec = (unsigned)(meta >> 32);
        if (d < best || (d == best && id < bid)) { best = d; bid = id; brec = rec; }
    }
    grp_argmin<G>(best, bid, brec, g);
    return brec;
}

// Slow path (point outside every accepted cell region): the 3 x 3 block of vertex-grid cells around the
// point, accepted when it proves that no vertex outside the block can be nearer; otherwise (hull faces
// bridging an opening of the part: the nearest vertex is far away) one coalesced brute-force pass over
// all front vertices -- a bounded ~n/32 iterations instead of a growing ring search.
template <int G, typename VG>
__device__ __forceinline__ unsigned nearest_vertex_grid(const VG &pk, const Ax &ax, const Vec3 &p, const Grp &g) {
    double q0 = comp(p, ax.a0), q1 = comp(p, ax.a1);
    int cx = (int)floor((q0 - pk.vg_o0) * pk.vg_inv);
    int cy = (int)floor((q1 - pk.vg_o1) * pk.vg_inv);
    cx = min(max(cx, 0), pk.vg_nx - 1);
    cy = min(max(cy, 0), pk.vg_ny - 1);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, pk.vg_nx - 1);
    const int y0 = max(cy - 1, 0), y1 = min(cy + 1, pk.vg_ny - 1);
    double bd = INFINITY;
    unsigned bi = 0xFFFFFFFFu, dummy = 0;
    // the (at most three) row ranges are looked up together, then scanned
    int begin[3], end[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int row = y0 + r;
        begin[r] = end[r] = 0;
        if (row <= y1) {
            begin[r] = __ldg(&pk.vg_start[row * pk.vg_nx + x0]);
            end[r] = __ldg(&pk.vg_start[row * pk.vg_nx + x1 + 1]);
        }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
        for (int j = begin[r] + g.gl; j < end[r]; j += G) {
            double dx = __ldg(&pk.vx[j]) - p.x, dy = __ldg(&pk.vy[j]) - p.y, dz = __ldg(&pk.vz[j]) - p.z;
            double d = dx * dx + dy * dy + dz * dz;
            unsigned id = (unsigned)__ldg(&pk.vid[j]);
            if (d < bd || (d == bd && id < bi)) { bd = d; bi = id; }
        }
    grp_argmin<G>(bd, bi, dummy, g);
    bool proven = (x0 == 0 && y0 == 0 && x1 == pk.vg_nx - 1 && y1 == pk.vg_ny - 1);
    if (!proven) {
        // every vertex outside the scanned block is at least m away in the (axis0, axis1) plane
        double m = INFINITY;
        if (x0 > 0) m = fmin(m, q0 - (pk.vg_o0 + x0 * pk.vg_cs));
        if (x1 < pk.vg_nx - 1) m = fmin(m, (pk.vg_o0 + (x1 + 1) * pk.vg_cs) - q0);
        if (y0 > 0) m = fmin(m, q1 - (pk.vg_o1 + y0 * pk.vg_cs));
        if (y1 < pk.vg_ny - 1) m = fmin(m, (pk.vg_o1 + (y1 + 1) * pk.vg_cs) - q1);
        m -= 1e-9;
        proven = m > 0.0 && bd < m * m;
    }
    if (!proven) {
        const int n = __ldg(&pk.vg_start[pk.vg_nx * pk.vg_ny]);
        bd = INFINITY; bi = 0xFFFFFFFFu;
#pragma unroll 4
        for (int j = g.gl; j < n; j += G) {
            double dx = __ldg(&pk.vx[j]) - p.x, dy = __ldg(&pk.vy[j]) - p.y, dz = __ldg(&pk.vz[j]) - p.z;
            double d = dx * dx + dy * dy + dz * dz;
            unsigned id = (unsigned)__ldg(&pk.vid[j]);
            if (d < bd || (d == bd && id < bi)) { bd = d; bi = id; }
        }
        grp_argmin<G>(bd, bi, dummy, g);
    }
    if (bi == 0xFFFFFFFFu) return 0xFFFFFFFFu;
    return __ldg(&pk.vrec[bi]);
}

// The fast move path's copies of ray_test's / hook_triangle's slow steps: real calls (noinline) with every argument
// by value, so that their registers and loops stay out of the calling kernel's budget.  They run for a few rays in
// a hundred thousand (rays that graze a move-cell border or leave the part), but a step is as slow as its slowest
// environment: sending such an environment through the whole generic move instead costs the step tens of microseconds.
struct VertexGridArgs {       // the vertex-grid members of DevPack, same names (nearest_vertex_grid is generic over the holder)
    int vg_nx, vg_ny;
    double vg_o0, vg_o1, vg_cs, vg_inv;
    const int *vg_start;
    const double *vx, *vy, *vz;
    const int *vid;
    const unsigned *vrec;
};
__device__ __forceinline__ VertexGridArgs vertex_grid_args(const DevPack &pk) {
    VertexGridArgs a;
    a.vg_nx = pk.vg_nx; a.vg_ny = pk.vg_ny; a.vg_o0 = pk.vg_o0; a.vg_o1 = pk.vg_o1; a.vg_cs = pk.vg_cs; a.vg_inv = pk.vg_inv;
    a.vg_start = pk.vg_start; a.vx = pk.vx; a.vy = pk.vy; a.vz = pk.vz; a.vid = pk.vid; a.vrec = pk.vrec;
    return a;
}
template <int G>
__device__ __noinline__ unsigned nearest_vertex_grid_call(VertexGridArgs a, int a0, int a1, Vec3 p, Grp g) {
    Ax ax; ax.a0 = a0; ax.a1 = a1;
    return nearest_vertex_grid<G>(a, ax, p, g);
}
struct SlabAll { double t_in, t_out; int outside; unsigned args; };
template <int G>
__device__ __noinline__ SlabAll slab_pass_all_call(const double2 *planes, int n, Vec3 frm, double d0, double d1, double d2, Grp g) {
    SlabAll o;
    const SlabResult r = slab_pass_all<G>(planes, n, frm, d0, d1, d2, g, &o.args);
    o.t_in = r.t_in; o.t_out = r.t_out; o.outside = r.outside ? 1 : 0;
    return o;
}

// Part._get_hook_point + _get_closest_bary (bullet_paint_wrapper.py:525-534, 508-523, 154-185):
// incident front triangles of the nearest vertex, one per lane of the group.  Returns the picked
// triangle's record (whose tail holds n, quat_from_normal(-n) and the shot-centre offset), or nullptr.
template <int G>
__device__ __forceinline__ const double *hook_triangle(const DevPack &pk, const Ax &ax, const Vec3 &point, const CellRef &ref, double2 vc0,
                                                       double2 vc1, const Grp &g PAINTRL_PROF_PARAM) {
    unsigned rec = ref.blob ? nearest_vertex_cell<G>(point, ref, vc0, vc1, g) : nearest_vertex_grid<G>(pk, ax, point, g);
    if (!ref.blob) g_dbg_grid_searches_inc();
    PAINTRL_PROF(10, g.gl == 0);
    if (rec == 0xFFFFFFFFu) return nullptr;
    const int deg = (int)(rec & 0xffu);
    const double *base = pk.trirec + (size_t)(rec >> 8) * kTriRec;
    if (deg <= 0) return nullptr;
    int pick = -1;
    double run_max = -INFINITY;   // max of min_uvw over the triangles scanned so far
    int run_arg = -1;             // last list position attaining it
    for (int b0 = 0; b0 < deg; b0 += G) {
        int k = b0 + g.gl;
        bool inside = false;
        double m = -INFINITY;
        if (k < deg) {
            const double2 *t = reinterpret_cast<const double2 *>(base + (size_t)k * kTriRec);
            double2 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2), t3 = __ldg(t + 3), t4 = __ldg(t + 4),
                    t5 = __ldg(t + 5), t6 = __ldg(t + 6);
            // a = (t0.x t0.y t1.x)  v0 = (t1.y t2.x t2.y)  v1 = (t3.x t3.y t4.x)  d00 t4.y  d01 t5.x  d11 t5.y  inv t6.x
            double v2x = point.x - t0.x, v2y = point.y - t0.y, v2z = point.z - t1.x;
            double d20 = npdot3(v2x, v2y, v2z, t1.y, t2.x, t2.y);
            double d21 = npdot3(v2x, v2y, v2z, t3.x, t3.y, t4.x);
            double d00 = t4.y, d01 = t5.x, d11 = t5.y, inv = t6.x;
            double bv = (d11 * d20 - d01 * d21) * inv;
            double bw = (d00 * d21 - d01 * d20) * inv;
            double bu = 1.0 - bv - bw;
            if (inv == 0.0) { bu = -1.0; bv = -1.0; bw = -1.0; }
            inside = (0.0 <= bu && bu <= 1.0 && 0.0 <= bv && bv <= 1.0 && 0.0 <= bw && bw <= 1.0);
            m = fmin(fmin(bu, bv), bw);
        }
        unsigned in_mask = grp_ballot<G>(inside, g);
        if (in_mask) { pick = b0 + __ffs(in_mask) - 1; break; }
        double cm = grp_max<G>(m, g);
        if (cm >= run_max) {   // `>=`: a later triangle wins ties (bullet_paint_wrapper.py:520)
            unsigned eq = grp_ballot<G>(k < deg && m == cm, g);
            run_max = cm;
            run_arg = b0 + 31 - __clz(eq);
        }
    }
    if (pick < 0) pick = (run_max >= -1.0) ? run_arg : 0;   // closest_uvw starts at -1 (:509)
    return base + (size_t)pick * kTriRec;
}

// bullet_paint_wrapper.py:844-851
__device__ __forceinline__ int grid_index_2(const DevPack &pk, double v) {
    double rel = (v - pk.range1_min) / (pk.range1_max - pk.range1_min);
    double scaled = rel * pk.grid_granularity;
    if (!(scaled > -1.0)) return 0;
    if (scaled >= (double)pk.grid_granularity) return pk.grid_granularity - 1;
    return (int)scaled;
}

__device__ __forceinline__ double clip01(double v) { return v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v); }

// bullet_paint_wrapper.py:965-978
__device__ __forceinline__ void normalized_pose(const DevPack &pk, const Ax &ax, const Vec3 &pose, double &a1, double &a2) {
    const double radius = kPaintRadius;
    double axis1_real = comp(pose, ax.a0), axis2_real = comp(pose, ax.a1);
    double axis2_in = (axis2_real - pk.range1_min + radius) / (pk.range1_max - pk.range1_min + 2 * radius);
    int gi = grid_index_2(pk, axis2_real);
    double lo = __ldg(&pk.grid_lo[gi]), hi = __ldg(&pk.grid_hi[gi]);
    double axis1_in;
    if (hi - lo == 0.0) axis1_in = 0.0;
    else axis1_in = (axis1_real - lo + radius) / (hi - lo + 2 * radius);
    a1 = clip01(axis1_in);
    a2 = clip01(axis2_in);
}

// robot_gym_env.py:92-98
__device__ __forceinline__ int handle_pos(double pos) {
    if (pos == 0.0) return 0;
    if (pos == 1.0) return 21;
    return (int)(pos * 20) + 1;
}

// numpy float64 floor_divide (npy_divmod), used by `angle // basis` (bullet_paint_wrapper.py:1030)
__device__ __forceinline__ double np_floor_divide(double a, double b) {
    double mod = fmod(a, b);
    double div = (a - mod) / b;
    if (mod != 0.0) {
        if ((b < 0.0) != (mod < 0.0)) { mod += b; div -= 1.0; }
    }
    double fd;
    if (div != 0.0) {
        fd = floor(div);
        if (div - fd > 0.5) fd += 1.0;
    } else {
        fd = copysign(0.0, a / b);
    }
    return fd;
}

// counter-based start-index stream for auto-reset (not in the reference: it draws from the
// process-global `random`, robot_gym_env.py:381)
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

}  // namespace paintrl
