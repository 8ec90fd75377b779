// paintrl_capi.cu -- host side of the C ABI in include/paintrl.h: builds the device tables from a
// PaintrlPartPack, owns per-environment state, launches the kernels of paintrl_kernels.cuh.
// Built with: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo (paintrl_b200/build.py)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <numeric>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/paintrl.h"
#include "paintrl_kernels.cuh"
#include "paintrl_raster.cuh"
#include "paintrl_param.cuh"
#include "paintrl_policy.cuh"
#include "paintrl_learn.cuh"
#include "paintrl_replay.cuh"

using namespace paintrl;

// Batches below this many environments per GPU take the one-kernel step (a warp runs move + paint of its environment
// back to back); from here on the two-kernel step with 8-lane move groups wins (measured: profiles/).
static const int kFusedBelowEnvs = 16384;

namespace {

thread_local std::string g_error;

int fail(int code, const std::string &msg) {
    g_error = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t err__ = (expr);                                                          \
        if (err__ != cudaSuccess)                                                            \
            return fail(PAINTRL_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__)); \
    } while (0)

// Device allocations of one engine.  Read-only tables (`upload`) are carved out of a few large slabs so that the step
// kernels can prefetch all of them into L2 with one strided loop (`static_ranges`); per-environment state (`alloc`)
// gets its own allocations.
struct DeviceArena {
    static constexpr size_t kSlabBytes = size_t(24) << 20;
    struct Slab { char *base; size_t cap, used; };
    std::vector<void *> ptrs;
    std::vector<Slab> slabs;
    ~DeviceArena() {
        for (void *p : ptrs) cudaFree(p);
    }
    cudaError_t suballoc(void **out, size_t bytes) {
        bytes = (std::max<size_t>(bytes, 16) + 255) & ~size_t(255);
        if (slabs.empty() || slabs.back().used + bytes > slabs.back().cap) {
            const size_t cap = std::max(bytes, kSlabBytes);
            void *p = nullptr;
            cudaError_t e = cudaMalloc(&p, cap);
            if (e != cudaSuccess) return e;
            ptrs.push_back(p);
            slabs.push_back(Slab{static_cast<char *>(p), cap, 0});
        }
        Slab &s = slabs.back();
        *out = s.base + s.used;
        s.used += bytes;
        return cudaSuccess;
    }
    template <typename T>
    cudaError_t upload(const std::vector<T> &host, const T **out) {
        void *p = nullptr;
        cudaError_t e = suballoc(&p, host.size() * sizeof(T));
        if (e != cudaSuccess) return e;
        if (!host.empty()) {
            e = cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) return e;
        }
        *out = reinterpret_cast<const T *>(p);
        return cudaSuccess;
    }
    cudaError_t alloc(void **out, size_t bytes) {
        cudaError_t e = cudaMalloc(out, std::max<size_t>(bytes, 16));
        if (e == cudaSuccess) ptrs.push_back(*out);
        return e;
    }
    size_t static_bytes() const {
        size_t n = 0;
        for (const Slab &s : slabs) n += s.used;
        return n;
    }
};

// The prologue of every create function: a device must exist, the index must name one, and it becomes current.
int select_device(int device) {
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
        return fail(PAINTRL_E_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(err));
    if (device < 0 || device >= count) return fail(PAINTRL_E_INVALID, "device index out of range");
    CUDA_TRY(cudaSetDevice(device));
    return PAINTRL_OK;
}

// The <MO, MX> instantiation of policy_act_kernel and ppo_grad_kernel for (obs_dim, n_out): f(MO, MX) is called with
// std::integral_constant arguments.  8 / 8 covers the reference's spaces; the other three take the rest up to 32 / 16.
template <class F>
void with_caps(int obs_dim, int n_out, F &&f) {
    using k8 = std::integral_constant<int, 8>;
    using k16 = std::integral_constant<int, 16>;
    using k32 = std::integral_constant<int, 32>;
    const bool small_obs = obs_dim <= 8, small_out = n_out + 1 <= 8;
    if (small_obs && small_out) f(k8(), k8());
    else if (small_obs) f(k8(), k16());
    else if (small_out) f(k32(), k8());
    else f(k32(), k16());
}

template <class K>
bool opt_in_smem(K *kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess;
}

template <class E>
void destroy_engine(E *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    delete h;
}

}  // namespace

struct PaintrlEngine {
    int device = 0;
    int num_envs = 0;
    int color = 0;
    DevPack pk{};
    DevConfig cfg{};
    DeviceArena arena;
    EnvState *states = nullptr;
    MoveOut *moves = nullptr;
    EnvStat *env_stats = nullptr;
    unsigned *bits = nullptr;        // [num_envs][n_words_pad] flip bit per texel slot
    int16_t *thick = nullptr;        // [num_envs][n_slots] HSI thickness plane (HSI only)
    unsigned *grid_cnt = nullptr;    // [num_envs][n_gcells_pad] (grid observation only)
    unsigned long long *stats = nullptr;
    ShotPoses *shots = nullptr;      // [num_envs] normal paint method: pose / orientation of the step's five shots
    unsigned *last_mask = nullptr;   // [num_envs][n_words_pad] normal paint method: texels of the previous shot
    bool paint_normal = false;
    unsigned *ready = nullptr;       // [num_envs] per-environment move -> paint hand-off flags: 1 = this step's move output is published;
                                     // the paint warp clears it.  All steps of one handle must be issued on ONE stream (or ordered streams).
    // staging for the host-buffer entry points
    void *stage_actions = nullptr;
    // paintrl_step_host: one contiguous block, laid out per call as obs | reward | penalty | actual | [next_obs] | done,
    // so that host buffers carved from one allocation in that order come back with a single copy
    unsigned char *stage_out = nullptr;
    // paintrl_step_host_submit / _wait: two staging slots, a copy-in and a copy-out stream of the library's own, so that
    // step t + 1's host->device copy and launch overlap step t's device->host copy and the host's wake-up
    void *slot_actions[2] = {nullptr, nullptr};
    unsigned char *slot_out[2] = {nullptr, nullptr};
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_step[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    bool slot_pending[2] = {false, false};
    unsigned long long launches = 0;
    double move_cell_planes_mean = 0.0, move_cell_verts_mean = 0.0;
    int move_lanes = 32;             // lanes per environment in move_fast_kernel of the two-kernel step (8 or 32)
    void *cold_args = nullptr;       // device copy of {pk, cfg, env arrays} for the paint warps' generic-move call (ColdArgs)
    int fused = -1;                  // PAINTRL_FUSED: 1 / 0 force the one-kernel / two-kernel step; -1: by batch size
    bool force_unstaged = false;     // PAINTRL_FORCE_UNSTAGED: run the global-memory bit-plane path (tests)
};

namespace {

// Host copy of the slab test (same formula as the device's; used only to sample the hull while
// building the move cells, so its rounding does not matter).  Optionally reports the planes that
// attain t_in / t_out.
bool host_ray(const PaintrlPartPack *pack, const double *frm, const double *d, double *t_hit, int *arg_in = nullptr,
              int *arg_out = nullptr) {
    double t_in = -INFINITY, t_out = INFINITY;
    int ai = -1, ao = -1;
    bool outside = false;
    for (int i = 0; i < pack->n_planes; ++i) {
        const double *n = pack->plane_n + 3 * i;
        double den = n[0] * d[0] + n[1] * d[1] + n[2] * d[2];
        double num = pack->plane_off[i] - (n[0] * frm[0] + n[1] * frm[1] + n[2] * frm[2]);
        if (den == 0.0) {
            if (num < 0.0) { outside = true; if (ai < 0) ai = i; }
            continue;
        }
        double t = num / den;
        if (den < 0.0) { if (t > t_in) { t_in = t; ai = i; } }
        else { if (t < t_out) { t_out = t; ao = i; } }
    }
    if (arg_in) *arg_in = ai;
    if (arg_out) *arg_out = ao;
    if (outside || !(t_in <= t_out) || !std::isfinite(t_in)) return false;
    *t_hit = t_in;
    return true;
}

// Move cells (see ray_test / nearest_vertex_cell in paintrl_device.cuh): a grid over (axis0, axis1).
// Cells under the hull: depth range [dlo, dhi] of the hull's tool-side surface over the cell
// (sampled, padded), the planes not satisfied with margin at every point of the box
// footprint x [dlo, dhi], and the front vertices that can be nearest to a point of the box.
// Only the two lists must be conservative; the depth range merely decides how often the fast path
// is accepted.  Cells beside the hull: the planes that decide a few sample rays (a miss is then
// usually proven from the list alone; nothing depends on it).
int build_move_cells(PaintrlEngine *e, const PaintrlPartPack *pack, const std::vector<int> &front,
                     const std::vector<unsigned> &vrec) {
    DevPack &pk = e->pk;
    pk.mc_nx = pk.mc_ny = 0;
    const int a0 = pack->axis0, a1 = pack->axis1, np = 3 - a0 - a1;
    const double cs = kPaintRadius / 4, pad = 0.15;
    const double o0 = pack->range0_min - pad, o1 = pack->range1_min - pad;
    int nx = (int)std::ceil((pack->range0_max + pad - o0) / cs), ny = (int)std::ceil((pack->range1_max + pad - o1) / cs);
    std::vector<uint2> entries;
    std::vector<double> blob;         // 4 doubles per 32-byte sector
    if (nx <= 0 || ny <= 0 || (long long)nx * ny > (1 << 21)) nx = ny = 0;   // fast path off
    entries.resize((size_t)nx * ny);
    std::vector<int> pidx;            // the current cell's plane indices
    std::vector<VertCand> vcs;        // the current cell's vertex candidates
    size_t plane_refs = 0;
    const double kPadBelow = 5e-4, kPadBelowEdge = 0.025, kPadAbove = 1e-4, kFootSlack = 1e-6, kMargin = 1e-9, kVertSlack = 1e-9;
    const int K = 5;
    // the tool hovers on the side the start normals point away from and looks along them
    const double side = pack->start_normal[np] <= 0.0 ? 1.0 : -1.0;
    double dir[3] = {0, 0, 0};
    dir[np] = -side;
    double hull_top = -INFINITY;   // highest tool-side depth of the hull (in tool-side units)
    for (int v = 0; v < pack->n_vertices; ++v) {
        const double *p = pack->vertices + 3 * v;
        if (p[0] == 10.0 && p[1] == 10.0 && p[2] == 10.0) continue;
        hull_top = std::max(hull_top, side * p[np]);
    }
    size_t planes_total = 0, verts_total = 0, inside_cells = 0;
    std::vector<int> tmp;
    for (int cy = 0; cy < ny; ++cy) {
        for (int cx = 0; cx < nx; ++cx) {
            struct { double a, b, c, rlo, rhi; int n_planes, n_verts; } mc = {0.0, 0.0, 0.0, 1.0, -1.0, 0, 0};
            pidx.clear();
            vcs.clear();
            unsigned long long fallback_link = 0;   // (sector offset | counts << 32) of the cell's fallback blob, 0: none
            bool too_long = false;
            // appends the blob of the current (mc, pidx, vcs) and returns its entry word: offset | n_planes << 32 | n_verts << 48
            auto emit_blob = [&]() -> unsigned long long {
                if (mc.n_planes > 0xffff || mc.n_verts > 0xffff || blob.size() / 4 > 0xfffffff0u) { too_long = true; return 0ull; }
                const unsigned long long word = (unsigned long long)(blob.size() / 4) | ((unsigned long long)mc.n_planes << 32) |
                                                ((unsigned long long)mc.n_verts << 48);
                double hdr[8] = {mc.a, mc.b, mc.c, mc.rlo, mc.rhi, 0.0, 0.0, 0.0};
                std::memcpy(&hdr[5], &fallback_link, 8);
                fallback_link = 0;
                blob.insert(blob.end(), hdr, hdr + 8);
                for (int p : pidx) {
                    const double pl[4] = {pack->plane_n[3 * p], pack->plane_n[3 * p + 1], pack->plane_n[3 * p + 2], pack->plane_off[p]};
                    blob.insert(blob.end(), pl, pl + 4);
                }
                for (const VertCand &vc : vcs) {
                    double v[4] = {vc.x, vc.y, vc.z, 0.0};
                    const unsigned long long meta = (unsigned long long)vc.id | ((unsigned long long)vc.rec << 32);
                    std::memcpy(&v[3], &meta, 8);
                    blob.insert(blob.end(), v, v + 4);
                }
                plane_refs += pidx.size();
                return word;
            };
            const double lo0 = o0 + cx * cs, hi0 = o0 + (cx + 1) * cs, lo1 = o1 + cy * cs, hi1 = o1 + (cy + 1) * cs;
            const double mid0 = 0.5 * (lo0 + hi0), mid1 = 0.5 * (lo1 + hi1);
            // sample the hull's tool-side surface over the footprint
            double sx[K * K], sy[K * K], sd[K * K];
            int hits = 0;
            for (int i = 0; i < K; ++i) {
                for (int j = 0; j < K; ++j) {
                    double frm[3];
                    frm[a0] = lo0 + (hi0 - lo0) * i / (K - 1);
                    frm[a1] = lo1 + (hi1 - lo1) * j / (K - 1);
                    frm[np] = side * 100.0;
                    double t;
                    if (host_ray(pack, frm, dir, &t)) {
                        sx[hits] = frm[a0] - mid0; sy[hits] = frm[a1] - mid1; sd[hits] = frm[np] + dir[np] * t;
                        ++hits;
                    }
                }
            }
            // plane fitted to the samples: depth ~ fa + fb (x0 - mid0) + fc (x1 - mid1)
            bool region = false;
            double fa = 0, fb = 0, fc = 0;
            if (hits >= 4) {
                double sxx = 0, sxy = 0, syy = 0, sx1 = 0, sy1 = 0, sxd = 0, syd = 0, sd1 = 0;
                for (int q = 0; q < hits; ++q) {
                    sxx += sx[q] * sx[q]; sxy += sx[q] * sy[q]; syy += sy[q] * sy[q];
                    sx1 += sx[q]; sy1 += sy[q]; sxd += sx[q] * sd[q]; syd += sy[q] * sd[q]; sd1 += sd[q];
                }
                const double n = hits;
                // normal equations [[n sx1 sy1] [sx1 sxx sxy] [sy1 sxy syy]] (fa fb fc) = (sd1 sxd syd)
                const double det = n * (sxx * syy - sxy * sxy) - sx1 * (sx1 * syy - sxy * sy1) + sy1 * (sx1 * sxy - sxx * sy1);
                if (std::fabs(det) > 1e-12 * n * (cs * cs) * (cs * cs)) {
                    fa = (sd1 * (sxx * syy - sxy * sxy) - sx1 * (sxd * syy - sxy * syd) + sy1 * (sxd * sxy - sxx * syd)) / det;
                    fb = (n * (sxd * syy - syd * sxy) - sd1 * (sx1 * syy - sxy * sy1) + sy1 * (sx1 * syd - sxd * sy1)) / det;
                    fc = (n * (sxx * syd - sxy * sxd) - sx1 * (sx1 * syd - sxd * sy1) + sd1 * (sx1 * sxy - sxx * sy1)) / det;
                    region = std::isfinite(fa) && std::isfinite(fb) && std::isfinite(fc);
                }
            }
            if (!region && hits >= 1) {
                // a corner or one edge of the footprint under the hull (too few samples, or all on one line:
                // the fit is singular): constant plane through the mean sampled depth
                fa = fb = fc = 0;
                for (int q = 0; q < hits; ++q) fa += sd[q] / hits;
                region = std::isfinite(fa);
            }
            if (region) {
                // ---- the hull surface passes over the cell: region hugging it
                double rmin = INFINITY, rmax = -INFINITY;
                for (int q = 0; q < hits; ++q) {
                    const double res = sd[q] - (fa + fb * sx[q] + fc * sy[q]);
                    rmin = std::min(rmin, res); rmax = std::max(rmax, res);
                }
                // tool side is +side: above the surface = larger side * depth.  A cell the silhouette of the hull
                // runs through (not every sample ray hit) also holds part of the hull's side wall, which tilted rays
                // enter well below the tool-side surface: its slab reaches kPadBelowEdge down (measured: entry
                // points up to 14 mm below the fitted plane; such cells sent 1 % of the environments through
                // the verify pass on every sub-step and were the tail of the move phase).
                // Two tiers for such cells: the PRIMARY region is the thin slab of an ordinary cell (short lists: almost
                // every ray enters through the tool-side surface), the deep slab is a FALLBACK blob linked from the
                // primary's header, tried when the entry point lies in this cell but not in the thin slab.  With the deep
                // slab alone these cells carried 80 planes and up to 258 vertex candidates (mean 16 / 14 elsewhere) and
                // their environments were the tail of the move phase.
                const bool edge_cell = hits < K * K;
                auto build_lists = [&](double below) {
                    pidx.clear();
                    vcs.clear();
                    const double rlo = rmin - (side > 0 ? below : kPadAbove), rhi = rmax + (side > 0 ? kPadAbove : below);
                    mc.a = fa - fb * mid0 - fc * mid1;
                    mc.b = fb;
                    mc.c = fc;
                    mc.rlo = rlo;
                    mc.rhi = rhi;
                    double corner[8][3];
                    double zmin = INFINITY, zmax = -INFINITY;
                    for (int c = 0; c < 8; ++c) {
                        corner[c][a0] = (c & 1) ? hi0 + kFootSlack : lo0 - kFootSlack;
                        corner[c][a1] = (c & 2) ? hi1 + kFootSlack : lo1 - kFootSlack;
                        corner[c][np] = mc.a + mc.b * corner[c][a0] + mc.c * corner[c][a1] + ((c & 4) ? rhi : rlo);
                        zmin = std::min(zmin, corner[c][np]); zmax = std::max(zmax, corner[c][np]);
                    }
                    zmin -= 1e-9; zmax += 1e-9;
                    for (int p = 0; p < pack->n_planes; ++p) {
                        const double *n = pack->plane_n + 3 * p;
                        double worst = -INFINITY;
                        for (int c = 0; c < 8; ++c)
                            worst = std::max(worst, n[0] * corner[c][0] + n[1] * corner[c][1] + n[2] * corner[c][2]);
                        if (worst > pack->plane_off[p] - kMargin) pidx.push_back(p);
                    }
                    mc.n_planes = (int)pidx.size();
                    // candidates for the nearest front vertex of any point of the region (its bounding box)
                    double blo[3], bhi[3];
                    blo[a0] = lo0 - kFootSlack; bhi[a0] = hi0 + kFootSlack;
                    blo[a1] = lo1 - kFootSlack; bhi[a1] = hi1 + kFootSlack;
                    blo[np] = zmin; bhi[np] = zmax;
                    double best_far = INFINITY;
                    for (int v : front) {
                        const double *p = pack->vertices + 3 * v;
                        double far2 = 0;
                        for (int k = 0; k < 3; ++k) {
                            double f = std::max(std::fabs(p[k] - blo[k]), std::fabs(p[k] - bhi[k]));
                            far2 += f * f;
                        }
                        best_far = std::min(best_far, std::sqrt(far2));
                    }
                    for (int v : front) {
                        const double *p = pack->vertices + 3 * v;
                        double near2 = 0;
                        for (int k = 0; k < 3; ++k) {
                            double g = std::max(0.0, std::max(blo[k] - p[k], p[k] - bhi[k]));
                            near2 += g * g;
                        }
                        if (std::sqrt(near2) <= best_far + kVertSlack) {
                            VertCand vc;
                            vc.x = p[0]; vc.y = p[1]; vc.z = p[2];
                            vc.id = (unsigned)v;
                            vc.rec = vrec[v];
                            vcs.push_back(vc);
                        }
                    }
                    // Pruning by domination: vertex v cannot be nearest to any point q of the box if another candidate u is
                    // strictly closer everywhere in it: |q-u|^2 < |q-v|^2  <=>  2 q.(v-u) < |v|^2 - |u|^2, linear in q, so
                    // the box corner that maximises the left side decides (slack 1e-9: far above FP64 round-off of the
                    // device's squared distances, so a dropped vertex is never nearest and never tied).  The box criterion
                    // alone keeps everything in a ring as wide as the box around the nearest vertex -- hundreds of vertices
                    // over a flat face whose own vertices are far away.
                    if (vcs.size() > 8) {
                        const size_t n = vcs.size();
                        std::vector<double> c0(n);          // distance from the box centre: likely dominators first
                        const double ctr[3] = {0.5 * (blo[0] + bhi[0]), 0.5 * (blo[1] + bhi[1]), 0.5 * (blo[2] + bhi[2])};
                        std::vector<int> order(n);
                        for (size_t i = 0; i < n; ++i) {
                            const double dx = vcs[i].x - ctr[0], dy = vcs[i].y - ctr[1], dz = vcs[i].z - ctr[2];
                            c0[i] = dx * dx + dy * dy + dz * dz;
                            order[i] = (int)i;
                        }
                        std::sort(order.begin(), order.end(), [&](int x, int y) { return c0[x] < c0[y]; });
                        std::vector<char> keep(n, 1);
                        const size_t n_dom = std::min<size_t>(n, 24);
                        for (size_t i = 0; i < n; ++i) {
                            const VertCand &v = vcs[i];
                            const double v2 = v.x * v.x + v.y * v.y + v.z * v.z;
                            for (size_t j = 0; j < n_dom; ++j) {
                                const int ui = order[j];
                                if ((size_t)ui == i) continue;
                                const VertCand &u = vcs[ui];
                                const double d[3] = {2.0 * (v.x - u.x), 2.0 * (v.y - u.y), 2.0 * (v.z - u.z)};
                                double lhs = 0.0;
                                for (int k = 0; k < 3; ++k) lhs += std::max(d[k] * blo[k], d[k] * bhi[k]);
                                const double rhs = v2 - (u.x * u.x + u.y * u.y + u.z * u.z);
                                if (lhs < rhs - 1e-9) { keep[i] = 0; break; }
                            }
                        }
                        // a dominator is never dominated itself by something it dominates: the nearest vertex of the box
                        // centre always survives, so the list cannot come out empty
                        size_t w = 0;
                        for (size_t i = 0; i < n; ++i)
                            if (keep[i]) vcs[w++] = vcs[i];
                        vcs.resize(w);
                    }
                    mc.n_verts = (int)vcs.size();
};
                if (edge_cell) {
                    build_lists(kPadBelowEdge);
                    fallback_link = emit_blob();
                }
                build_lists(kPadBelow);
                planes_total += mc.n_planes;
                verts_total += mc.n_verts;
                ++inside_cells;
            } else {
                // ---- beside (or straddling the edge of) the hull: planes deciding a few sample rays
                tmp.clear();
                const double tilt = 0.35;
                const double sample[9][4] = {{mid0, mid1, 0, 0},    {mid0, mid1, tilt, 0}, {mid0, mid1, -tilt, 0},
                                             {mid0, mid1, 0, tilt}, {mid0, mid1, 0, -tilt}, {lo0, lo1, 0, 0},
                                             {hi0, lo1, 0, 0},      {lo0, hi1, 0, 0},       {hi0, hi1, 0, 0}};
                for (int q = 0; q < 9; ++q) {
                    double frm[3], d[3];
                    frm[a0] = sample[q][0]; frm[a1] = sample[q][1];
                    frm[np] = side * (hull_top + kHookDistance);
                    d[a0] = sample[q][2]; d[a1] = sample[q][3]; d[np] = -side;
                    double nrm = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
                    for (int k = 0; k < 3; ++k) d[k] /= nrm;
                    double t;
                    int ai, ao;
                    host_ray(pack, frm, d, &t, &ai, &ao);
                    if (ai >= 0) tmp.push_back(ai);
                    if (ao >= 0) tmp.push_back(ao);
                }
                std::sort(tmp.begin(), tmp.end());
                tmp.erase(std::unique(tmp.begin(), tmp.end()), tmp.end());
                for (int p : tmp) pidx.push_back(p);
                mc.n_planes = (int)tmp.size();
            }
            // ---- the cell's blob: region, copies of its planes, its vertex candidates
            if (too_long) return fail(PAINTRL_E_INVALID, "move cell list too long");
            const unsigned long long primary = emit_blob();
            if (too_long) return fail(PAINTRL_E_INVALID, "move cell list too long");
            uint2 &en = entries[(size_t)cy * nx + cx];
            en.x = (unsigned)(primary & 0xffffffffu);
            en.y = (unsigned)(primary >> 32);
        }
    }
    blob.resize(blob.size() + 4 * 64, 0.0);   // lanes may read one round of sectors past a short list
    pk.mc_nx = nx; pk.mc_ny = ny;
    pk.mc_o0 = o0; pk.mc_o1 = o1; pk.mc_inv = 1.0 / cs;
    CUDA_TRY(e->arena.upload(entries, &pk.mc_entry));
    {
        const double *dev = nullptr;
        CUDA_TRY(e->arena.upload(blob, &dev));
        pk.mc_blob = reinterpret_cast<const double2 *>(dev);
    }
    e->move_cell_planes_mean = inside_cells ? (double)planes_total / inside_cells : 0.0;
    e->move_cell_verts_mean = inside_cells ? (double)verts_total / inside_cells : 0.0;
    if (getenv("PAINTRL_DEBUG"))
        fprintf(stderr, "[paintrl] move cells %d x %d, %zu with a surface region: %.2f planes, %.2f vertex candidates per cell; %zu plane refs, blobs %.1f MB\n",
                nx, ny, inside_cells, e->move_cell_planes_mean, e->move_cell_verts_mean, plane_refs, blob.size() * 8 / 1e6);
    return PAINTRL_OK;
}

inline float ulp_f32(float v) { return std::nextafter(std::fabs(v), INFINITY) - std::fabs(v); }

// Host-side construction of the acceleration tables (see DESIGN.md "Data layout in HBM").
int build_tables(PaintrlEngine *e, const PaintrlPartPack *pack, const PaintrlConfig *cfg) {
    DevPack &pk = e->pk;
    const int n = pack->n_texels;
    const int a0 = pack->axis0, a1 = pack->axis1;
    pk.n_texels = n;
    pk.axis0 = a0;
    pk.axis1 = a1;
    pk.status_init = pack->status_init;

    // ---- collision planes
    pk.n_planes = pack->n_planes;
    std::vector<double4> planes(pack->n_planes);
    for (int i = 0; i < pack->n_planes; ++i)
        planes[i] = make_double4(pack->plane_n[3 * i], pack->plane_n[3 * i + 1], pack->plane_n[3 * i + 2], pack->plane_off[i]);
    CUDA_TRY(e->arena.upload(planes, &pk.planes));

    // ---- incident-triangle records per vertex (uv_map order): barycentric constants, corrected
    // normal n, and for orn = -n the quaternion (robot.py:93-100) and shot-centre offset
    // R(q)(0,0,0.1) (robot.py:277-278), evaluated here with the very functions the device uses.
    for (int i = 0; i < pack->vtri_start[pack->n_vertices]; ++i)
        if (pack->vtri_idx[i] < 0 || pack->vtri_idx[i] >= pack->n_tris) return fail(PAINTRL_E_INVALID, "vtri_idx out of range");
    std::vector<unsigned> vrec(pack->n_vertices, 0xFFFFFFFFu);
    {
        const int n_rec = pack->vtri_start[pack->n_vertices];
        if (n_rec >= (1 << 24)) return fail(PAINTRL_E_INVALID, "too many vertex-triangle incidences");
        std::vector<double> rec((size_t)std::max(n_rec, 1) * kTriRec, 0.0);
        for (int v = 0; v < pack->n_vertices; ++v) {
            const int begin = pack->vtri_start[v], deg = pack->vtri_start[v + 1] - begin;
            if (deg > 255) return fail(PAINTRL_E_INVALID, "vertex with more than 255 incident front triangles");
            vrec[v] = ((unsigned)begin << 8) | (unsigned)deg;
            for (int k = 0; k < deg; ++k) {
                const int t = pack->vtri_idx[begin + k];
                double *o = &rec[(size_t)(begin + k) * kTriRec];
                for (int c = 0; c < 3; ++c) {
                    o[c] = pack->tri_a[3 * t + c];
                    o[3 + c] = pack->tri_v0[3 * t + c];
                    o[6 + c] = pack->tri_v1[3 * t + c];
                    o[13 + c] = pack->tri_n[3 * t + c];
                }
                o[9] = pack->tri_d00[t]; o[10] = pack->tri_d01[t]; o[11] = pack->tri_d11[t]; o[12] = pack->tri_inv_denom[t];
                Vec3 orn = {-o[13], -o[14], -o[15]};
                quat_from_normal(orn, o + 16);
                const Vec3 zero = {0.0, 0.0, 0.0};
                Vec3 off = transform_point(zero, o + 16, 0.0, 0.0, 0.1);
                // transform_point adds pos last: (rot + 0.0) == rot exactly except for -0.0, which the
                // device-side `off + pos` cannot distinguish either
                o[20] = off.x; o[21] = off.y; o[22] = off.z;
            }
        }
        CUDA_TRY(e->arena.upload(rec, &pk.trirec));
        CUDA_TRY(e->arena.upload(vrec, &pk.vrec));
    }

    // ---- vertex grid for the slow path (vertices parked at IRRELEVANT_POSE (10,10,10) can never be nearest; skip them)
    std::vector<int> front;
    for (int v = 0; v < pack->n_vertices; ++v) {
        const double *p = pack->vertices + 3 * v;
        if (p[0] == 10.0 && p[1] == 10.0 && p[2] == 10.0) continue;
        front.push_back(v);
    }
    if (front.empty()) return fail(PAINTRL_E_INVALID, "part pack has no front-side vertices");
    double vmin0 = INFINITY, vmax0 = -INFINITY, vmin1 = INFINITY, vmax1 = -INFINITY;
    for (int v : front) {
        const double *p = pack->vertices + 3 * v;
        vmin0 = std::min(vmin0, p[a0]); vmax0 = std::max(vmax0, p[a0]);
        vmin1 = std::min(vmin1, p[a1]); vmax1 = std::max(vmax1, p[a1]);
    }
    double area = std::max((vmax0 - vmin0) * (vmax1 - vmin1), 1e-12);
    pk.vg_cs = std::max(2.0 * std::sqrt(area / (double)front.size()), 1e-6);
    pk.vg_inv = 1.0 / pk.vg_cs;
    pk.vg_o0 = vmin0;
    pk.vg_o1 = vmin1;
    pk.vg_nx = std::min(4096, (int)std::floor((vmax0 - vmin0) * pk.vg_inv) + 1);
    pk.vg_ny = std::min(4096, (int)std::floor((vmax1 - vmin1) * pk.vg_inv) + 1);
    {
        const int cells = pk.vg_nx * pk.vg_ny;
        std::vector<int> cell_of(front.size());
        std::vector<int> start(cells + 1, 0);
        for (size_t i = 0; i < front.size(); ++i) {
            const double *p = pack->vertices + 3 * front[i];
            int cx = std::min(std::max((int)std::floor((p[a0] - pk.vg_o0) * pk.vg_inv), 0), pk.vg_nx - 1);
            int cy = std::min(std::max((int)std::floor((p[a1] - pk.vg_o1) * pk.vg_inv), 0), pk.vg_ny - 1);
            cell_of[i] = cy * pk.vg_nx + cx;
            start[cell_of[i] + 1]++;
        }
        for (int c = 0; c < cells; ++c) start[c + 1] += start[c];
        std::vector<int> order(front.size());
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return cell_of[x] < cell_of[y]; });
        std::vector<double> vx(front.size()), vy(front.size()), vz(front.size());
        std::vector<int> vid(front.size());
        for (size_t j = 0; j < order.size(); ++j) {
            int v = front[order[j]];
            vx[j] = pack->vertices[3 * v];
            vy[j] = pack->vertices[3 * v + 1];
            vz[j] = pack->vertices[3 * v + 2];
            vid[j] = v;
        }
        CUDA_TRY(e->arena.upload(start, &pk.vg_start));
        CUDA_TRY(e->arena.upload(vx, &pk.vx));
        CUDA_TRY(e->arena.upload(vy, &pk.vy));
        CUDA_TRY(e->arena.upload(vz, &pk.vz));
        CUDA_TRY(e->arena.upload(vid, &pk.vid));
    }
    {
        int rc = build_move_cells(e, pack, front, vrec);
        if (rc != PAINTRL_OK) return rc;
    }

    // ---- texel layout "rows and words": rows = strips along axis1 (row(y) = floor((y - o1) * inv)),
    // the texels of a row sorted by their axis0 coordinate and packed 32 to a word, every row starting
    // a new word.  A static cell table along axis0 (cell(x) = floor((x - o0) * inv)) gives, per row,
    // the index of the first texel of each cell.
    double tmin0 = INFINITY, tmax0 = -INFINITY, tmin1 = INFINITY, tmax1 = -INFINITY;
    double tmin[3] = {INFINITY, INFINITY, INFINITY}, tmax[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = 0; i < n; ++i) {
        const double *p = pack->texel_pos + 3 * i;
        tmin0 = std::min(tmin0, p[a0]); tmax0 = std::max(tmax0, p[a0]);
        tmin1 = std::min(tmin1, p[a1]); tmax1 = std::max(tmax1, p[a1]);
        for (int k = 0; k < 3; ++k) { tmin[k] = std::min(tmin[k], p[k]); tmax[k] = std::max(tmax[k], p[k]); }
    }
    const double ext0 = std::max(tmax0 - tmin0, 1e-9), ext1 = std::max(tmax1 - tmin1, 1e-9);
    pk.n_rows = (n / 32 <= 4096) ? 32 : kMaxRows;
    pk.row_h = ext1 * (1.0 + 1e-9) / pk.n_rows;
    pk.row_inv = 1.0 / pk.row_h;
    pk.row_o1 = tmin1;
    pk.ncx = (int)std::min<long long>(std::max<long long>((long long)n / (2 * pk.n_rows), 16), 1 << 20);
    pk.cx_inv = pk.ncx / (ext0 * (1.0 + 1e-9));
    pk.cx_o0 = tmin0;
    std::vector<int> row_of(n), cell_of(n);
    std::vector<int> row_count(pk.n_rows, 0);
    for (int i = 0; i < n; ++i) {
        const double *p = pack->texel_pos + 3 * i;
        // the same two FP64 operations the device applies to the TCP (section4_counts / row_ranks)
        const int r = (int)std::floor((p[a1] - pk.row_o1) * pk.row_inv);
        const int c = (int)std::floor((p[a0] - pk.cx_o0) * pk.cx_inv);
        if (r < 0 || r >= pk.n_rows || c < 0 || c >= pk.ncx) return fail(PAINTRL_E_INVALID, "texel outside its own row / cell grid");
        row_of[i] = r;
        cell_of[i] = c;
        row_count[r]++;
    }
    std::vector<int> row_word0(pk.n_rows + 1, 0);
    for (int r = 0; r < pk.n_rows; ++r) {
        const int words = (row_count[r] + 31) / 32;
        if (words >= (1 << 18)) return fail(PAINTRL_E_INVALID, "texel row too long");
        row_word0[r + 1] = row_word0[r] + words;
    }
    pk.n_words = std::max(row_word0[pk.n_rows], 1);
    pk.n_words_pad = ((pk.n_words + 31) / 32) * 32;
    pk.n_slots = pk.n_words * 32;
    std::vector<int> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
        if (row_of[x] != row_of[y]) return row_of[x] < row_of[y];
        return pack->texel_pos[3 * x + a0] < pack->texel_pos[3 * y + a0];
    });
    std::vector<int> slot_to_pack(pk.n_slots, -1), pack_to_slot(n, 0);
    std::vector<int> cell_start((size_t)pk.n_rows * (pk.ncx + 1), 0);
    std::vector<unsigned> word_info(pk.n_words, 0);
    {
        int pos = 0;
        for (int r = 0; r < pk.n_rows; ++r) {
            int *cs = &cell_start[(size_t)r * (pk.ncx + 1)];
            int c_next = 0;
            for (int i = 0; i < row_count[r]; ++i) {
                const int t = order[pos + i];
                const int slot = row_word0[r] * 32 + i;
                slot_to_pack[slot] = t;
                pack_to_slot[t] = slot;
                while (c_next <= cell_of[t]) cs[c_next++] = i;   // monotone: the row is sorted by axis0
            }
            while (c_next <= pk.ncx) cs[c_next++] = row_count[r];
            for (int w = row_word0[r]; w < row_word0[r + 1]; ++w) {
                const int wi = w - row_word0[r];
                const int valid = std::min(32, row_count[r] - 32 * wi);
                word_info[w] = (unsigned)r | ((unsigned)valid << 8) | ((unsigned)wi << 14);
            }
            pos += row_count[r];
        }
    }
    CUDA_TRY(e->arena.upload(row_word0, &pk.row_word0));
    CUDA_TRY(e->arena.upload(row_count, &pk.row_count));
    CUDA_TRY(e->arena.upload(cell_start, &pk.cell_start));
    CUDA_TRY(e->arena.upload(word_info, &pk.word_info));
    CUDA_TRY(e->arena.upload(slot_to_pack, &pk.slot_to_pack));
    CUDA_TRY(e->arena.upload(pack_to_slot, &pk.pack_to_slot));
    {   // normal paint method: the kd-tree's twin among texels at one position (PaintrlPartPack::texel_nn_rep), per slot
        std::vector<int> rep(pk.n_slots, 0);
        for (int j = 0; j < pk.n_slots; ++j) {
            const int t = slot_to_pack[j];
            int r = t;
            if (t >= 0 && pack->texel_nn_rep) {
                r = pack->texel_nn_rep[t];
                if (r < 0 || r >= n) return fail(PAINTRL_E_INVALID, "texel_nn_rep out of range");
            }
            rep[j] = t >= 0 ? pack_to_slot[r] : j;
        }
        CUDA_TRY(e->arena.upload(rep, &pk.nn_rep_slot));
        // Nearest-texel grid of the normal paint method (Part.paint's cKDTree.query, bullet_paint_wrapper.py:565): square
        // cells of two texel pitches over the principal plane, the texels of a cell stored together as (x, y, z, slot) --
        // a query scans a 3 x 3 block of about 36 texels instead of whole stretches of the 37 mm rows of the step's layout.
        pk.nn_nx = pk.nn_ny = 0;
        if (cfg->paint_method == 1 && n > 0) {
            double lo0 = INFINITY, hi0 = -INFINITY, lo1 = INFINITY, hi1 = -INFINITY;
            for (int t = 0; t < n; ++t) {
                const double *p = pack->texel_pos + 3 * t;
                lo0 = std::min(lo0, p[a0]); hi0 = std::max(hi0, p[a0]);
                lo1 = std::min(lo1, p[a1]); hi1 = std::max(hi1, p[a1]);
            }
            const double area = std::max((hi0 - lo0) * (hi1 - lo1), 1e-12);
            const double g = std::max(2.0 * std::sqrt(area / n), 1e-6);
            const int nx = std::max(1, std::min(4096, (int)std::floor((hi0 - lo0) / g) + 1));
            const int ny = std::max(1, std::min(4096, (int)std::floor((hi1 - lo1) / g) + 1));
            const double inv = 1.0 / g;
            auto cell_of = [&](const double *p) {
                const int cx = std::min(std::max((int)std::floor((p[a0] - lo0) * inv), 0), nx - 1);
                const int cy = std::min(std::max((int)std::floor((p[a1] - lo1) * inv), 0), ny - 1);
                return cy * nx + cx;
            };
            std::vector<int> start((size_t)nx * ny + 1, 0);
            for (int t = 0; t < n; ++t) start[cell_of(pack->texel_pos + 3 * t) + 1]++;
            for (size_t c = 0; c < (size_t)nx * ny; ++c) start[c + 1] += start[c];
            std::vector<int> fill(start.begin(), start.end() - 1);
            std::vector<double> pos4((size_t)n * 4, 0.0);
            for (int j = 0; j < pk.n_slots; ++j) {          // in slot order: ties inside a cell go to the lower slot, as before
                const int t = slot_to_pack[j];
                if (t < 0) continue;
                const double *p = pack->texel_pos + 3 * t;
                const size_t at = (size_t)fill[cell_of(p)]++;
                pos4[4 * at] = p[0]; pos4[4 * at + 1] = p[1]; pos4[4 * at + 2] = p[2];
                const long long slot = j;
                std::memcpy(&pos4[4 * at + 3], &slot, 8);
            }
            pk.nn_nx = nx; pk.nn_ny = ny;
            pk.nn_o0 = lo0; pk.nn_o1 = lo1; pk.nn_inv = inv; pk.nn_cell = g;
            CUDA_TRY(e->arena.upload(start, &pk.nn_start));
            const double *dev = nullptr;
            CUDA_TRY(e->arena.upload(pos4, &dev));
            pk.nn_pos = reinterpret_cast<const double2 *>(dev);
        }
    }

    // ---- grid-observation cells (bullet_paint_wrapper.py:1072-1112)
    std::vector<uint16_t> gcell(pk.n_slots, 0);
    pk.n_gcells = pk.n_gcells_pad = 0;
    pk.gtotal = nullptr;
    pk.gcell = nullptr;
    if (cfg->obs_mode == PAINTRL_OBS_GRID) {
        const int g = cfg->obs_grad, vgran = pack->grid_granularity;
        const int v_interval = (int)((double)vgran / (double)g);
        if (v_interval <= 0) return fail(PAINTRL_E_INVALID, "OBS_GRAD larger than GRID_GRANULARITY");
        const double axis_2_step = (pack->range1_max - pack->range1_min) / vgran;
        std::vector<int> gtotal((size_t)g * g, 0);
        for (int j = 0; j < pk.n_slots; ++j) {
            if (slot_to_pack[j] < 0) continue;
            const double *p = pack->texel_pos + 3 * slot_to_pack[j];
            double yq = (p[a1] - pack->range1_min) / axis_2_step;
            if (!(yq > -1.0)) return fail(PAINTRL_E_INVALID, "texel below the silhouette table (reference KeyError)");
            int y_grid = std::min(vgran - 1, (int)yq);
            double range = pack->grid_hi[y_grid] - pack->grid_lo[y_grid];
            int x_grid = 0;
            if (range != 0) {
                double x_step = range / g;
                double xq = (p[a0] - pack->grid_lo[y_grid]) / x_step;
                if (!(xq > -1.0)) return fail(PAINTRL_E_INVALID, "texel left of its silhouette row (reference KeyError)");
                x_grid = std::min(g - 1, (int)xq);
            }
            int v_target = y_grid / v_interval;
            if (v_target >= g)
                return fail(PAINTRL_E_INVALID, "OBS_GRAD does not tile GRID_GRANULARITY (reference KeyError)");
            gcell[j] = (uint16_t)(v_target * g + x_grid);
            gtotal[v_target * g + x_grid]++;
        }
        pk.n_gcells = g * g;
        pk.n_gcells_pad = ((g * g + 3) / 4) * 4;
        CUDA_TRY(e->arena.upload(gtotal, &pk.gtotal));
        CUDA_TRY(e->arena.upload(gcell, &pk.gcell));
    }

    // ---- slot tables: exact FP64 positions, and FP32 origin-relative positions (ball pre-test)
    {
        std::vector<double> tx(pk.n_slots + 32, 1e30), ty(pk.n_slots + 32, 1e30), tz(pk.n_slots + 32, 1e30);   // padded: row_ranks reads 4 keys at a time
        std::vector<float> fx(pk.n_slots, 1e30f), fy(pk.n_slots, 1e30f), fz(pk.n_slots, 1e30f);
        pk.org0 = 0.5 * (tmin[0] + tmax[0]); pk.org1 = 0.5 * (tmin[1] + tmax[1]); pk.org2 = 0.5 * (tmin[2] + tmax[2]);
        float max_abs = 0.f;
        for (int j = 0; j < pk.n_slots; ++j) {
            if (slot_to_pack[j] < 0) continue;
            const double *p = pack->texel_pos + 3 * slot_to_pack[j];
            tx[j] = p[0]; ty[j] = p[1]; tz[j] = p[2];
            fx[j] = (float)(p[0] - pk.org0); fy[j] = (float)(p[1] - pk.org1); fz[j] = (float)(p[2] - pk.org2);
            max_abs = std::max(max_abs, std::max(std::fabs(fx[j]), std::max(std::fabs(fy[j]), std::fabs(fz[j]))));
        }
        // FP32 ball test error bound (see stamp()): |d2_f32 - d2_f64| < 4 ulp(2 max|coord|) * sqrt(3) * 2r
        const double bound = 4.0 * (double)ulp_f32(2.f * max_abs + (float)(2 * kPaintRadius)) * 1.7320508 * 2 * kPaintRadius + 4e-9;
        if (bound > (double)kBallEps) return fail(PAINTRL_E_INVALID, "part too large for the FP32 ball pre-test");
        CUDA_TRY(e->arena.upload(tx, &pk.tx));
        CUDA_TRY(e->arena.upload(ty, &pk.ty));
        CUDA_TRY(e->arena.upload(tz, &pk.tz));
        CUDA_TRY(e->arena.upload(fx, &pk.fx));
        CUDA_TRY(e->arena.upload(fy, &pk.fy));
        CUDA_TRY(e->arena.upload(fz, &pk.fz));
        // origin-relative FP32 copies of the row / cell grids (stamp_ranges)
        const double org_a0 = a0 == 0 ? pk.org0 : (a0 == 1 ? pk.org1 : pk.org2);
        const double org_a1 = a1 == 0 ? pk.org0 : (a1 == 1 ? pk.org1 : pk.org2);
        pk.rel_row_o1 = (float)(pk.row_o1 - org_a1);
        pk.rel_row_h = (float)pk.row_h;
        pk.rel_cx_o0 = (float)(pk.cx_o0 - org_a0);
        pk.rel_cx_inv = (float)pk.cx_inv;
    }

    // ---- silhouette table, ranges
    pk.grid_granularity = pack->grid_granularity;
    {
        std::vector<double> lo(pack->grid_lo, pack->grid_lo + pack->grid_granularity);
        std::vector<double> hi(pack->grid_hi, pack->grid_hi + pack->grid_granularity);
        CUDA_TRY(e->arena.upload(lo, &pk.grid_lo));
        CUDA_TRY(e->arena.upload(hi, &pk.grid_hi));
    }
    pk.range0_min = pack->range0_min; pk.range0_max = pack->range0_max;
    pk.range1_min = pack->range1_min; pk.range1_max = pack->range1_max;
    pk.lwr = pack->length_width_ratio;

    // ---- start points
    pk.n_starts = pack->n_starts;
    {
        std::vector<double> sp(pack->start_pos, pack->start_pos + 3 * (size_t)pack->n_starts);
        std::vector<double> sn(pack->start_normal, pack->start_normal + 3 * (size_t)pack->n_starts);
        CUDA_TRY(e->arena.upload(sp, &pk.start_pos));
        CUDA_TRY(e->arena.upload(sn, &pk.start_normal));
    }
    return PAINTRL_OK;
}

int obs_dim_of(const PaintrlConfig *cfg) {
    switch (cfg->obs_mode) {
        case PAINTRL_OBS_SECTION: return cfg->obs_grad + 2;
        case PAINTRL_OBS_GRID: return cfg->obs_grad * cfg->obs_grad;
        case PAINTRL_OBS_SIMPLE: return 2;
        default: return cfg->obs_grad + 1;
    }
}

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

EnvArrays env_arrays(PaintrlEngine *e) {
    EnvArrays ea;
    ea.states = e->states;
    ea.moves = e->moves;
    ea.env_stats = e->env_stats;
    ea.bits = e->bits;
    ea.thick = e->thick;
    ea.grid_cnt = e->grid_cnt;
    ea.ready = e->ready;
    ea.shots = e->shots;
    ea.last_mask = e->last_mask;
    return ea;
}

int launch_check(PaintrlEngine *e, const char *what) {
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string(what) + ": " + cudaGetErrorString(err));
    e->launches++;
    return PAINTRL_OK;
}

// launch_check for a step's second launch.  On failure the move grid is already in flight and will raise hand-off flags
// nobody consumes: clear them behind it, or the next step's paint warps would pass their acquire on stale move outputs.
int paint_check(PaintrlEngine *e, const char *what, cudaError_t err, cudaStream_t s) {
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err != cudaSuccess) {
        cudaGetLastError();
        cudaMemsetAsync(e->ready, 0, sizeof(unsigned) * (size_t)e->num_envs, s);
        return fail(PAINTRL_E_CUDA, std::string(what) + ": " + cudaGetErrorString(err));
    }
    e->launches++;
    return PAINTRL_OK;
}

// The I/O buffers of paintrl_step / paintrl_step_subset, checked and packed for the kernels.
int step_io(PaintrlHandle h, const void *actions_dev, double *obs_dev, double *reward_dev, double *penalty_dev, double *actual_dev,
            uint8_t *done_dev, int32_t *new_texels_dev, double *next_obs_dev, const int32_t *reset_start_idx_dev, StepIO *io) {
    if (!actions_dev || !obs_dev || !reward_dev || !penalty_dev || !actual_dev || !done_dev)
        return fail(PAINTRL_E_INVALID, "null I/O buffer");
    {   // the kernels store 8-byte (4-byte for new_texels / start indices) elements: refuse misaligned buffers
        const uintptr_t a8 = (uintptr_t)actions_dev | (uintptr_t)obs_dev | (uintptr_t)reward_dev | (uintptr_t)penalty_dev |
                             (uintptr_t)actual_dev | (uintptr_t)next_obs_dev;
        const uintptr_t a4 = (uintptr_t)new_texels_dev | (uintptr_t)reset_start_idx_dev;
        if ((a8 & 7u) || (a4 & 3u)) return fail(PAINTRL_E_INVALID, "misaligned I/O buffer (float64 / int64 buffers need 8-byte alignment)");
    }
    io->actions = actions_dev; io->obs = obs_dev; io->reward = reward_dev; io->penalty = penalty_dev;
    io->actual = actual_dev; io->done = done_dev; io->new_texels = new_texels_dev;
    io->next_obs = h->cfg.auto_reset ? next_obs_dev : nullptr;
    io->reset_start_idx = reset_start_idx_dev;
    return PAINTRL_OK;
}

// The environments of a subset step: the list env_ids (env_lo must be 0) or the range env_lo .. env_lo + n - 1.
int check_subset(PaintrlHandle h, const int32_t *env_ids, int32_t env_lo, int32_t n) {
    if (n < 1 || n > h->num_envs) return fail(PAINTRL_E_INVALID, "bad env count: n must be in [1, num_envs]");
    if (env_ids) {
        if (env_lo != 0) return fail(PAINTRL_E_INVALID, "env_lo must be 0 when an env_ids list is given");
        if ((uintptr_t)env_ids & 3u) return fail(PAINTRL_E_INVALID, "misaligned env_ids (int32 needs 4-byte alignment)");
    } else if (env_lo < 0 || (int64_t)env_lo + n > h->num_envs) {
        return fail(PAINTRL_E_INVALID, "env range [env_lo, env_lo + n) outside the batch");
    }
    return PAINTRL_OK;
}

// One step of the environments `sel` selects (SUBSET) or of the whole batch (!SUBSET, sel = {nullptr, 0, num_envs}),
// I/O row k = the k-th selected environment.  The kernel shape follows the paint method and the number of environments
// stepped: the beam-fan method, else the one-kernel step, else the two-kernel step.
template <bool SUBSET>
int launch_step(PaintrlHandle h, const EnvSel &sel, const StepIO &io, void *stream) {
    CUDA_TRY(cudaSetDevice(h->device));
    const int n = sel.n, threads = kWarpsPerBlock * 32;
    cudaStream_t s = as_stream(stream);
    const EnvArrays ea = env_arrays(h);
    const ColdArgs *cold = (const ColdArgs *)h->cold_args;
    if (h->paint_normal) {
        // Robot.PAINT_METHOD == 'normal': the generic move kernel (it also hands over the shots' poses), then the beam-fan
        // paint kernel, one warp per environment
        move_kernel<SUBSET><<<(n * 32 + threads - 1) / threads, threads, 0, s>>>(h->pk, h->cfg, ea, h->num_envs, io.actions, sel);
        int rc = launch_check(h, "move_kernel");
        if (rc != PAINTRL_OK) return rc;
        if (h->color == 0) paint_normal_kernel<0, SUBSET><<<n, 32, 0, s>>>(h->pk, h->cfg, ea, h->num_envs, io, cold, sel);
        else paint_normal_kernel<1, SUBSET><<<n, 32, 0, s>>>(h->pk, h->cfg, ea, h->num_envs, io, cold, sel);
        return paint_check(h, "paint_normal_kernel", cudaSuccess, s);
    }
    const bool staged = h->pk.n_words_pad <= kStageWords && !h->force_unstaged;
    const bool ax12 = h->pk.axis0 == 1 && h->pk.axis1 == 2, discrete = h->cfg.action_mode == 0;
    // K(args..., AX12, DISCRETE) with the part's axes and the action mode as compile-time constants
#define PAINTRL_AX_DI(K, ...)                                                                                       \
    do {                                                                                                            \
        if (ax12 && discrete) K(__VA_ARGS__, true, true);                                                           \
        else if (ax12) K(__VA_ARGS__, true, false);                                                                 \
        else if (discrete) K(__VA_ARGS__, false, true);                                                             \
        else K(__VA_ARGS__, false, false);                                                                          \
    } while (0)
    if (h->fused >= 0 ? h->fused == 1 : n < kFusedBelowEnvs) {
        // one launch, one warp per environment for the whole step (paintrl_kernels.cuh step_fused_kernel)
#define PAINTRL_STEP_FUSED(C, ST, AX, DI)                                                                           \
    step_fused_kernel<C, ST, AX, DI, SUBSET><<<(n + kFusedWarpsPerBlock - 1) / kFusedWarpsPerBlock,                \
                                               32 * kFusedWarpsPerBlock, 0, s>>>(h->pk, h->cfg, ea, h->num_envs, io, cold, sel)
        if (h->color == 0) { if (staged) PAINTRL_AX_DI(PAINTRL_STEP_FUSED, 0, true); else PAINTRL_AX_DI(PAINTRL_STEP_FUSED, 0, false); }
        else { if (staged) PAINTRL_AX_DI(PAINTRL_STEP_FUSED, 1, true); else PAINTRL_AX_DI(PAINTRL_STEP_FUSED, 1, false); }
#undef PAINTRL_STEP_FUSED
        return launch_check(h, "step_fused_kernel");
    }
    // The lean move kernel, h->move_lanes lanes per environment: rays decided by their move cell alone; the rest is
    // handed to the paint warps (kReadyBailed).
    const int mblocks = (int)(((long long)n * h->move_lanes + threads - 1) / threads);
#define PAINTRL_STEP_MOVE(G, AX, DI) move_fast_kernel<G, AX, DI, SUBSET><<<mblocks, threads, 0, s>>>(h->pk, h->cfg, ea, h->num_envs, io.actions, sel)
    if (h->move_lanes == 8) PAINTRL_AX_DI(PAINTRL_STEP_MOVE, 8); else PAINTRL_AX_DI(PAINTRL_STEP_MOVE, 32);
#undef PAINTRL_STEP_MOVE
#undef PAINTRL_AX_DI
    int rc = launch_check(h, "move_fast_kernel");
    if (rc != PAINTRL_OK) return rc;
    // the paint kernel, one warp per block, as a programmatic dependent launch after the move kernel (see
    // griddepcontrol.* in the kernels)
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(n); lc.blockDim = dim3(32); lc.dynamicSmemBytes = 0; lc.stream = s;
    cudaLaunchAttribute lattr[1];
    lattr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    lattr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = lattr; lc.numAttrs = 1;
    cudaError_t perr;
#define PAINTRL_STEP_PAINT(C, ST)                                                                                   \
    do {                                                                                                            \
        if (ax12) perr = cudaLaunchKernelEx(&lc, paint_kernel<C, ST, true, SUBSET>, h->pk, h->cfg, ea, h->num_envs, io, cold, sel);  \
        else perr = cudaLaunchKernelEx(&lc, paint_kernel<C, ST, false, SUBSET>, h->pk, h->cfg, ea, h->num_envs, io, cold, sel);      \
    } while (0)
    if (h->color == 0) { if (staged) PAINTRL_STEP_PAINT(0, true); else PAINTRL_STEP_PAINT(0, false); }
    else { if (staged) PAINTRL_STEP_PAINT(1, true); else PAINTRL_STEP_PAINT(1, false); }
#undef PAINTRL_STEP_PAINT
    return paint_check(h, "paint_kernel", perr, s);
}

// paintrl_step_host_submit (subset == false, the whole batch) and paintrl_step_host_submit_range (the environments
// env_lo .. env_lo + n - 1): host buffers of n rows, staged in the slot's device buffers in the same order.
int host_submit(PaintrlHandle h, int32_t slot, bool subset, int32_t env_lo, int32_t n, const void *actions_host, double *obs_host,
                double *reward_host, double *penalty_host, double *actual_host, uint8_t *done_host, double *next_obs_host,
                void *stream) {
    if (slot < 0 || slot > 1) return fail(PAINTRL_E_INVALID, "slot must be 0 or 1");
    if (!actions_host || !obs_host || !reward_host || !penalty_host || !actual_host || !done_host)
        return fail(PAINTRL_E_INVALID, "null I/O buffer");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t s = as_stream(stream);
    const size_t nenv = (size_t)n;
    const size_t abytes = (h->cfg.action_mode == 0 ? sizeof(long long) : sizeof(double) * h->cfg.action_shape) * nenv;
    const size_t obytes = sizeof(double) * h->cfg.obs_dim * nenv;
    const bool want_next = next_obs_host != nullptr, dev_next = want_next && h->cfg.auto_reset;
    // a slot that is submitted again before it was waited for: its previous copy-out must have drained first
    if (h->slot_pending[slot]) {
        CUDA_TRY(cudaStreamWaitEvent(h->copy_in, h->ev_done[slot], 0));
        CUDA_TRY(cudaStreamWaitEvent(s, h->ev_done[slot], 0));
    }
    // copy-in stream: the actions, then the step on the caller's stream behind it
    CUDA_TRY(cudaMemcpyAsync(h->slot_actions[slot], actions_host, abytes, cudaMemcpyHostToDevice, h->copy_in));
    CUDA_TRY(cudaEventRecord(h->ev_in[slot], h->copy_in));
    CUDA_TRY(cudaStreamWaitEvent(s, h->ev_in[slot], 0));
    unsigned char *d = h->slot_out[slot];
    double *d_obs = reinterpret_cast<double *>(d);
    double *d_sc = reinterpret_cast<double *>(d + obytes);
    double *d_next = dev_next ? reinterpret_cast<double *>(d + obytes + 3 * sizeof(double) * nenv) : nullptr;
    uint8_t *d_done = d + obytes + 3 * sizeof(double) * nenv + (dev_next ? obytes : 0);
    int rc = subset ? paintrl_step_subset(h, nullptr, env_lo, n, h->slot_actions[slot], d_obs, d_sc, d_sc + nenv, d_sc + 2 * nenv,
                                          d_done, nullptr, d_next, nullptr, stream)
                    : paintrl_step(h, h->slot_actions[slot], d_obs, d_sc, d_sc + nenv, d_sc + 2 * nenv, d_done, nullptr, d_next, nullptr, stream);
    if (rc != PAINTRL_OK) return rc;
    CUDA_TRY(cudaEventRecord(h->ev_step[slot], s));
    // copy-out stream: the results, as one copy when the host buffers are carved from one allocation in staging order
    CUDA_TRY(cudaStreamWaitEvent(h->copy_out, h->ev_step[slot], 0));
    struct Seg { void *dst; const void *src; size_t n; };
    Seg segs[7] = {};
    int ns = 0;
    auto push = [&](void *dst, const void *src, size_t n) {
        if (ns > 0 && (const char *)segs[ns - 1].src + segs[ns - 1].n == (const char *)src &&
            (char *)segs[ns - 1].dst + segs[ns - 1].n == (char *)dst) {
            segs[ns - 1].n += n;
        } else {
            segs[ns].dst = dst; segs[ns].src = src; segs[ns].n = n; ++ns;
        }
    };
    push(obs_host, d_obs, obytes);
    push(reward_host, d_sc, sizeof(double) * nenv);
    push(penalty_host, d_sc + nenv, sizeof(double) * nenv);
    push(actual_host, d_sc + 2 * nenv, sizeof(double) * nenv);
    if (dev_next) push(next_obs_host, d_next, obytes);
    push(done_host, d_done, nenv);
    if (want_next && !dev_next) push(next_obs_host, d_obs, obytes);
    for (int i = 0; i < ns; ++i) CUDA_TRY(cudaMemcpyAsync(segs[i].dst, segs[i].src, segs[i].n, cudaMemcpyDeviceToHost, h->copy_out));
    CUDA_TRY(cudaEventRecord(h->ev_done[slot], h->copy_out));
    h->slot_pending[slot] = true;
    return PAINTRL_OK;
}

}  // namespace

extern "C" {

int32_t paintrl_abi_version(void) { return PAINTRL_ABI_VERSION; }

/* ---- the grid-world ParamTestEnv (PaintRLEnv/param_test_env.py), see paintrl_param.cuh ---- */
struct PaintrlParamEngine {
    int device = 0;
    ParamWorld w{};
    DeviceArena arena;
    int *bad_action = nullptr;
    unsigned long long launches = 0;
};

int paintrl_param_create(const PaintrlParamConfig *cfg, int32_t num_envs, int32_t device, PaintrlParamHandle *out) {
    if (!cfg || !out) return fail(PAINTRL_E_INVALID, "null argument");
    if (cfg->abi_version != PAINTRL_ABI_VERSION) return fail(PAINTRL_E_INVALID, "ABI version mismatch");
    if (num_envs <= 0) return fail(PAINTRL_E_INVALID, "num_envs must be positive");
    if (cfg->size < 3 || cfg->size > 255) return fail(PAINTRL_E_INVALID, "size must be in 3..255");
    if (cfg->obs_mode < 0 || cfg->obs_mode > 3) return fail(PAINTRL_E_INVALID, "unknown observation mode");
    if (cfg->obs_mode == kParamObsGrid && cfg->size != 22)
        return fail(PAINTRL_E_INVALID, "the grid observation is defined for size 22 only (param_test_env.py:50-63 indexes a 10 x 10 table)");
    CUDA_TRY(cudaSetDevice(device));
    PaintrlParamEngine *e = new PaintrlParamEngine();
    e->device = device;
    ParamWorld &w = e->w;
    w.num_envs = num_envs;
    w.size = cfg->size;
    w.episode_max_length = std::max(cfg->max_len, (cfg->size - 2) * (cfg->size - 2));   /* param_test_env.py:112 */
    w.repeat_termination = cfg->termination_by_repeat ? 1 : 0;
    w.obs_mode = cfg->obs_mode;
    w.obs_dim = cfg->obs_mode == kParamObsSection ? 6 : cfg->obs_mode == kParamObsSimple ? 2
              : cfg->obs_mode == kParamObsDirect ? cfg->size * cfg->size + 2 : 102;
    w.auto_reset = cfg->auto_reset ? 1 : 0;
    w.init_reward_counter = (cfg->size - 2) * (cfg->size - 2);
    const size_t cells = (size_t)cfg->size * cfg->size * num_envs;
    bool ok = e->arena.alloc((void **)&w.world, cells) == cudaSuccess && e->arena.alloc((void **)&w.visit, cells * sizeof(uint16_t)) == cudaSuccess &&
              e->arena.alloc((void **)&w.pos_i, sizeof(int) * num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&w.pos_j, sizeof(int) * num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&w.reward_counter, sizeof(int) * num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&w.step_counter, sizeof(int) * num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&w.flags, num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&w.stats, 2 * sizeof(unsigned long long)) == cudaSuccess &&
              e->arena.alloc((void **)&e->bad_action, sizeof(int)) == cudaSuccess;
    if (!ok) { delete e; return fail(PAINTRL_E_CUDA, "device allocation failed (grid world)"); }
    cudaError_t err = cudaMemset(w.stats, 0, 2 * sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(e->bad_action, 0, sizeof(int));
    if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, cudaGetErrorString(err)); }
    param_reset_kernel<<<(num_envs + 127) / 128, 128>>>(w, nullptr, num_envs, nullptr);
    err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, cudaGetErrorString(err)); }
    *out = e;
    return PAINTRL_OK;
}

void paintrl_param_destroy(PaintrlParamHandle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    delete h;
}

int32_t paintrl_param_obs_dim(PaintrlParamHandle h) { return h ? h->w.obs_dim : 0; }

int paintrl_param_reset(PaintrlParamHandle h, const int32_t *env_ids_dev, int32_t n, double *obs_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (n <= 0 || n > h->w.num_envs || (!env_ids_dev && n != h->w.num_envs)) return fail(PAINTRL_E_INVALID, "bad env count");
    CUDA_TRY(cudaSetDevice(h->device));
    param_reset_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(h->w, env_ids_dev, n, obs_dev);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return PAINTRL_OK;
}

int paintrl_param_step(PaintrlParamHandle h, const int64_t *actions_dev, double *obs_dev, double *reward_dev, double *penalty_dev,
                       double *actual_dev, uint8_t *done_dev, double *next_obs_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!actions_dev || !obs_dev || !reward_dev || !penalty_dev || !actual_dev || !done_dev)
        return fail(PAINTRL_E_INVALID, "null I/O buffer");
    CUDA_TRY(cudaSetDevice(h->device));
    param_step_kernel<<<(h->w.num_envs + 127) / 128, 128, 0, as_stream(stream)>>>(
        h->w, reinterpret_cast<const long long *>(actions_dev), obs_dev, reward_dev, penalty_dev, actual_dev, done_dev, next_obs_dev,
        h->bad_action);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return PAINTRL_OK;
}

int paintrl_param_tables(PaintrlParamHandle h, const int32_t *env_ids_dev, int32_t n, int32_t *world_dev, int32_t *visit_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (n <= 0 || n > h->w.num_envs || (!env_ids_dev && n != h->w.num_envs)) return fail(PAINTRL_E_INVALID, "bad env count");
    CUDA_TRY(cudaSetDevice(h->device));
    const int cells = h->w.size * h->w.size;
    param_tables_kernel<<<dim3((cells + 127) / 128, n), 128, 0, as_stream(stream)>>>(h->w, env_ids_dev, n, world_dev, visit_dev);
    h->launches++;
    CUDA_TRY(cudaGetLastError());
    return PAINTRL_OK;
}

int paintrl_param_stats(PaintrlParamHandle h, uint64_t *env_steps, uint64_t *episodes_ended, uint64_t *kernel_launches,
                        int32_t *bad_action_seen) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    unsigned long long host[2];
    int bad = 0;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(host, h->w.stats, sizeof(host), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&bad, h->bad_action, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) CUDA_TRY(cudaMemset(h->bad_action, 0, sizeof(int)));      /* reported once, then cleared */
    if (env_steps) *env_steps = host[0];
    if (episodes_ended) *episodes_ended = host[1];
    if (kernel_launches) *kernel_launches = h->launches;
    if (bad_action_seen) *bad_action_seen = bad;
    return PAINTRL_OK;
}


/* Part.preprocess texel rasterisation on the GPU (see paintrl_raster.cuh and paintrl.h). */
int paintrl_rasterize_texels(const double *tri_a, const double *tri_b, const double *tri_c, const double *tri_uv,
                             int32_t n_tris, int32_t width, int32_t height, int32_t device, int32_t capacity,
                             int32_t *texel_ij_out, double *texel_pos_out, int32_t *n_texels_out) {
    if (!tri_a || !tri_b || !tri_c || !tri_uv || !n_texels_out) return fail(PAINTRL_E_INVALID, "null argument");
    if (n_tris <= 0 || width <= 0 || height <= 0 || (long long)width * height > (1ll << 29) || n_tris > (1 << 28))
        return fail(PAINTRL_E_INVALID, "bad triangle count or texture size");
    if (capacity > 0 && (!texel_ij_out || !texel_pos_out)) return fail(PAINTRL_E_INVALID, "null output buffer");
    CUDA_TRY(cudaSetDevice(device));
    const size_t n_pix = (size_t)width * height;
    DeviceArena arena;
    double *d_a = nullptr, *d_b = nullptr, *d_c = nullptr, *d_uv = nullptr;
    int *d_owner = nullptr, *d_bad = nullptr;
    if (arena.alloc((void **)&d_a, sizeof(double) * 3 * n_tris) != cudaSuccess || arena.alloc((void **)&d_b, sizeof(double) * 3 * n_tris) != cudaSuccess ||
        arena.alloc((void **)&d_c, sizeof(double) * 3 * n_tris) != cudaSuccess || arena.alloc((void **)&d_uv, sizeof(double) * 6 * n_tris) != cudaSuccess ||
        arena.alloc((void **)&d_owner, sizeof(int) * n_pix) != cudaSuccess || arena.alloc((void **)&d_bad, sizeof(int)) != cudaSuccess)
        return fail(PAINTRL_E_CUDA, "device allocation failed (rasteriser)");
    CUDA_TRY(cudaMemcpy(d_a, tri_a, sizeof(double) * 3 * n_tris, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_b, tri_b, sizeof(double) * 3 * n_tris, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_c, tri_c, sizeof(double) * 3 * n_tris, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_uv, tri_uv, sizeof(double) * 6 * n_tris, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemset(d_owner, 0xff, sizeof(int) * n_pix));
    CUDA_TRY(cudaMemset(d_bad, 0, sizeof(int)));
    raster_owner_kernel<<<(n_tris + 3) / 4, 128>>>(d_uv, n_tris, width, height, d_owner, d_bad);
    CUDA_TRY(cudaGetLastError());
    std::vector<int> owner(n_pix);
    int bad = 0;
    CUDA_TRY(cudaMemcpy(owner.data(), d_owner, sizeof(int) * n_pix, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) return fail(PAINTRL_E_INVALID, "a UV coordinate maps to a negative pixel coordinate");
    std::vector<int> pix;
    for (size_t k = 0; k < n_pix; ++k)
        if (owner[k] >= 0) pix.push_back((int)k);
    *n_texels_out = (int32_t)pix.size();
    if (capacity <= 0) return PAINTRL_OK;                 /* count only */
    if ((size_t)capacity < pix.size()) return fail(PAINTRL_E_INVALID, "output capacity is smaller than the texel count");
    if (pix.empty()) return PAINTRL_OK;
    int *d_pix = nullptr, *d_ij = nullptr;
    double *d_pos = nullptr;
    if (arena.alloc((void **)&d_pix, sizeof(int) * pix.size()) != cudaSuccess || arena.alloc((void **)&d_ij, sizeof(int) * 2 * pix.size()) != cudaSuccess ||
        arena.alloc((void **)&d_pos, sizeof(double) * 3 * pix.size()) != cudaSuccess)
        return fail(PAINTRL_E_CUDA, "device allocation failed (rasteriser output)");
    CUDA_TRY(cudaMemcpy(d_pix, pix.data(), sizeof(int) * pix.size(), cudaMemcpyHostToDevice));
    raster_position_kernel<<<(unsigned)((pix.size() + 255) / 256), 256>>>(d_a, d_b, d_c, d_uv, width, height, d_owner, d_pix,
                                                                          (int)pix.size(), d_ij, d_pos);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(texel_ij_out, d_ij, sizeof(int) * 2 * pix.size(), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(texel_pos_out, d_pos, sizeof(double) * 3 * pix.size(), cudaMemcpyDeviceToHost));
    return PAINTRL_OK;
}

/* Part._get_exact_boundary scans on the GPU (see paintrl_raster.cuh and paintrl.h). */
int paintrl_silhouette_march(const double *plane_n, const double *plane_off, int32_t n_planes, const double *points,
                             const int8_t *is_min, int32_t n_scans, int32_t proof_axis, int32_t non_principal_axis,
                             int32_t steps_range, int32_t device, double *boundary_out, int8_t *found_out) {
    if (!plane_n || !plane_off || !points || !is_min || !boundary_out || !found_out) return fail(PAINTRL_E_INVALID, "null argument");
    if (n_planes <= 0 || n_scans < 0 || steps_range < 0 || proof_axis < 0 || proof_axis > 2 || non_principal_axis < 0 ||
        non_principal_axis > 2 || proof_axis == non_principal_axis)
        return fail(PAINTRL_E_INVALID, "bad plane / scan count or axes");
    if (n_scans == 0) return PAINTRL_OK;
    CUDA_TRY(cudaSetDevice(device));
    std::vector<double4> planes((size_t)n_planes);
    for (int q = 0; q < n_planes; ++q) planes[q] = make_double4(plane_n[3 * q], plane_n[3 * q + 1], plane_n[3 * q + 2], plane_off[q]);
    DeviceArena arena;
    double4 *d_planes = nullptr;
    double *d_points = nullptr, *d_bound = nullptr;
    signed char *d_min = nullptr, *d_found = nullptr;
    if (arena.alloc((void **)&d_planes, sizeof(double4) * n_planes) != cudaSuccess || arena.alloc((void **)&d_points, sizeof(double) * 3 * n_scans) != cudaSuccess ||
        arena.alloc((void **)&d_bound, sizeof(double) * n_scans) != cudaSuccess || arena.alloc((void **)&d_min, n_scans) != cudaSuccess ||
        arena.alloc((void **)&d_found, n_scans) != cudaSuccess)
        return fail(PAINTRL_E_CUDA, "device allocation failed (silhouette scans)");
    CUDA_TRY(cudaMemcpy(d_planes, planes.data(), sizeof(double4) * n_planes, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_points, points, sizeof(double) * 3 * n_scans, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_min, is_min, n_scans, cudaMemcpyHostToDevice));
    silhouette_march_kernel<<<(n_scans + 3) / 4, 128>>>(d_planes, n_planes, d_points, d_min, n_scans, proof_axis, non_principal_axis,
                                                        steps_range, d_bound, d_found);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(boundary_out, d_bound, sizeof(double) * n_scans, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(found_out, d_found, n_scans, cudaMemcpyDeviceToHost));
    return PAINTRL_OK;
}

/* ---- the rollout policy (paint_ppo.py:179-183), see paintrl_policy.cuh ---- */
struct PaintrlPolicyEngine {
    int device = 0;
    int capacity = 0;
    PolicyParams pp{};
    DeviceArena arena;
    unsigned long long launches = 0;
};

int paintrl_policy_create(const PaintrlPolicyConfig *cfg, int32_t device, PaintrlPolicyHandle *out) {
    if (!cfg || !out) return fail(PAINTRL_E_INVALID, "null argument");
    if (cfg->abi_version != PAINTRL_ABI_VERSION) return fail(PAINTRL_E_INVALID, "ABI version mismatch");
    if (cfg->obs_dim <= 0 || cfg->obs_dim > kPolMaxObs) return fail(PAINTRL_E_INVALID, "the policy kernel takes observations of 1..32 entries");
    if (cfg->n_out <= 0 || cfg->n_out + 1 > kPolMaxOut) return fail(PAINTRL_E_INVALID, "the policy kernel takes 1..15 action outputs");
    if (cfg->capacity <= 0) return fail(PAINTRL_E_INVALID, "capacity must be positive");
    if (!cfg->w1 || !cfg->b1 || !cfg->w2 || !cfg->b2 || !cfg->w3 || !cfg->b3) return fail(PAINTRL_E_INVALID, "null weight pointer");
    int rc = select_device(device);
    if (rc != PAINTRL_OK) return rc;
    PaintrlPolicyEngine *e = new PaintrlPolicyEngine();
    e->device = device;
    e->capacity = cfg->capacity;
    PolicyParams &pp = e->pp;
    pp.obs_dim = cfg->obs_dim; pp.n_out = cfg->n_out; pp.discrete = cfg->discrete ? 1 : 0; pp.seed = cfg->seed;
    const int nout1 = cfg->n_out + 1;
    std::vector<float> w1(cfg->w1, cfg->w1 + (size_t)cfg->obs_dim * kPolH1), b1(cfg->b1, cfg->b1 + kPolH1), b2(cfg->b2, cfg->b2 + kPolH2),
        w3(cfg->w3, cfg->w3 + (size_t)kPolH2 * nout1), b3(cfg->b3, cfg->b3 + nout1);
    // W2 [256 in][128 out] FP32 -> BF16 B operand [n = out][k = in] in the tensor core's canonical K-major layout
    std::vector<__nv_bfloat16> w2p((size_t)kPolH1 * kPolH2);
    for (int n = 0; n < kPolH2; ++n)
        for (int k = 0; k < kPolH1; ++k) w2p[pol_w2_byte(k, n) / 2] = __float2bfloat16_rn(cfg->w2[(size_t)k * kPolH2 + n]);
    bool ok = e->arena.upload(w1, &pp.w1) == cudaSuccess && e->arena.upload(b1, &pp.b1) == cudaSuccess &&
              e->arena.upload(w2p, &pp.w2_packed) == cudaSuccess && e->arena.upload(b2, &pp.b2) == cudaSuccess &&
              e->arena.upload(w3, &pp.w3) == cudaSuccess && e->arena.upload(b3, &pp.b3) == cudaSuccess &&
              e->arena.alloc((void **)&pp.counters, sizeof(unsigned) * (size_t)cfg->capacity) == cudaSuccess;
    if (ok) ok = cudaMemset(pp.counters, 0, sizeof(unsigned) * (size_t)cfg->capacity) == cudaSuccess;
    with_caps(pp.obs_dim, pp.n_out, [&](auto mo, auto mx) {
        ok = ok && opt_in_smem(policy_act_kernel<mo, mx, false>, kPolSmemBytes) && opt_in_smem(policy_act_kernel<mo, mx, true>, kPolSmemBytes) &&
             (pp.discrete || opt_in_smem(policy_act_kernel<mo, mx, false, true>, kPolSmemBytes));
    });
    if (!ok) { delete e; cudaGetLastError(); return fail(PAINTRL_E_CUDA, "setting up the policy engine failed (allocation / shared memory opt-in)"); }
    *out = e;
    return PAINTRL_OK;
}

void paintrl_policy_destroy(PaintrlPolicyHandle h) { destroy_engine(h); }

// how policy_act_kernel picks actions: the engine's own head, epsilon-greedy (EPS) or the diagonal Gaussian (DIAG)
enum PolicyMode { kActSample, kActEpsilon, kActDiag };

static int policy_launch(PaintrlPolicyHandle h, const PolicyIO &io, PolicyMode mode, void *stream) {
    const dim3 pgrid((io.batch + kPolRows - 1) / kPolRows);
    cudaStream_t s = as_stream(stream);
    with_caps(h->pp.obs_dim, h->pp.n_out, [&](auto mo, auto mx) {
        if (mode == kActEpsilon) policy_act_kernel<mo, mx, true><<<pgrid, kPolThreads, kPolSmemBytes, s>>>(h->pp, io);
        else if (mode == kActDiag) policy_act_kernel<mo, mx, false, true><<<pgrid, kPolThreads, kPolSmemBytes, s>>>(h->pp, io);
        else policy_act_kernel<mo, mx, false><<<pgrid, kPolThreads, kPolSmemBytes, s>>>(h->pp, io);
    });
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("policy_act_kernel: ") + cudaGetErrorString(err));
    h->launches++;
    return PAINTRL_OK;
}

int paintrl_policy_act(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, void *actions_dev, float *logp_dev, float *value_dev,
                       float *logits_dev, int32_t sample, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!obs_dev || !value_dev || (sample && (!actions_dev || !logp_dev))) return fail(PAINTRL_E_INVALID, "null I/O buffer");
    if (batch <= 0 || batch > h->capacity) return fail(PAINTRL_E_INVALID, "batch exceeds the policy engine's capacity");
    CUDA_TRY(cudaSetDevice(h->device));
    PolicyIO io;
    io.obs = obs_dev; io.batch = batch;
    io.act_discrete = h->pp.discrete ? reinterpret_cast<long long *>(actions_dev) : nullptr;
    io.act_continuous = h->pp.discrete ? nullptr : reinterpret_cast<double *>(actions_dev);
    io.logp = logp_dev; io.value = value_dev; io.logits = logits_dev; io.sample = sample ? 1 : 0;
    return policy_launch(h, io, kActSample, stream);
}

int paintrl_policy_act_epsilon(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, void *actions_dev, float *value_dev,
                               float *logits_dev, const float *epsilon_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!h->pp.discrete) return fail(PAINTRL_E_INVALID, "epsilon-greedy actions need a discrete policy engine");
    if (!obs_dev || !actions_dev || !value_dev || !epsilon_dev) return fail(PAINTRL_E_INVALID, "null I/O buffer");
    if (batch <= 0 || batch > h->capacity) return fail(PAINTRL_E_INVALID, "batch exceeds the policy engine's capacity");
    CUDA_TRY(cudaSetDevice(h->device));
    PolicyIO io{};
    io.obs = obs_dev; io.batch = batch;
    io.act_discrete = reinterpret_cast<long long *>(actions_dev);
    io.value = value_dev; io.logits = logits_dev; io.sample = 1; io.epsilon = epsilon_dev;
    return policy_launch(h, io, kActEpsilon, stream);
}

int paintrl_policy_act_diag_gaussian(PaintrlPolicyHandle h, const double *obs_dev, int32_t batch, double *actions_dev, float *logp_dev,
                                     float *value_dev, float *logits_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (h->pp.discrete) return fail(PAINTRL_E_INVALID, "diagonal-Gaussian actions need a continuous policy engine");
    if (h->pp.n_out % 2) return fail(PAINTRL_E_INVALID, "diagonal-Gaussian actions need an even n_out (a mean and a log-std per action dimension)");
    if (!obs_dev || !actions_dev || !logp_dev || !value_dev) return fail(PAINTRL_E_INVALID, "null I/O buffer");
    if (batch <= 0 || batch > h->capacity) return fail(PAINTRL_E_INVALID, "batch exceeds the policy engine's capacity");
    CUDA_TRY(cudaSetDevice(h->device));
    PolicyIO io{};
    io.obs = obs_dev; io.batch = batch;
    io.act_continuous = actions_dev;
    io.logp = logp_dev; io.value = value_dev; io.logits = logits_dev; io.sample = 1;
    return policy_launch(h, io, kActDiag, stream);
}

/* ---- the PPO learner, see paintrl_learn.cuh ---- */
int32_t paintrl_policy_num_params(int32_t obs_dim, int32_t n_out) {
    if (obs_dim <= 0 || obs_dim > kPolMaxObs || n_out <= 0 || n_out + 1 > kPolMaxOut) return fail(PAINTRL_E_INVALID, "the policy kernel takes observations of 1..32 entries and 1..15 action outputs");
    return pol_num_params(obs_dim, n_out);
}

int paintrl_policy_set_params(PaintrlPolicyHandle h, const float *params_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!params_dev) return fail(PAINTRL_E_INVALID, "null parameter buffer");
    CUDA_TRY(cudaSetDevice(h->device));
    const PolicyParams &pp = h->pp;
    const int n = pol_num_params(pp.obs_dim, pp.n_out);
    policy_pack_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(params_dev, pp.obs_dim, pp.n_out, const_cast<float *>(pp.w1),
                                                                        const_cast<float *>(pp.b1), const_cast<__nv_bfloat16 *>(pp.w2_packed),
                                                                        const_cast<float *>(pp.b2), const_cast<float *>(pp.w3), const_cast<float *>(pp.b3));
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("policy_pack_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

// What the PPO and the DQN learner handles share: the network shape, the per-CTA partial gradients and statistics that
// ppo_reduce_kernel sums, and the arena that owns them.
struct LearnerEngine {
    int device = 0;
    int obs_dim = 0, n_out = 0, max_minibatch = 0;
    int nparams = 0, max_ctas = 0;
    float *partial = nullptr, *partial_stats = nullptr;
    DeviceArena arena;
};

struct PaintrlPpoEngine : LearnerEngine {
    PaintrlPpoConfig cfg{};
};

static int learner_check(int abi_version, int obs_dim, int n_out, int max_minibatch) {
    if (abi_version != PAINTRL_ABI_VERSION) return fail(PAINTRL_E_INVALID, "ABI version mismatch");
    if (obs_dim <= 0 || obs_dim > kPolMaxObs) return fail(PAINTRL_E_INVALID, "the learner kernel takes observations of 1..32 entries");
    if (n_out <= 0 || n_out + 1 > kPolMaxOut) return fail(PAINTRL_E_INVALID, "the learner kernel takes 1..15 action outputs");
    if (max_minibatch <= 0) return fail(PAINTRL_E_INVALID, "max_minibatch must be positive");
    return PAINTRL_OK;
}

// Device, shape, the partial buffers and the shared-memory opt-in of every loss stage for this shape.  The caller
// deletes e when this fails.
static int learner_init(LearnerEngine *e, int device, int obs_dim, int n_out, int max_minibatch) {
    int rc = select_device(device);
    if (rc != PAINTRL_OK) return rc;
    e->device = device;
    e->obs_dim = obs_dim; e->n_out = n_out; e->max_minibatch = max_minibatch;
    e->nparams = pol_num_params(obs_dim, n_out);
    e->max_ctas = (max_minibatch + kPolRows - 1) / kPolRows;
    bool ok = e->arena.alloc((void **)&e->partial, sizeof(float) * (size_t)e->max_ctas * e->nparams) == cudaSuccess &&
              e->arena.alloc((void **)&e->partial_stats, sizeof(float) * (size_t)e->max_ctas * kLrnStatStride) == cudaSuccess;
    with_caps(obs_dim, n_out, [&](auto mo, auto mx) {
        ok = ok && opt_in_smem(ppo_grad_kernel<mo, mx, kLossPpo>, kLrnSmemBytes) && opt_in_smem(ppo_grad_kernel<mo, mx, kLossDqn>, kLrnSmemBytes) &&
             opt_in_smem(ppo_grad_kernel<mo, mx, kLossDqnPer>, kLrnSmemBytes) && opt_in_smem(ppo_grad_kernel<mo, mx, kLossPpoDiag>, kLrnSmemBytes);
    });
    if (!ok) { cudaGetLastError(); return fail(PAINTRL_E_CUDA, "setting up the learner failed (allocation / shared memory opt-in)"); }
    return PAINTRL_OK;
}

// the launch arguments every learner call fills the same way
static PpoGradArgs learner_args(const LearnerEngine *h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev) {
    PpoGradArgs a{};
    a.obs_dim = h->obs_dim; a.n_out = h->n_out; a.n = n; a.nparams = h->nparams;
    a.params = params_dev; a.idx = idx_dev; a.obs = obs_dev;
    a.partial = h->partial; a.partial_stats = h->partial_stats;
    return a;
}

static int learner_launch(const PpoGradArgs &a, void *stream, int loss = kLossPpo) {
    const dim3 grid((a.n + kPolRows - 1) / kPolRows);
    cudaStream_t s = as_stream(stream);
    with_caps(a.obs_dim, a.n_out, [&](auto mo, auto mx) {
        if (loss == kLossDqn) ppo_grad_kernel<mo, mx, kLossDqn><<<grid, kPolThreads, kLrnSmemBytes, s>>>(a);
        else if (loss == kLossPpoDiag) ppo_grad_kernel<mo, mx, kLossPpoDiag><<<grid, kPolThreads, kLrnSmemBytes, s>>>(a);
        else if (loss == kLossDqnPer) ppo_grad_kernel<mo, mx, kLossDqnPer><<<grid, kPolThreads, kLrnSmemBytes, s>>>(a);
        else ppo_grad_kernel<mo, mx, kLossPpo><<<grid, kPolThreads, kLrnSmemBytes, s>>>(a);
    });
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("ppo_grad_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

// grad = the CTA-order sum of the partial gradients of a launch over n samples; stats = the means of its first nstats
static int learner_reduce(const LearnerEngine *h, int32_t n, float inv_n, float *grad_dev, float *stats_dev, int nstats, void *stream) {
    const int nparts = (n + kPolRows - 1) / kPolRows;
    ppo_reduce_kernel<<<(h->nparams + 255) / 256, 256, 0, as_stream(stream)>>>(h->partial, nparts, h->nparams, grad_dev, h->partial_stats,
                                                                                inv_n, stats_dev, nstats);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("ppo_reduce_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

int paintrl_ppo_create(const PaintrlPpoConfig *cfg, int32_t device, PaintrlPpoHandle *out) {
    if (!cfg || !out) return fail(PAINTRL_E_INVALID, "null argument");
    int rc = learner_check(cfg->abi_version, cfg->obs_dim, cfg->n_out, cfg->max_minibatch);
    if (rc != PAINTRL_OK) return rc;
    if (!(cfg->clip_param > 0.f) || !(cfg->vf_clip_param > 0.f) || !(cfg->vf_loss_coeff >= 0.f) || !(cfg->entropy_coeff >= 0.f))
        return fail(PAINTRL_E_INVALID, "clip_param and vf_clip_param must be positive, vf_loss_coeff and entropy_coeff non-negative");
    PaintrlPpoEngine *e = new PaintrlPpoEngine();
    e->cfg = *cfg;
    rc = learner_init(e, device, cfg->obs_dim, cfg->n_out, cfg->max_minibatch);
    if (rc != PAINTRL_OK) { delete e; return rc; }
    *out = e;
    return PAINTRL_OK;
}

void paintrl_ppo_destroy(PaintrlPpoHandle h) { destroy_engine(h); }

// paintrl_ppo_grad (loss kLossPpo) and paintrl_ppo_grad_diag_gaussian (kLossPpoDiag), after their handle checks
static int ppo_grad(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                    const void *actions_dev, const float *logp_old_dev, const float *value_old_dev, const float *logits_old_dev,
                    const float *adv_dev, const float *vtarg_dev, float kl_coeff, float *grad_dev, float *stats_dev, void *stream, int loss) {
    if (!params_dev || !idx_dev || !obs_dev || !actions_dev || !logp_old_dev || !value_old_dev || !logits_old_dev || !adv_dev ||
        !vtarg_dev || !grad_dev || !stats_dev)
        return fail(PAINTRL_E_INVALID, "null buffer");
    if (n <= 0 || n > h->max_minibatch) return fail(PAINTRL_E_INVALID, "n must be in [1, max_minibatch]");
    if (!(kl_coeff >= 0.f)) return fail(PAINTRL_E_INVALID, "kl_coeff must be non-negative");
    CUDA_TRY(cudaSetDevice(h->device));
    PpoGradArgs a = learner_args(h, params_dev, idx_dev, n, obs_dev);
    a.discrete = h->cfg.discrete ? 1 : 0;
    a.actions = actions_dev; a.logp_old = logp_old_dev; a.value_old = value_old_dev; a.logits_old = logits_old_dev;
    a.adv = adv_dev; a.vtarg = vtarg_dev;
    a.clip = h->cfg.clip_param; a.vf_clip = h->cfg.vf_clip_param; a.vf_coeff = h->cfg.vf_loss_coeff; a.ent_coeff = h->cfg.entropy_coeff;
    a.kl_coeff = kl_coeff; a.inv_n = 1.f / (float)n;
    int rc = learner_launch(a, stream, loss);
    if (rc != PAINTRL_OK) return rc;
    return learner_reduce(h, n, a.inv_n, grad_dev, stats_dev, kLrnStats, stream);
}

int paintrl_ppo_grad(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                     const void *actions_dev, const float *logp_old_dev, const float *value_old_dev, const float *logits_old_dev,
                     const float *adv_dev, const float *vtarg_dev, float kl_coeff, float *grad_dev, float *stats_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    return ppo_grad(h, params_dev, idx_dev, n, obs_dev, actions_dev, logp_old_dev, value_old_dev, logits_old_dev, adv_dev, vtarg_dev,
                    kl_coeff, grad_dev, stats_dev, stream, kLossPpo);
}

int paintrl_ppo_grad_diag_gaussian(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                                   const void *actions_dev, const float *logp_old_dev, const float *value_old_dev,
                                   const float *logits_old_dev, const float *adv_dev, const float *vtarg_dev, float kl_coeff,
                                   float *grad_dev, float *stats_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (h->cfg.discrete) return fail(PAINTRL_E_INVALID, "the diagonal-Gaussian loss needs a continuous learner handle");
    if (h->n_out % 2) return fail(PAINTRL_E_INVALID, "the diagonal-Gaussian loss needs an even n_out (a mean and a log-std per action dimension)");
    return ppo_grad(h, params_dev, idx_dev, n, obs_dev, actions_dev, logp_old_dev, value_old_dev, logits_old_dev, adv_dev, vtarg_dev,
                    kl_coeff, grad_dev, stats_dev, stream, kLossPpoDiag);
}

int paintrl_ppo_forward(PaintrlPpoHandle h, const float *params_dev, const int32_t *idx_dev, int32_t n, const double *obs_dev,
                        float *out_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!params_dev || !idx_dev || !obs_dev || !out_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (n <= 0 || n > h->max_minibatch) return fail(PAINTRL_E_INVALID, "n must be in [1, max_minibatch]");
    CUDA_TRY(cudaSetDevice(h->device));
    PpoGradArgs a = learner_args(h, params_dev, idx_dev, n, obs_dev);
    a.discrete = h->cfg.discrete ? 1 : 0;
    a.forward_only = 1;
    a.fwd_out = out_dev;
    return learner_launch(a, stream);
}

int paintrl_adam_step(float *params_dev, const float *grad_dev, float *m_dev, float *v_dev, int32_t n_params, float lr, float beta1,
                      float beta2, float eps, int32_t step, void *stream) {
    if (!params_dev || !grad_dev || !m_dev || !v_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (n_params <= 0) return fail(PAINTRL_E_INVALID, "n_params must be positive");
    if (step < 1) return fail(PAINTRL_E_INVALID, "step counts from 1");
    if (!(lr >= 0.f) || !(beta1 >= 0.f && beta1 < 1.f) || !(beta2 >= 0.f && beta2 < 1.f) || !(eps > 0.f))
        return fail(PAINTRL_E_INVALID, "lr >= 0, beta1 / beta2 in [0, 1) and eps > 0 are required");
    const double bc1 = 1.0 - std::pow((double)beta1, (double)step), bc2 = 1.0 - std::pow((double)beta2, (double)step);
    adam_kernel<<<(n_params + 255) / 256, 256, 0, as_stream(stream)>>>(params_dev, grad_dev, m_dev, v_dev, n_params, (float)(lr / bc1), beta1,
                                                                        beta2, eps, (float)std::sqrt(bc2));
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("adam_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

/* ---- double DQN on the learner kernel's loss template, see paintrl_learn.cuh ---- */
struct PaintrlDqnEngine : LearnerEngine {
    PaintrlDqnConfig cfg{};
    float *next_online = nullptr, *next_target = nullptr;   // [max_minibatch][n_out + 1]: the head on s'
};

int paintrl_dqn_create(const PaintrlDqnConfig *cfg, int32_t device, PaintrlDqnHandle *out) {
    if (!cfg || !out) return fail(PAINTRL_E_INVALID, "null argument");
    int rc = learner_check(cfg->abi_version, cfg->obs_dim, cfg->n_out, cfg->max_minibatch);
    if (rc != PAINTRL_OK) return rc;
    if (!(cfg->gamma > 0.f && cfg->gamma <= 1.f)) return fail(PAINTRL_E_INVALID, "gamma must be in (0, 1]");
    PaintrlDqnEngine *e = new PaintrlDqnEngine();
    e->cfg = *cfg;
    rc = learner_init(e, device, cfg->obs_dim, cfg->n_out, cfg->max_minibatch);
    const size_t heads = sizeof(float) * (size_t)cfg->max_minibatch * (cfg->n_out + 1);
    if (rc == PAINTRL_OK &&
        (e->arena.alloc((void **)&e->next_online, heads) != cudaSuccess || e->arena.alloc((void **)&e->next_target, heads) != cudaSuccess)) {
        cudaGetLastError();
        rc = fail(PAINTRL_E_CUDA, "setting up the DQN learner failed (allocation)");
    }
    if (rc != PAINTRL_OK) { delete e; return rc; }
    *out = e;
    return PAINTRL_OK;
}

void paintrl_dqn_destroy(PaintrlDqnHandle h) { destroy_engine(h); }

// paintrl_dqn_grad and paintrl_dqn_grad_weighted: weight_dev / td_out_dev are null for the unweighted loss
static int dqn_grad(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev, int32_t n,
                    const double *obs_dev, const int64_t *actions_dev, const float *reward_dev, const double *next_obs_dev,
                    const uint8_t *done_dev, const float *weight_dev, float *td_out_dev, float *grad_dev, float *stats_dev, void *stream) {
    CUDA_TRY(cudaSetDevice(h->device));
    // the head on s' under the online, then the target parameters: the forward-only path of the same kernel
    PpoGradArgs a = learner_args(h, params_dev, idx_dev, n, next_obs_dev);
    a.discrete = 1;
    a.forward_only = 1; a.fwd_out = h->next_online;
    int rc = learner_launch(a, stream);
    if (rc != PAINTRL_OK) return rc;
    a.params = target_params_dev; a.fwd_out = h->next_target;
    rc = learner_launch(a, stream);
    if (rc != PAINTRL_OK) return rc;
    a.forward_only = 0; a.obs = obs_dev; a.params = params_dev; a.fwd_out = nullptr;
    a.actions = actions_dev; a.reward = reward_dev; a.done = done_dev; a.next_online = h->next_online; a.next_target = h->next_target;
    a.gamma = h->cfg.gamma; a.inv_n = 1.f / (float)n;
    a.weight = weight_dev; a.td_out = td_out_dev;
    const bool weighted = weight_dev != nullptr;
    rc = learner_launch(a, stream, weighted ? kLossDqnPer : kLossDqn);
    if (rc != PAINTRL_OK) return rc;
    return learner_reduce(h, n, a.inv_n, grad_dev, stats_dev, weighted ? kDqnPerStats : kDqnStats, stream);
}

static int dqn_grad_check(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev, int32_t n,
                          const double *obs_dev, const int64_t *actions_dev, const float *reward_dev, const double *next_obs_dev,
                          const uint8_t *done_dev, float *grad_dev, float *stats_dev) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!params_dev || !target_params_dev || !idx_dev || !obs_dev || !actions_dev || !reward_dev || !next_obs_dev || !done_dev ||
        !grad_dev || !stats_dev)
        return fail(PAINTRL_E_INVALID, "null buffer");
    if (n <= 0 || n > h->max_minibatch) return fail(PAINTRL_E_INVALID, "n must be in [1, max_minibatch]");
    return PAINTRL_OK;
}

int paintrl_dqn_grad(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev, int32_t n,
                     const double *obs_dev, const int64_t *actions_dev, const float *reward_dev, const double *next_obs_dev,
                     const uint8_t *done_dev, float *grad_dev, float *stats_dev, void *stream) {
    const int rc = dqn_grad_check(h, params_dev, target_params_dev, idx_dev, n, obs_dev, actions_dev, reward_dev, next_obs_dev, done_dev,
                                  grad_dev, stats_dev);
    if (rc != PAINTRL_OK) return rc;
    return dqn_grad(h, params_dev, target_params_dev, idx_dev, n, obs_dev, actions_dev, reward_dev, next_obs_dev, done_dev, nullptr,
                    nullptr, grad_dev, stats_dev, stream);
}

int paintrl_dqn_grad_weighted(PaintrlDqnHandle h, const float *params_dev, const float *target_params_dev, const int32_t *idx_dev,
                              int32_t n, const double *obs_dev, const int64_t *actions_dev, const float *reward_dev,
                              const double *next_obs_dev, const uint8_t *done_dev, const float *weight_dev, float *td_out_dev,
                              float *grad_dev, float *stats_dev, void *stream) {
    const int rc = dqn_grad_check(h, params_dev, target_params_dev, idx_dev, n, obs_dev, actions_dev, reward_dev, next_obs_dev, done_dev,
                                  grad_dev, stats_dev);
    if (rc != PAINTRL_OK) return rc;
    if (!weight_dev || !td_out_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    return dqn_grad(h, params_dev, target_params_dev, idx_dev, n, obs_dev, actions_dev, reward_dev, next_obs_dev, done_dev, weight_dev,
                    td_out_dev, grad_dev, stats_dev, stream);
}

/* ---- prioritized replay: the sum / min trees of paintrl_replay.cuh ---- */
static int prio_check_tree(const double *sum_tree_dev, const double *min_tree_dev, int32_t tree_leaves, int32_t capacity) {
    if (!sum_tree_dev || !min_tree_dev) return fail(PAINTRL_E_INVALID, "null tree buffer");
    if (capacity < 1) return fail(PAINTRL_E_INVALID, "capacity must be positive");
    if (tree_leaves < capacity || (tree_leaves & (tree_leaves - 1)) != 0)
        return fail(PAINTRL_E_INVALID, "tree_leaves must be a power of two at or above the capacity");
    return PAINTRL_OK;
}

// every internal node from its two children: one launch per group of up to log2(kPrioSubtree) levels, bottom up
static int prio_rebuild(double *sum, double *mn, int L, cudaStream_t s) {
    for (int base = L; base > 1;) {
        const int width = std::min(base, kPrioSubtree);
        prio_build_kernel<<<base / width, kPrioBuildThreads, 0, s>>>(sum, mn, base, width);
        base /= width;
    }
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("prio_build_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

int paintrl_prio_fill(double *sum_tree_dev, double *min_tree_dev, int32_t tree_leaves, int32_t capacity, int32_t start, int32_t count,
                      const double *max_priority_dev, double alpha, void *stream) {
    int rc = prio_check_tree(sum_tree_dev, min_tree_dev, tree_leaves, capacity);
    if (rc != PAINTRL_OK) return rc;
    if (!max_priority_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (start < 0 || start >= capacity) return fail(PAINTRL_E_INVALID, "start must be in [0, capacity)");
    if (count < 1 || count > capacity) return fail(PAINTRL_E_INVALID, "count must be in [1, capacity]");
    if (!(alpha >= 0.0 && std::isfinite(alpha))) return fail(PAINTRL_E_INVALID, "alpha must be finite and non-negative");
    cudaStream_t s = as_stream(stream);
    prio_fill_kernel<<<(count + kPrioThreads - 1) / kPrioThreads, kPrioThreads, 0, s>>>(sum_tree_dev, min_tree_dev, tree_leaves, capacity,
                                                                                          start, count, max_priority_dev, alpha);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("prio_fill_kernel: ") + cudaGetErrorString(err));
    return prio_rebuild(sum_tree_dev, min_tree_dev, tree_leaves, s);
}

int paintrl_prio_update(double *sum_tree_dev, double *min_tree_dev, int32_t tree_leaves, int32_t capacity, const int32_t *idx_dev,
                        const float *td_dev, int32_t n, double *max_priority_dev, double alpha, double eps, void *stream) {
    int rc = prio_check_tree(sum_tree_dev, min_tree_dev, tree_leaves, capacity);
    if (rc != PAINTRL_OK) return rc;
    if (!idx_dev || !td_dev || !max_priority_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (n < 1 || n > kPrioMaxBatch) return fail(PAINTRL_E_INVALID, "n must be in [1, 2^24]");
    if (!(alpha >= 0.0 && std::isfinite(alpha))) return fail(PAINTRL_E_INVALID, "alpha must be finite and non-negative");
    if (!(eps > 0.0 && std::isfinite(eps))) return fail(PAINTRL_E_INVALID, "eps must be finite and positive");
    cudaStream_t s = as_stream(stream);
    prio_update_kernel<<<(n + kPrioThreads - 1) / kPrioThreads, kPrioThreads, 0, s>>>(sum_tree_dev, min_tree_dev, tree_leaves, idx_dev,
                                                                                        td_dev, n, max_priority_dev, alpha, eps);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("prio_update_kernel: ") + cudaGetErrorString(err));
    return prio_rebuild(sum_tree_dev, min_tree_dev, tree_leaves, s);
}

int paintrl_prio_sample(const double *sum_tree_dev, const double *min_tree_dev, int32_t tree_leaves, int32_t capacity, int32_t size,
                        const double *u_dev, int32_t n, double beta, int32_t *idx_out_dev, float *weight_out_dev, void *stream) {
    int rc = prio_check_tree(sum_tree_dev, min_tree_dev, tree_leaves, capacity);
    if (rc != PAINTRL_OK) return rc;
    if (!u_dev || !idx_out_dev || !weight_out_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (size < 1 || size > capacity) return fail(PAINTRL_E_INVALID, "size must be in [1, capacity]");
    if (n < 1 || n > kPrioMaxBatch) return fail(PAINTRL_E_INVALID, "n must be in [1, 2^24]");
    if (!(beta >= 0.0 && beta <= 1.0)) return fail(PAINTRL_E_INVALID, "beta must be in [0, 1]");
    prio_sample_kernel<<<(n + kPrioThreads - 1) / kPrioThreads, kPrioThreads, 0, as_stream(stream)>>>(
        sum_tree_dev, min_tree_dev, tree_leaves, u_dev, n, beta, idx_out_dev, weight_out_dev);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("prio_sample_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

int paintrl_clip_grad_norm(float *grad_dev, int32_t n, float max_norm, float *norm_out_dev, void *stream) {
    if (!grad_dev || !norm_out_dev) return fail(PAINTRL_E_INVALID, "null buffer");
    if (n <= 0) return fail(PAINTRL_E_INVALID, "n must be positive");
    if (!(max_norm > 0.f)) return fail(PAINTRL_E_INVALID, "max_norm must be positive");
    clip_grad_norm_kernel<<<1, kClipThreads, 0, as_stream(stream)>>>(grad_dev, n, max_norm, norm_out_dev);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(PAINTRL_E_CUDA, std::string("clip_grad_norm_kernel: ") + cudaGetErrorString(err));
    return PAINTRL_OK;
}

const char *paintrl_last_error(void) { return g_error.c_str(); }

/* Debug only (not in paintrl.h): phase cycle counters of a -DPAINTRL_PROFILE build; returns 0 slots otherwise. */
int paintrl_debug_profile(unsigned long long *out64, int reset) {
#ifdef PAINTRL_PROFILE
    cudaDeviceSynchronize();
    if (out64) cudaMemcpyFromSymbol(out64, g_prof, 64 * sizeof(unsigned long long));
    if (reset) {
        unsigned long long z[64] = {0};
        cudaMemcpyToSymbol(g_prof, z, sizeof(z));
    }
    return 64;
#else
    (void)out64; (void)reset;
    return 0;
#endif
}

/* Debug only: the last step's phase cycles per environment ([n][32] u32, slot 14 = the move counters). */
int paintrl_debug_fast_reasons(unsigned long long *out8) {
#ifdef PAINTRL_PROFILE
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(out8, g_fast_reasons, 8 * sizeof(unsigned long long)) == cudaSuccess ? 1 : -1;
#else
    (void)out8;
    return 0;
#endif
}

int paintrl_debug_profile_env(unsigned *out, int n) {
#ifdef PAINTRL_PROFILE
    cudaDeviceSynchronize();
    n = std::min(n, 65536);
    if (out && n > 0) cudaMemcpyFromSymbol(out, g_prof_env, (size_t)n * 32 * sizeof(unsigned));
    return n;
#else
    (void)out; (void)n;
    return 0;
#endif
}

/* Debug only: rays that left the fast path (instrumented build); returns the number copied (<= max_rays). */
int paintrl_debug_rays(double *out, int max_rays, int reset) {
#ifdef PAINTRL_PROFILE
    cudaDeviceSynchronize();
    unsigned long long counts[4];
    cudaMemcpyFromSymbol(counts, g_dbg_counts, sizeof(counts));
    int n = (int)std::min<unsigned long long>(std::min<unsigned long long>(counts[1], 4096), (unsigned long long)max_rays);
    if (out && n > 0) cudaMemcpyFromSymbol(out, g_dbg_rays, (size_t)n * 8 * sizeof(double));
    if (reset) {
        unsigned long long z[4] = {0, 0, 0, 0};
        cudaMemcpyToSymbol(g_dbg_counts, z, sizeof(z));
    }
    return n;
#else
    (void)out; (void)max_rays; (void)reset;
    return 0;
#endif
}

/* Debug only: the last step's per-environment timeline of a -DPAINTRL_TRACE build ([n][8] u64: move start / end,
 * paint start / dependency resolved / inputs loaded / end (globaltimer ns), move SM, paint SM); returns rows copied. */
int paintrl_debug_trace(unsigned long long *out, int n) {
#ifdef PAINTRL_TRACE
    cudaDeviceSynchronize();
    n = std::min(n, 65536);
    if (out && n > 0) cudaMemcpyFromSymbol(out, g_trace, (size_t)n * 8 * sizeof(unsigned long long));
    return n;
#else
    (void)out; (void)n;
    return 0;
#endif
}

int paintrl_create(const PaintrlPartPack *pack, const PaintrlConfig *cfg, int32_t num_envs, int32_t device,
                   PaintrlHandle *out) {
    if (!pack || !cfg || !out) return fail(PAINTRL_E_INVALID, "null argument");
    if (pack->abi_version != PAINTRL_ABI_VERSION || cfg->abi_version != PAINTRL_ABI_VERSION)
        return fail(PAINTRL_E_INVALID, "ABI version mismatch");
    if (num_envs <= 0) return fail(PAINTRL_E_INVALID, "num_envs must be positive");
    if (pack->n_texels <= 0 || pack->n_planes <= 0 || pack->n_vertices <= 0 || pack->n_tris <= 0 || pack->n_starts <= 0)
        return fail(PAINTRL_E_INVALID, "empty part pack table");
    if (pack->axis0 < 0 || pack->axis0 > 2 || pack->axis1 < 0 || pack->axis1 > 2 || pack->axis0 == pack->axis1)
        return fail(PAINTRL_E_INVALID, "bad principal axes");
    if (cfg->action_mode == PAINTRL_ACTION_DISCRETE && (cfg->discrete_granularity <= 0 || !cfg->discrete_table))
        return fail(PAINTRL_E_INVALID, "discrete actions need discrete_granularity > 0 and a discrete_table");
    if (cfg->action_mode == PAINTRL_ACTION_CONTINUOUS && cfg->action_shape != 1 && cfg->action_shape != 2)
        return fail(PAINTRL_E_INVALID, "ACTION_SHAPE must be 1 or 2");
    if (cfg->obs_mode < 0 || cfg->obs_mode > 3 || cfg->obs_grad <= 0) return fail(PAINTRL_E_INVALID, "bad observation mode");
    const int od = obs_dim_of(cfg);
    if (od > kMaxObs) return fail(PAINTRL_E_INVALID, "observation larger than 128 entries is not supported");
    if (cfg->color_mode == PAINTRL_COLOR_HSI && (pack->status_init > 32767 || pack->status_init < -32768))
        return fail(PAINTRL_E_INVALID, "status_init out of int16 range");
    if (cfg->color_mode == PAINTRL_COLOR_RGB && (pack->status_init > 255 || pack->status_init < 0))
        return fail(PAINTRL_E_INVALID, "status_init out of uint8 range");

    int rc = select_device(device);
    if (rc != PAINTRL_OK) return rc;

    PaintrlEngine *e = new PaintrlEngine();
    e->device = device;
    e->num_envs = num_envs;
    e->color = cfg->color_mode == PAINTRL_COLOR_RGB ? 0 : 1;
    rc = build_tables(e, pack, cfg);
    if (rc != PAINTRL_OK) { delete e; return rc; }

    DevConfig &c = e->cfg;
    c.action_mode = cfg->action_mode;
    c.action_shape = cfg->action_mode == PAINTRL_ACTION_CONTINUOUS ? cfg->action_shape : 1;
    c.discrete_granularity = cfg->discrete_granularity;
    c.discrete_table = nullptr;
    if (cfg->action_mode == PAINTRL_ACTION_DISCRETE) {
        std::vector<double> t(cfg->discrete_table, cfg->discrete_table + 3 * ((size_t)cfg->discrete_granularity + 1));
        if (e->arena.upload(t, &c.discrete_table) != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, "upload discrete table"); }
    }
    c.obs_mode = cfg->obs_mode; c.obs_grad = cfg->obs_grad; c.obs_dim = od;
    c.color_mode = cfg->color_mode; c.termination_mode = cfg->termination_mode;
    c.switch_threshold = cfg->switch_threshold;
    c.expected_episode_length = cfg->expected_episode_length;
    c.episode_max_length = cfg->episode_max_length;
    c.turning_penalty = cfg->turning_penalty; c.overlap_penalty = cfg->overlap_penalty;
    c.max_possible_point = cfg->max_possible_point;
    // robot_gym_env.py:297, 302 -- same operations, evaluated once
    c.expected_avg_reward = cfg->max_possible_point / (double)(cfg->expected_episode_length * 100);
    c.hybrid_threshold = cfg->switch_threshold * cfg->max_possible_point / 100;
    c.auto_reset = cfg->auto_reset;
    c.paint_method = cfg->paint_method == PAINTRL_PAINT_NORMAL ? 1 : 0;
    c.n_beams = 0;
    c.beam_plain = nullptr;
    if (c.paint_method == 1) {
        if (cfg->n_beams <= 0 || cfg->n_beams > kMaxBeams || !cfg->beam_plain) { delete e; return fail(PAINTRL_E_INVALID, "the normal paint method needs a beam table of 1..512 rays"); }
        if (e->pk.n_words_pad > kStageWords) { delete e; return fail(PAINTRL_E_INVALID, "the normal paint method supports textures of up to 16384 front texels"); }
        std::vector<double> plain(cfg->beam_plain, cfg->beam_plain + 3 * (size_t)cfg->n_beams);
        if (e->arena.upload(plain, &c.beam_plain) != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, "upload beam table"); }
        c.n_beams = cfg->n_beams;
        e->paint_normal = true;
    }
    { const char *bm = getenv("PAINTRL_DEBUG_BAIL_MOD"); c.debug_bail_mod = bm ? std::max(0, atoi(bm)) : 0; }
    c.seed = cfg->seed;

    const size_t bits_bytes = (size_t)num_envs * e->pk.n_words_pad * sizeof(unsigned);
    const size_t thick_bytes = e->color == 1 ? (size_t)num_envs * e->pk.n_slots * sizeof(int16_t) : 0;
    const size_t gcnt_bytes = (size_t)num_envs * e->pk.n_gcells_pad * sizeof(unsigned);
    const size_t adim = c.action_mode == 0 ? sizeof(long long) : sizeof(double) * c.action_shape;
    double *reset_obs = nullptr;
    bool ok = e->arena.alloc((void **)&e->states, sizeof(EnvState) * (size_t)num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->moves, sizeof(MoveOut) * (size_t)num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->env_stats, sizeof(EnvStat) * (size_t)num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->bits, bits_bytes) == cudaSuccess &&
              (thick_bytes == 0 || e->arena.alloc((void **)&e->thick, thick_bytes) == cudaSuccess) &&
              (gcnt_bytes == 0 || e->arena.alloc((void **)&e->grid_cnt, gcnt_bytes) == cudaSuccess) &&
              e->arena.alloc((void **)&e->stats, 8 * sizeof(unsigned long long)) == cudaSuccess &&
              e->arena.alloc((void **)&e->ready, sizeof(unsigned) * (size_t)num_envs) == cudaSuccess &&
              (!e->paint_normal || (e->arena.alloc((void **)&e->shots, sizeof(ShotPoses) * (size_t)num_envs) == cudaSuccess &&
                                    e->arena.alloc((void **)&e->last_mask, bits_bytes) == cudaSuccess)) &&
              e->arena.alloc((void **)&reset_obs, sizeof(double) * od * (size_t)e->pk.n_starts) == cudaSuccess &&
              e->arena.alloc(&e->stage_actions, adim * num_envs) == cudaSuccess &&
              e->arena.alloc(&e->slot_actions[0], adim * num_envs) == cudaSuccess &&
              e->arena.alloc(&e->slot_actions[1], adim * num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->slot_out[0], (sizeof(double) * (2 * od + 3) + 1) * (size_t)num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->slot_out[1], (sizeof(double) * (2 * od + 3) + 1) * (size_t)num_envs) == cudaSuccess &&
              e->arena.alloc((void **)&e->stage_out, (sizeof(double) * (2 * od + 3) + 1) * (size_t)num_envs) == cudaSuccess;
    if (!ok) { delete e; return fail(PAINTRL_E_CUDA, "device allocation failed (state / status planes)"); }
    cudaError_t err = cudaMemset(e->states, 0, sizeof(EnvState) * (size_t)num_envs);
    if (err == cudaSuccess) err = cudaMemset(e->moves, 0xff, sizeof(MoveOut) * (size_t)num_envs);   // miss_cache = none
    if (err == cudaSuccess) err = cudaMemset(e->env_stats, 0, sizeof(EnvStat) * (size_t)num_envs);
    if (err == cudaSuccess) err = cudaMemset(e->bits, 0, bits_bytes);
    if (err == cudaSuccess && e->thick) {   // the initial colour everywhere; resets only rewrite what an episode touched (clear_planes)
        fill_thickness_kernel<<<1184, 256>>>(e->thick, thick_bytes / sizeof(int16_t), (int16_t)e->pk.status_init);
        err = cudaGetLastError();
    }
    if (err == cudaSuccess && e->grid_cnt) err = cudaMemset(e->grid_cnt, 0, gcnt_bytes);
    if (err == cudaSuccess) err = cudaMemset(e->stats, 0, 8 * sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(e->ready, 0, sizeof(unsigned) * (size_t)num_envs);
    if (err == cudaSuccess && e->paint_normal) err = cudaMemset(e->shots, 0, sizeof(ShotPoses) * (size_t)num_envs);
    if (err == cudaSuccess && e->paint_normal) err = cudaMemset(e->last_mask, 0, bits_bytes);
    if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, std::string("initialising device state: ") + cudaGetErrorString(err)); }
    // observation of a fresh environment at every start point, from environment 0's all-zero planes
    e->pk.reset_obs = reset_obs;
    reset_obs_kernel<<<(e->pk.n_starts + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32>>>(
        e->pk, e->cfg, e->bits, e->grid_cnt, reset_obs);
    err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, cudaGetErrorString(err)); }
    {
        // lanes per environment in the move phase: a full warp while the batch alone cannot fill the GPU
        // (the phase is latency-bound there), 8 lanes once it can (then instruction issue is the limit)
        const char *ml = getenv("PAINTRL_MOVE_LANES");
        int lanes = ml ? atoi(ml) : (num_envs < 16384 ? 32 : 8);   // measured: 4096 envs 60 vs 103 us, 16384 envs 292 vs 249 us (32 vs 8 lanes)
        e->move_lanes = lanes == 8 ? 8 : 32;
        e->force_unstaged = getenv("PAINTRL_FORCE_UNSTAGED") != nullptr;
        const char *fu = getenv("PAINTRL_FUSED");
        e->fused = fu ? (atoi(fu) != 0 ? 1 : 0) : -1;
    }
    err = cudaStreamCreateWithFlags(&e->copy_in, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->copy_out, cudaStreamNonBlocking);
    for (int k = 0; k < 2 && err == cudaSuccess; ++k) {
        err = cudaEventCreateWithFlags(&e->ev_in[k], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_step[k], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_done[k], cudaEventDisableTiming);
    }
    if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, std::string("creating the copy streams: ") + cudaGetErrorString(err)); }
    {
        // L2 prefetch ranges of the static tables (tables beyond 48 MB -- multi-megapixel textures -- are left to
        // demand loads)
        e->pk.pf_n = 0;
        if (e->arena.static_bytes() <= (size_t(48) << 20) && e->arena.slabs.size() <= 4) {
            for (const DeviceArena::Slab &s : e->arena.slabs) {
                e->pk.pf_base[e->pk.pf_n] = s.base;
                e->pk.pf_lines[e->pk.pf_n] = (unsigned)((s.used + 127) / 128);
                e->pk.pf_n++;
            }
        }
    }
    {
        ColdArgs ca;
        ca.pk = e->pk; ca.cfg = e->cfg; ca.ea = env_arrays(e);
        err = e->arena.alloc(&e->cold_args, sizeof(ColdArgs));
        if (err == cudaSuccess) err = cudaMemcpy(e->cold_args, &ca, sizeof(ColdArgs), cudaMemcpyHostToDevice);
        if (err != cudaSuccess) { delete e; return fail(PAINTRL_E_CUDA, std::string("uploading the kernel-argument copy: ") + cudaGetErrorString(err)); }
    }
    *out = e;
    return PAINTRL_OK;
}

void paintrl_destroy(PaintrlHandle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (int k = 0; k < 2; ++k) {
        if (h->ev_in[k]) cudaEventDestroy(h->ev_in[k]);
        if (h->ev_step[k]) cudaEventDestroy(h->ev_step[k]);
        if (h->ev_done[k]) cudaEventDestroy(h->ev_done[k]);
    }
    if (h->copy_in) cudaStreamDestroy(h->copy_in);
    if (h->copy_out) cudaStreamDestroy(h->copy_out);
    delete h;
}

int32_t paintrl_num_envs(PaintrlHandle h) { return h ? h->num_envs : 0; }
int32_t paintrl_obs_dim(PaintrlHandle h) { return h ? h->cfg.obs_dim : 0; }
int32_t paintrl_action_dim(PaintrlHandle h) { return h ? h->cfg.action_shape : 0; }
int32_t paintrl_num_texels(PaintrlHandle h) { return h ? h->pk.n_texels : 0; }
int32_t paintrl_status_bytes(PaintrlHandle h) { return h ? (h->color == 0 ? 1 : 2) : 0; }
int64_t paintrl_state_bytes_per_env(PaintrlHandle h) {
    if (!h) return 0;
    return (int64_t)h->pk.n_words_pad * 4 + (h->color == 1 ? (int64_t)h->pk.n_slots * 2 : 0) + (int64_t)h->pk.n_gcells_pad * 4 +
           (int64_t)(sizeof(EnvState) + sizeof(MoveOut) + sizeof(EnvStat) + sizeof(unsigned));
}

static int reset_like(PaintrlHandle h, const int32_t *env_ids, int32_t n, const int32_t *start_idx, const double *pos,
                      const double *normal, double *obs, void *stream, int mode) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (n <= 0 || n > h->num_envs) return fail(PAINTRL_E_INVALID, "bad env count");
    if (!env_ids && n != h->num_envs) return fail(PAINTRL_E_INVALID, "env_ids == NULL requires n == num_envs");
    CUDA_TRY(cudaSetDevice(h->device));
    const int blocks = (n + kWarpsPerBlock - 1) / kWarpsPerBlock;
    reset_kernel<<<blocks, kWarpsPerBlock * 32, 0, as_stream(stream)>>>(h->pk, h->cfg, env_arrays(h), h->num_envs, env_ids, n, start_idx,
                                                                         pos, normal, obs, mode);
    return launch_check(h, "reset_kernel");
}

int paintrl_reset(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, const int32_t *start_idx_dev, double *obs_dev,
                  void *stream) {
    return reset_like(h, env_ids_dev, n, start_idx_dev, nullptr, nullptr, obs_dev, stream, 0);
}

int paintrl_set_pose(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, const double *pos_dev,
                     const double *normal_dev, double *obs_dev, void *stream) {
    if (!pos_dev || !normal_dev) return fail(PAINTRL_E_INVALID, "null pose");
    return reset_like(h, env_ids_dev, n, nullptr, pos_dev, normal_dev, obs_dev, stream, 1);
}

int paintrl_step(PaintrlHandle h, const void *actions_dev, double *obs_dev, double *reward_dev, double *penalty_dev,
                 double *actual_dev, uint8_t *done_dev, int32_t *new_texels_dev, double *next_obs_dev,
                 const int32_t *reset_start_idx_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    StepIO io;
    const int rc = step_io(h, actions_dev, obs_dev, reward_dev, penalty_dev, actual_dev, done_dev, new_texels_dev, next_obs_dev,
                           reset_start_idx_dev, &io);
    if (rc != PAINTRL_OK) return rc;
    return launch_step<false>(h, EnvSel{nullptr, 0, h->num_envs}, io, stream);
}

int paintrl_step_subset(PaintrlHandle h, const int32_t *env_ids_dev, int32_t env_lo, int32_t n, const void *actions_dev,
                        double *obs_dev, double *reward_dev, double *penalty_dev, double *actual_dev, uint8_t *done_dev,
                        int32_t *new_texels_dev, double *next_obs_dev, const int32_t *reset_start_idx_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    int rc = check_subset(h, env_ids_dev, env_lo, n);
    if (rc != PAINTRL_OK) return rc;
    StepIO io;
    rc = step_io(h, actions_dev, obs_dev, reward_dev, penalty_dev, actual_dev, done_dev, new_texels_dev, next_obs_dev,
                 reset_start_idx_dev, &io);
    if (rc != PAINTRL_OK) return rc;
    return launch_step<true>(h, EnvSel{env_ids_dev, env_lo, n}, io, stream);
}

int paintrl_step_host(PaintrlHandle h, const void *actions_host, double *obs_host, double *reward_host,
                      double *penalty_host, double *actual_host, uint8_t *done_host, double *next_obs_host,
                      void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (!actions_host || !obs_host || !reward_host || !penalty_host || !actual_host || !done_host)
        return fail(PAINTRL_E_INVALID, "null I/O buffer");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t s = as_stream(stream);
    const size_t nenv = (size_t)h->num_envs;
    const size_t abytes = (h->cfg.action_mode == 0 ? sizeof(long long) : sizeof(double) * h->cfg.action_shape) * nenv;
    const size_t obytes = sizeof(double) * h->cfg.obs_dim * nenv;
    const bool want_next = next_obs_host != nullptr, dev_next = want_next && h->cfg.auto_reset;
    CUDA_TRY(cudaMemcpyAsync(h->stage_actions, actions_host, abytes, cudaMemcpyHostToDevice, s));
    // device staging in the order obs | reward | penalty | actual | [next_obs] | done, no gaps
    unsigned char *d = h->stage_out;
    double *d_obs = reinterpret_cast<double *>(d);
    double *d_sc = reinterpret_cast<double *>(d + obytes);
    double *d_next = dev_next ? reinterpret_cast<double *>(d + obytes + 3 * sizeof(double) * nenv) : nullptr;
    uint8_t *d_done = d + obytes + 3 * sizeof(double) * nenv + (dev_next ? obytes : 0);
    int rc = paintrl_step(h, h->stage_actions, d_obs, d_sc, d_sc + nenv, d_sc + 2 * nenv, d_done, nullptr, d_next, nullptr, stream);
    if (rc != PAINTRL_OK) return rc;
    // device -> host: segments that are adjacent on both sides travel as one copy
    struct Seg { void *dst; const void *src; size_t n; };
    Seg segs[7] = {};
    int ns = 0;
    auto push = [&](void *dst, const void *src, size_t n) {
        if (ns > 0 && (const char *)segs[ns - 1].src + segs[ns - 1].n == (const char *)src &&
            (char *)segs[ns - 1].dst + segs[ns - 1].n == (char *)dst) {
            segs[ns - 1].n += n;
        } else {
            segs[ns].dst = dst; segs[ns].src = src; segs[ns].n = n; ++ns;
        }
    };
    push(obs_host, d_obs, obytes);
    push(reward_host, d_sc, sizeof(double) * nenv);
    push(penalty_host, d_sc + nenv, sizeof(double) * nenv);
    push(actual_host, d_sc + 2 * nenv, sizeof(double) * nenv);
    if (dev_next) push(next_obs_host, d_next, obytes);
    push(done_host, d_done, nenv);
    if (want_next && !dev_next) push(next_obs_host, d_obs, obytes);   // no auto-reset: the next observation is this one
    for (int i = 0; i < ns; ++i) CUDA_TRY(cudaMemcpyAsync(segs[i].dst, segs[i].src, segs[i].n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return PAINTRL_OK;
}

int paintrl_step_host_submit(PaintrlHandle h, int32_t slot, const void *actions_host, double *obs_host, double *reward_host,
                             double *penalty_host, double *actual_host, uint8_t *done_host, double *next_obs_host, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    return host_submit(h, slot, false, 0, h->num_envs, actions_host, obs_host, reward_host, penalty_host, actual_host, done_host,
                       next_obs_host, stream);
}

int paintrl_step_host_submit_range(PaintrlHandle h, int32_t slot, int32_t env_lo, int32_t n, const void *actions_host,
                                   double *obs_host, double *reward_host, double *penalty_host, double *actual_host,
                                   uint8_t *done_host, double *next_obs_host, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    const int rc = check_subset(h, nullptr, env_lo, n);
    if (rc != PAINTRL_OK) return rc;
    return host_submit(h, slot, true, env_lo, n, actions_host, obs_host, reward_host, penalty_host, actual_host, done_host,
                       next_obs_host, stream);
}

int paintrl_step_host_wait(PaintrlHandle h, int32_t slot) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (slot < 0 || slot > 1) return fail(PAINTRL_E_INVALID, "slot must be 0 or 1");
    if (!h->slot_pending[slot]) return fail(PAINTRL_E_STATE, "nothing was submitted on this slot");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaEventSynchronize(h->ev_done[slot]));
    h->slot_pending[slot] = false;
    return PAINTRL_OK;
}

int paintrl_get_state(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, int16_t *status_dev, double *pose_dev,
                      double *quat_dev, double *scalars_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (n <= 0 || n > h->num_envs || (!env_ids_dev && n != h->num_envs)) return fail(PAINTRL_E_INVALID, "bad env count");
    CUDA_TRY(cudaSetDevice(h->device));
    dim3 grid(std::max(1, std::min(64, (h->pk.n_texels + 255) / 256)), n);
    get_state_kernel<<<grid, 256, 0, as_stream(stream)>>>(h->pk, env_arrays(h), h->num_envs, env_ids_dev, n, status_dev, pose_dev, quat_dev,
                                                          scalars_dev);
    return launch_check(h, "get_state_kernel");
}

int paintrl_set_state(PaintrlHandle h, const int32_t *env_ids_dev, int32_t n, const int16_t *status_dev,
                      const double *pose_dev, const double *quat_dev, const double *scalars_dev, void *stream) {
    if (!h) return fail(PAINTRL_E_INVALID, "null handle");
    if (n <= 0 || n > h->num_envs || (!env_ids_dev && n != h->num_envs)) return fail(PAINTRL_E_INVALID, "bad env count");
    CUDA_TRY(cudaSetDevice(h->device));
    set_scalars_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(env_arrays(h), h->num_envs, env_ids_dev, n, pose_dev, quat_dev,
                                                                        scalars_dev, status_dev ? 1 : 0);
    int rc = launch_check(h, "set_scalars_kernel");
    if (rc != PAINTRL_OK || !status_dev) return rc;
    set_status_kernel<<<(n + 3) / 4, 128, 0, as_stream(stream)>>>(h->pk, env_arrays(h), h->num_envs, env_ids_dev, n, status_dev);
    return launch_check(h, "set_status_kernel");
}

int paintrl_job_status(PaintrlHandle h, int32_t *painted_dev, void *stream) {
    if (!h || !painted_dev) return fail(PAINTRL_E_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(h->device));
    const int blocks = (h->num_envs + 3) / 4;
    job_status_kernel<<<blocks, 128, 0, as_stream(stream)>>>(h->pk, env_arrays(h), h->num_envs, painted_dev);
    return launch_check(h, "job_status_kernel");
}

int paintrl_stats(PaintrlHandle h, PaintrlStats *out) {
    if (!h || !out) return fail(PAINTRL_E_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(h->device));
    unsigned long long host[5];
    CUDA_TRY(cudaMemset(h->stats, 0, sizeof(host)));
    stats_kernel<<<std::max(1, std::min(64, (h->num_envs + 255) / 256)), 256>>>(h->env_stats, h->num_envs, h->stats);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(host, h->stats, sizeof(host), cudaMemcpyDeviceToHost));
    out->episodes_ended = host[0];
    out->footprint_texels = host[1];
    out->ray_full_scans = host[2] & 0xffffffffull;
    if (getenv("PAINTRL_DEBUG"))
        fprintf(stderr, "[paintrl] rays: %llu full plane scans, %llu verify passes over %llu env-steps\n",
                host[2] & 0xffffffffull, host[2] >> 32, host[3]);
    out->env_steps = host[3];
    out->kernel_launches = h->launches;
    out->move_bailouts = host[4];
    return PAINTRL_OK;
}

}  // extern "C"
