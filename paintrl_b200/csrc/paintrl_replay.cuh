// paintrl_replay.cuh -- prioritized replay on the device (RLlib's PrioritizedReplayBuffer): a sum tree and a min tree
// over the replay ring's priorities, the sampling descent, and the priority updates the DQN learner issues after every
// gradient step.  The trees are caller-owned FP64 buffers; the kernels keep no state.
//
// Layout: L = a power of two >= the ring's capacity.  sum[2L], min[2L]: node 1 is the root, node i has children 2i and
// 2i + 1, leaf r (ring row r) is node L + r.  A filled leaf holds p_r^alpha in both trees; an unfilled one holds 0 in
// the sum tree and +inf in the min tree.
//
// Internal nodes are a pure function of the leaves: every node is sum[2i] + sum[2i + 1] and fmin(min[2i], min[2i + 1]),
// recomputed from its children after every leaf write (prio_build_kernel) -- never updated incrementally.  The tree is
// therefore the same bits whatever order leaves were written in and whatever implementation rebuilt it.
#pragma once

namespace paintrl {

constexpr int kPrioSubtree = 2048;             // leaves of one prio_build_kernel CTA
constexpr int kPrioBuildThreads = 1024;
constexpr int kPrioThreads = 256;
constexpr int kPrioMaxBatch = 1 << 24;         // largest n of a sample or update call (they take no handle to size it)

// Rebuild the kPrioSubtree-wide (or narrower, `width`) subtrees above one level of the tree: CTA b takes the level's
// nodes [base + b width, base + (b + 1) width) and writes the width - 1 nodes above them, up to the subtree root
// base / width + b.  base is the level's first node index, which is also its node count.  The first level is read from
// global memory; the levels above it are built in shared memory, one level per pass, each node from its two children.
__global__ void __launch_bounds__(kPrioBuildThreads) prio_build_kernel(double *sum, double *mn, int base, int width) {
    __shared__ double ssum[kPrioSubtree], smin[kPrioSubtree];      // local heap: node 1 the subtree root
    const int tid = threadIdx.x;
    const long long root = base / width + blockIdx.x;
    // local node k at depth d (k in [2^d, 2^(d+1))) is global node root * 2^d + (k - 2^d)
    for (int w = width >> 1, first = 1; w >= 1; w >>= 1, first = 0) {
        const int depth = 31 - __clz(w);
        for (int k = w + tid; k < 2 * w; k += kPrioBuildThreads) {
            double s, m;
            if (first) {
                const long long g = (root << (depth + 1)) + 2 * (k - w);                  // the left child, a level node
                s = sum[g] + sum[g + 1];
                m = fmin(mn[g], mn[g + 1]);
            } else {
                s = ssum[2 * k] + ssum[2 * k + 1];
                m = fmin(smin[2 * k], smin[2 * k + 1]);
            }
            ssum[k] = s;
            smin[k] = m;
            const long long g = (root << depth) + (k - w);
            sum[g] = s;
            mn[g] = m;
        }
        __syncthreads();
    }
}

// After a gradient step: leaf idx[j] <- (|td_j| + eps)^alpha in FP64, and max_priority <- max(max_priority, |td_j| +
// eps) with an integer atomicMax on the FP64 bits (monotone for non-negative doubles, so exact and order-free).
// Duplicate indices carry bit-identical td, so they write the same leaf value.
__global__ void prio_update_kernel(double *sum, double *mn, int L, const int *idx, const float *td, int n, double *max_priority,
                                   double alpha, double eps) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double p = fabs((double)td[j]) + eps;
    const double leaf = pow(p, alpha);
    const long long g = (long long)L + idx[j];
    sum[g] = leaf;
    mn[g] = leaf;
    atomicMax(reinterpret_cast<unsigned long long *>(max_priority), (unsigned long long)__double_as_longlong(p));
}

// On insertion: ring rows [start, start + count) mod capacity get max_priority^alpha (RLlib gives new transitions the
// largest priority seen so far).
__global__ void prio_fill_kernel(double *sum, double *mn, int L, int capacity, int start, int count, const double *max_priority,
                                 double alpha) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const double leaf = pow(*max_priority, alpha);
    int r = start + j;
    if (r >= capacity) r -= capacity;
    sum[(long long)L + r] = leaf;
    mn[(long long)L + r] = leaf;
}

// One sample per thread: mass = u_j * root (clamped below the root), descend -- left when the mass is below the left
// child's sum, otherwise subtract it and go right, but only when the right child's sum is positive.  Every node on the
// path then has a positive sum, so the leaf reached has a positive priority, and unfilled rows (sum 0) are never
// returned.  weight = (p_i / p_min)^(-beta) in FP64, p_min the min-tree root: RLlib's (N P(i))^-beta / max_j
// (N P(j))^-beta, at most 1, and exactly 1 on the minimum-priority rows.
__global__ void prio_sample_kernel(const double *sum, const double *mn, int L, const double *u, int n, double beta, int *idx_out,
                                   float *weight_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double root = sum[1];
    double mass = u[j] * root;
    if (!(mass < root)) mass = nextafter(root, 0.0);
    int i = 1;
    while (i < L) {
        const double left = sum[2 * i];
        if (mass < left) {
            i = 2 * i;
        } else if (sum[2 * i + 1] > 0.0) {
            mass -= left;
            i = 2 * i + 1;
        } else {
            i = 2 * i;
        }
    }
    idx_out[j] = i - L;
    weight_out[j] = (float)pow(sum[i] / mn[1], -beta);
}

}  // namespace paintrl
