"""NumPy restatements of the prioritized-replay pieces (helpers, no tests): the sum / min tree rebuild, the sampling
descent and the importance weights of csrc/paintrl_replay.cuh, and the n-step transitions of `dqn.ReplayBuffer.add` as
a plain per-transition loop.  The tree and descent replicas use the same FP64 operations in the same order as the
kernels (one addition or fmin per node, one subtraction per right turn), so they must agree bit for bit."""
import numpy as np


def empty_tree(L):
    return np.zeros(2 * L), np.full(2 * L, np.inf)


def rebuild(sum_tree, min_tree, L):
    """Every internal node from its two children, bottom up (in place)."""
    n = L // 2
    while n >= 1:
        sum_tree[n:2 * n] = sum_tree[2 * n:4 * n:2] + sum_tree[2 * n + 1:4 * n:2]
        min_tree[n:2 * n] = np.fmin(min_tree[2 * n:4 * n:2], min_tree[2 * n + 1:4 * n:2])
        n //= 2
    return sum_tree, min_tree


def tree_from_leaves(leaves, L):
    """Trees of L leaves whose first len(leaves) are `leaves` (0 = unfilled) and the rest unfilled."""
    s, m = empty_tree(L)
    leaves = np.asarray(leaves, dtype=np.float64)
    s[L:L + len(leaves)] = leaves
    m[L:L + len(leaves)] = np.where(leaves > 0, leaves, np.inf)
    return rebuild(s, m, L)


def descend(sum_tree, L, u):
    """The rows prio_sample_kernel returns for uniforms u (FP64)."""
    u = np.asarray(u, dtype=np.float64)
    root = sum_tree[1]
    mass = u * root
    mass = np.where(mass < root, mass, np.nextafter(root, 0.0))
    i = np.ones(u.shape, dtype=np.int64)
    while True:
        if (i >= L).all():
            break
        left = sum_tree[2 * i]
        right = sum_tree[2 * i + 1]
        go_right = ~(mass < left) & (right > 0.0)
        mass = np.where(go_right, mass - left, mass)
        i = 2 * i + go_right.astype(np.int64)
    return i - L


def weights(sum_tree, min_tree, L, idx, beta):
    """(p_i / p_min)^(-beta) in FP64 (NumPy's pow; the kernel's CUDA pow may differ in the last bits)."""
    return (sum_tree[L + np.asarray(idx)] / min_tree[1]) ** (-float(beta))


def nstep_ring(frags, n, gamma, capacity):
    """The ring (obs, next_obs, actions, reward, done) after inserting `frags` in order into an empty buffer, built
    transition by transition: the fragments are concatenated per environment, transition t (global time) is emitted
    once steps t .. t + n - 1 have all been seen, in (t, env) order, and lands on ring row (emission index) % capacity.
    Returns the ring and the count of transitions whose window an episode end cut at each offset k < n."""
    obs = np.concatenate([f.obs[:f.T].numpy() for f in frags])
    term = np.concatenate([f.term_obs.numpy() for f in frags])
    act = np.concatenate([f.actions.numpy() for f in frags])
    r = np.concatenate([f.actual.numpy() for f in frags])
    done = np.concatenate([f.done.numpy() for f in frags])
    G, B = r.shape
    D = obs.shape[2]
    ring = (np.zeros((capacity, D)), np.zeros((capacity, D)), np.zeros(capacity, np.int64), np.zeros(capacity, np.float32),
            np.zeros(capacity, np.uint8))
    cut_at = np.zeros(n, dtype=np.int64)
    q = 0
    for t in range(G - n + 1):
        for b in range(B):
            R, m = 0.0, n
            for k in range(n):
                R += gamma ** k * r[t + k, b]
                if done[t + k, b]:
                    m = k + 1
                    cut_at[k] += 1
                    break
            row = q % capacity
            ring[0][row] = obs[t, b]
            ring[1][row] = term[t + m - 1, b]
            ring[2][row] = act[t, b]
            ring[3][row] = np.float32(R)
            ring[4][row] = done[t + m - 1, b]
            q += 1
    return ring, q, cut_at
