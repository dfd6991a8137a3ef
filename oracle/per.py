"""numpy restatement of the prioritized-replay store of fastdeepqlearning_b200/csrc/per.cu (proportional PER, Schaul et al. 2016):
the same 32-ary layout and child order, the same fp64 node sums (butterfly order of a warp reduction), the descent from given
stratum offsets xi, the importance weights and the priority update rule."""
import numpy as np

K = 32


def _levels_of(n0):
    ns = [int(n0)]
    while len(ns) == 1 or ns[-1] > 1:
        ns.append((ns[-1] + K - 1) // K)
    return ns


def _node_sums(child_sums):
    """fp64 sums of consecutive groups of 32 in the order of a warp's xor butterfly (lane 0's result)."""
    n = (len(child_sums) + K - 1) // K
    x = np.zeros(n * K, np.float64)
    x[:len(child_sums)] = child_sums
    x = x.reshape(n, K)
    h = K // 2
    while h >= 1:
        x = x[:, :h] + x[:, h:2 * h]
        h //= 2
    return x[:, 0]


def _node_mins(child_mins):
    n = (len(child_mins) + K - 1) // K
    x = np.full(n * K, np.inf, np.float32)
    x[:len(child_mins)] = child_mins
    return x.reshape(n, K).min(1)


def build(leaves):
    """[(sums, mins)] of levels 1 .. L above the fp32 leaves (root last); a min covers positive leaves only (+inf: none)."""
    leaves = np.asarray(leaves, np.float32)
    out = []
    s = leaves.astype(np.float64)
    m = np.where(leaves > 0, leaves, np.float32(np.inf)).astype(np.float32)
    for _ in range(len(_levels_of(len(leaves))) - 1):
        s, m = _node_sums(s), _node_mins(m)
        out.append((s, m))
    return out


def descend(leaves, tree, targets):
    """Leaf of each fp64 target: per level the first child whose running sum (sequential fp64) exceeds the remaining target, the last
    positive child when rounding left none."""
    leaves = np.asarray(leaves, np.float32)
    res = np.empty(len(targets), np.int64)
    for i, t in enumerate(np.asarray(targets, np.float64)):
        node = 0
        for l in range(len(tree), 0, -1):
            below = leaves.astype(np.float64) if l == 1 else tree[l - 2][0]
            v = below[K * node:K * node + K]
            incl = np.cumsum(v)
            hit = np.nonzero(incl > t)[0]
            if len(hit):
                c = int(hit[0])
            else:
                pos = np.nonzero(v > 0)[0]
                c = int(pos[-1]) if len(pos) else 0
            t -= incl[c - 1] if c > 0 else 0.0
            node = K * node + c
        res[i] = node
    return res


def targets(tree, xi):
    """Stratified targets S (b + xi_b) / n."""
    S = tree[-1][0][0]
    n = len(xi)
    return S * ((np.arange(n, dtype=np.float64) + np.asarray(xi, np.float64)) / np.float64(n))


def sample(leaves, xi, beta):
    """(starts, is_weight) for injected xi: weight = (q_min / q[start])^beta in fp64, stored as fp32."""
    leaves = np.asarray(leaves, np.float32)
    tree = build(leaves)
    starts = descend(leaves, tree, targets(tree, xi))
    qmin = np.float64(tree[-1][1][0])
    w = (qmin / leaves[starts].astype(np.float64)) ** np.float64(np.float32(beta))
    return starts, w.astype(np.float32)


def update(leaves, q_max, starts, loss, contig, alpha, eps, eta):
    """New (leaves, q_max) after one update: per window delta = eta max + (1 - eta) mean of its contiguous transitions' loss (fp32 max
    and sequential fp32 sum, 0 when none), q = fp32((delta + eps)^alpha) floored at the smallest normal fp32; a non-finite loss or q
    writes the q_max of before the update; a 0 leaf stays 0; duplicates: the largest window index wins."""
    leaves = np.array(leaves, np.float32, copy=True)
    loss = np.asarray(loss, np.float32).reshape(-1, len(starts))
    contig = np.ones_like(loss) if contig is None else np.asarray(contig, np.float32).reshape(loss.shape)
    alpha, eps, eta = (np.float64(np.float32(x)) for x in (alpha, eps, eta))
    q_old = np.float32(q_max)
    new_max = np.float32(0)
    last = {int(s): b for b, s in enumerate(starts)}
    for s, b in last.items():
        if not leaves[s] > 0:
            continue
        vals = [loss[t, b] for t in range(loss.shape[0]) if contig[t, b] != 0]
        bad = any(not np.isfinite(v) for v in vals)
        if vals:
            mx = np.float32(max(vals)) if not bad else np.float32(0)
            sm = np.float32(0)
            for v in vals:
                sm = np.float32(sm + v)
            delta = eta * np.float64(mx) + (1.0 - eta) * np.float64(np.float32(sm / np.float32(len(vals))))
        else:
            delta = 0.0
        with np.errstate(over="ignore", invalid="ignore"):
            q = np.float32((delta + eps) ** alpha)
        if bad or not np.isfinite(q):
            q = q_old
        else:
            q = max(q, np.float32(np.finfo(np.float32).tiny))
            new_max = max(new_max, q)
        leaves[s] = q
    return leaves, max(q_old, new_max)


def eligible(capacity, length, T):
    """The eligibility invariant: leaf r is positive iff r < len - T."""
    return np.arange(capacity) < length - T
