"""NumPy restatement of sr_mrf_select (include/sr_b200.h, stereoreconstruction_b200/csrc/sr_mrf.cuh): the model,
the checkerboard schedule and the FP32 summation order, so that the GPU's labels, maps and energy can be compared
bit for bit; exact dynamic programming (Viterbi) on chains; random and adversarial peak lists.

Every FP32 value is a numpy float32 array or np.float32 scalar (NEP 50: a Python float next to a float32 array
would also stay float32, but the constants are typed to keep that independent of the numpy version)."""
import numpy as np

F = np.float32
K, U, L = 9, 9, 10
FLT_MAX = float(np.finfo(np.float32).max)
INF32 = F(np.inf)
SR_INDEX_NONE = -1
# the direction a message travels (sender -> receiver offset dy, dx) for targets left, right, up, down; the
# receiver files it under the opposite side
OFFSETS = ((0, -1), (0, 1), (-1, 0), (1, 0))
SLOT = (1, 0, 3, 2)


def _term(v):
    return F(0.0) if v == 0 else F(v)


def terms(mp):
    """(D(U), smooth_weight, smooth_trunc, unknown_pair) as the kernels use them (FP32, +0 for a zero)."""
    return _term(mp.unknown_cost), _term(mp.smooth_weight), _term(mp.smooth_trunc), _term(mp.unknown_pair)


def prepare(peaks, P):
    """unary (9, h, w) and z / step (9, h, w) in float32 from (h, w, 9, 2) float64 lists and the sr_params P:
    +INF and NaN for a slot that is no hypothesis."""
    ncc = np.moveaxis(peaks[..., 0], -1, 0)
    z = np.moveaxis(peaks[..., 1], -1, 0)
    hyp = np.isfinite(ncc) & np.isfinite(z) & ~((ncc == 0.0) & (z == -1.0))
    step = (P.max_depth - P.min_depth) / (P.num_levels - 1.0)
    with np.errstate(all="ignore"):
        d = np.maximum((1.0 - ncc) / (1.0 - P.ncc_threshold), 0.0).astype(F)
        s = np.clip(z / step, -FLT_MAX, FLT_MAX).astype(F)
    return np.where(hyp, d, INF32), np.where(hyp, s, F(np.nan))


def vpair(zk, zl, weight, trunc):
    with np.errstate(invalid="ignore"):
        return weight * np.fmin(np.abs(zk - zl), trunc)


def shift(a, dy, dx, fill):
    """b[..., y, x] = a[..., y + dy, x + dx], `fill` outside the image."""
    b = np.full_like(a, fill)
    h, w = a.shape[-2:]
    ys, yd = slice(max(dy, 0), h + min(dy, 0)), slice(max(-dy, 0), h + min(-dy, 0))
    xs, xd = slice(max(dx, 0), w + min(dx, 0)), slice(max(-dx, 0), w + min(-dx, 0))
    b[..., yd, xd] = a[..., ys, xs]
    return b


def half_sweep(msg, unary, zs, inmask, colour, mp):
    """Messages sent by the in-mask pixels with (x + y) & 1 == colour, in place."""
    du, wt, tr, up = terms(mp)
    h, w = inmask.shape
    yy, xx = np.mgrid[0:h, 0:w]
    sender = inmask & (((yy + xx) & 1) == colour)
    D = np.concatenate([unary, np.full((1, h, w), du, F)])
    hyp = ~np.isnan(zs)
    for t, (dy, dx) in enumerate(OFFSETS):
        has = sender & shift(inmask, dy, dx, False)
        if not has.any():
            continue
        S = D.copy()
        for d in range(4):
            if d != t:
                S = S + msg[d]
        hmin = np.where(hyp, S[:K], INF32).min(axis=0)
        zq = shift(zs, dy, dx, F(np.nan))
        hypq = ~np.isnan(zq)
        m = np.empty((L, h, w), F)
        m[U] = np.minimum(S[U], hmin + up)
        mn = m[U].copy()
        from_u = S[U] + up
        for l in range(K):
            v = from_u.copy()
            for k in range(K):
                v = np.minimum(v, np.where(hyp[k], S[k] + vpair(zs[k], zq[l], wt, tr), INF32))
            mn = np.minimum(mn, np.where(hypq[l], v, INF32))
            m[l] = v
        out = np.where(np.concatenate([hypq, np.ones((1, h, w), bool)]), m - mn, F(0.0))
        recv = shift(has, -dy, -dx, False)  # receivers of the senders that have a neighbour on side t
        msg[SLOT[t]][:, recv] = out[:, has]


def run_bp(unary, zs, inmask, mp):
    h, w = inmask.shape
    msg = np.zeros((4, L, h, w), F)
    for _ in range(mp.iterations):
        half_sweep(msg, unary, zs, inmask, 0, mp)
        half_sweep(msg, unary, zs, inmask, 1, mp)
    return msg


def labels_from(msg, unary, zs, inmask, mp):
    """argmin of D + from left + right + up + down; the highest hypothesis slot wins a tie, U loses every tie."""
    du = terms(mp)[0]
    b = np.full(inmask.shape, du, F)
    for d in range(4):
        b = b + msg[d, U]
    lab = np.full(inmask.shape, U, np.int32)
    for k in range(K):
        bk = unary[k]
        for d in range(4):
            bk = bk + msg[d, k]
        take = ~np.isnan(zs[k]) & (bk <= b)
        b = np.where(take, bk, b)
        lab = np.where(take, k, lab)
    return np.where(inmask, lab, -1)


def pair_terms(la, za, lb, zb, mp):
    """FP32 V between labellings la (with its z / step za) and lb (zb), elementwise."""
    _, wt, tr, up = terms(mp)
    ka, kb = np.clip(la, 0, K - 1), np.clip(lb, 0, K - 1)
    ga = np.take_along_axis(za, ka[None], 0)[0]
    gb = np.take_along_axis(zb, kb[None], 0)[0]
    v = vpair(ga, gb, wt, tr)
    v = np.where((la == U) != (lb == U), up, v)
    return np.where((la == U) & (lb == U), F(0.0), v)


def energy(lab, unary, zs, inmask, mp):
    """Energy of a labelling: the FP32 unary and pairwise terms summed in FP64."""
    du = terms(mp)[0]
    k = np.clip(lab, 0, K - 1)
    d = np.where(lab == U, du, np.take_along_axis(unary, k[None], 0)[0])
    e = d[inmask].astype(np.float64).sum()
    for dy, dx in ((0, 1), (1, 0)):
        both = inmask & shift(inmask, dy, dx, False)
        v = pair_terms(lab, zs, shift(lab, dy, dx, U), shift(zs, dy, dx, F(np.nan)), mp)
        e += v[both].astype(np.float64).sum()
    return float(e)


def mrf_select(peaks, mask, P, mp, depth0=None, best0=None, index0=None):
    """The oracle of sr_mrf_select: (labels, depth, best, index, energy).  depth0/best0/index0 are the view's maps
    before the call (masked pixels keep them); labels are 0..8, 9 = U, -1 off the mask."""
    h, w = mask.shape
    inmask = mask == 255
    unary, zs = prepare(peaks, P)
    msg = run_bp(unary, zs, inmask, mp)
    lab = labels_from(msg, unary, zs, inmask, mp)
    depth = np.full((h, w), np.nan) if depth0 is None else depth0.copy()
    best = np.full((h, w), np.nan) if best0 is None else best0.copy()
    index = np.full((h, w), SR_INDEX_NONE, np.int32) if index0 is None else index0.copy()
    hyp_here = inmask & (lab != U)
    k = np.clip(lab, 0, K - 1)
    pz = np.take_along_axis(peaks[..., 1], k[..., None], -1)[..., 0]
    pc = np.take_along_axis(peaks[..., 0], k[..., None], -1)[..., 0]
    depth[inmask] = np.where(hyp_here, pz, -1.0)[inmask]
    best[inmask] = np.where(hyp_here, pc, 0.0)[inmask]
    index[inmask] = np.where(hyp_here, lab, SR_INDEX_NONE)[inmask]
    return lab, depth, best, index, energy(lab, unary, zs, inmask, mp)


def viterbi_chain(unary, zs, mp):
    """Exact minimum energy (FP64 sum of the FP32 terms) and a minimising labelling of a chain: unary and zs of
    shape (9, N) with every node in the model."""
    du, wt, tr, up = terms(mp)
    N = unary.shape[1]
    D = np.concatenate([unary, np.full((1, N), du, F)]).astype(np.float64)
    hyp = np.concatenate([~np.isnan(zs), np.ones((1, N), bool)])
    D[~hyp] = np.inf
    cost = D[:, 0].copy()
    back = np.zeros((N, L), np.int64)
    for i in range(1, N):
        a = np.arange(L)[:, None]
        b = np.arange(L)[None, :]
        la, lb = np.broadcast_to(a, (L, L)), np.broadcast_to(b, (L, L))
        za = np.broadcast_to(zs[np.clip(la, 0, K - 1), i - 1], (L, L)).copy()
        zb = np.broadcast_to(zs[np.clip(lb, 0, K - 1), i], (L, L)).copy()
        V = vpair(za, zb, wt, tr)
        V = np.where((la == U) != (lb == U), up, V)
        V = np.where((la == U) & (lb == U), F(0.0), V).astype(np.float64)
        V[~hyp[:, i - 1], :] = np.inf
        V[:, ~hyp[:, i]] = np.inf
        tot = cost[:, None] + V
        back[i] = np.argmin(tot, axis=0)
        cost = tot[back[i], np.arange(L)] + D[:, i]
    lab = np.zeros(N, np.int64)
    lab[-1] = int(np.argmin(cost))
    for i in range(N - 1, 0, -1):
        lab[i - 1] = back[i, lab[i]]
    return float(cost.min()), lab


def random_lists(h, w, rng, P, adversarial=True):
    """(h, w, 9, 2) peak lists: ascending (ncc, depth) lists of 0..9 candidates above the threshold padded with
    (0, -1) in front, as a run keeps them; with `adversarial`, also all-padding pixels, NaN and infinite depths,
    NaN ncc, duplicate pairs and unsorted lists."""
    lists = np.zeros((h, w, K, 2))
    lists[..., 1] = -1.0
    step = (P.max_depth - P.min_depth) / (P.num_levels - 1.0)
    count = rng.randint(0, K + 1, size=(h, w))
    ncc = rng.uniform(P.ncc_threshold, 1.0, size=(h, w, K))
    z = P.min_depth + step * rng.randint(0, P.num_levels, size=(h, w, K))
    order = np.lexsort((z, ncc), axis=-1)
    ncc = np.take_along_axis(ncc, order, -1)
    z = np.take_along_axis(z, order, -1)
    for k in range(K):
        real = k >= K - count
        lists[..., k, 0] = np.where(real, ncc[..., k], 0.0)
        lists[..., k, 1] = np.where(real, z[..., k], -1.0)
    if adversarial:
        flat = lists.reshape(-1, K, 2)
        n = flat.shape[0]
        pick = rng.permutation(n)
        q = max(1, n // 12)
        flat[pick[:q]] = (0.0, -1.0)                                   # all padding
        flat[pick[q:2 * q], rng.randint(0, K), 1] = np.nan             # NaN depth
        flat[pick[2 * q:3 * q], rng.randint(0, K), 1] = np.inf         # infinite depth
        flat[pick[3 * q:4 * q], rng.randint(0, K), 0] = np.nan         # NaN ncc
        flat[pick[4 * q:5 * q], K - 2] = flat[pick[4 * q:5 * q], K - 1]  # duplicate of the best pair
        for i in pick[5 * q:6 * q]:                                    # unsorted
            flat[i] = flat[i][rng.permutation(K)]
        flat[pick[6 * q:6 * q + 1], 0] = (1.5, P.max_depth)            # ncc above 1: D clamps to 0
    return lists
