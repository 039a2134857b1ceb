"""NumPy FP64 restatement of sr_fuse_points (the model in include/sr_b200.h), with the flags of every decision.

The geometry comes in as arguments: `rays[v]` is view v's (h, w, 6) unproject grid at the image scale and
`project(u, xyz)` returns (xy, ok) of cam_project into view u.  With the oracle's Scene.unproject_grid /
project_points this is a CPU reference; with the library's ctx.unproject_grid / ctx.project_points the GPU
comparisons test the fusion logic alone."""
import numpy as np

from test_gpu_point_cloud import reference_points


def view_points(cam, rays, depth, min_depth):
    """(h*w, 3) point of every pixel (NaN without one) and the (h*w,) has-a-point flags (sr_get_points' rule)."""
    n = depth.size
    p, idx, _ = reference_points(cam, rays, depth, min_depth)
    pts = np.full((n, 3), np.nan)
    pts[idx] = p
    has = np.zeros(n, bool)
    has[idx] = True
    return pts, has


def fuse(cams, rays, project, depths, imgs, min_depth, scale, max_dist, min_views, points=None):
    """The fused cloud and the decisions behind it.  `points`, when given, replaces view_points: per view the
    (h*w, 3) points and (h*w,) flags (e.g. from the library's sr_get_points, so that every sum compares bit for bit).

    Returns a dict with
      xyz (m, 3), rgb (m, 3) uint8, source (m, 2) int32  the cloud, view-major, row-major within a view;
      support[v]   (h*w,) support of every pixel, -1 without a point;
      kept[v], blocked[v]  (h*w,) kept, and kept but not emitted (a confirming lower view's pixel is kept);
      lower_unkept[v]  emitted although a confirming lower view's pixel is not kept;
      reject       counts of rejected matches: off_image (projection fails or falls outside), no_point (pixel q
                   has no point), distance (|X - X_u| not finite or >= max_dist);
      ties         (distances |X - X_u| within 1e-9 * max(1, max_dist) of max_dist, in-image projected
                   coordinates within 1e-9 of an integer): the near-tie guard."""
    V = len(depths)
    h, w = depths[0].shape
    n = h * w
    if points is None:
        points = [view_points(cams[v], rays[v], depths[v], min_depth) for v in range(V)]
    P, has = zip(*points)
    rgb_all = [np.asarray(im)[..., :3].reshape(-1, 3).astype(np.int64) for im in imgs]
    reject = dict(off_image=0, no_point=0, distance=0)
    ties = [0, 0]
    support, agree_of, q_of, fused_xyz, fused_rgb = [], [], [], [], []
    for v in range(V):
        S = np.flatnonzero(has[v])
        X = P[v][S]
        total = X.copy()  # X first, then the agreeing views in ascending order
        col = rgb_all[v][S].copy()
        sup = np.zeros(len(S), np.int64)
        agree, qs = {}, {}
        for u in range(V):
            if u == v:
                continue
            xy, ok = project(u, X)
            with np.errstate(invalid="ignore"):
                x2, y2 = xy[:, 0] * scale, xy[:, 1] * scale
                inb = (ok != 0) & (x2 >= 0) & (y2 >= 0) & (x2 < w) & (y2 < h)
            q = np.zeros(len(S), np.int64)
            q[inb] = y2[inb].astype(np.int64) * w + x2[inb].astype(np.int64)
            c = np.concatenate([x2[inb], y2[inb]])
            ties[1] += int((np.abs(c - np.round(c)) <= 1e-9).sum())
            qp = inb & has[u][q]
            Xu = P[u][q]
            d = X - Xu
            with np.errstate(invalid="ignore", over="ignore"):
                dist = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
                a = qp & np.isfinite(dist) & (dist < max_dist)
            dq = dist[qp]
            ties[0] += int((np.abs(dq[np.isfinite(dq)] - max_dist) <= 1e-9 * max(1.0, max_dist)).sum())
            reject["off_image"] += int((~inb).sum())
            reject["no_point"] += int((inb & ~qp).sum())
            reject["distance"] += int((qp & ~a).sum())
            total[a] = total[a] + Xu[a]
            col[a] += rgb_all[u][q[a]]
            sup += a
            agree[u], qs[u] = a, q
        m = 1 + sup
        fused_xyz.append(total / m.astype(np.float64)[:, None])
        fused_rgb.append(((col + (m // 2)[:, None]) // m[:, None]).astype(np.uint8))
        s_full = np.full(n, -1, np.int64)
        s_full[S] = sup
        support.append(s_full)
        agree_of.append(agree)
        q_of.append(qs)
    kept = [support[v] >= min_views for v in range(V)]
    xyz, rgb, source, blocked, lower_unkept = [], [], [], [], []
    for v in range(V):
        S = np.flatnonzero(has[v])
        k = kept[v][S]
        blk = np.zeros(len(S), bool)
        unk = np.zeros(len(S), bool)
        for u in range(v):
            a, q = agree_of[v][u], q_of[v][u]
            ku = kept[u][q]
            blk |= a & ku
            unk |= a & ~ku
        emit = k & ~blk
        b_full = np.zeros(n, bool)
        b_full[S] = k & blk
        u_full = np.zeros(n, bool)
        u_full[S] = emit & unk
        blocked.append(b_full)
        lower_unkept.append(u_full)
        xyz.append(fused_xyz[v][emit])
        rgb.append(fused_rgb[v][emit])
        source.append(np.stack([np.full(int(emit.sum()), v), S[emit]], 1).astype(np.int32))
    return dict(xyz=np.concatenate(xyz).reshape(-1, 3), rgb=np.concatenate(rgb).reshape(-1, 3),
                source=np.concatenate(source).reshape(-1, 2), support=support, kept=kept, blocked=blocked,
                lower_unkept=lower_unkept, reject=reject, ties=tuple(ties))


def assert_same_cloud(got, want, what=""):
    """(view, pixel) sequence and rgb identical, xyz within 1e-12 relative."""
    xyz, rgb, src = got
    assert src.shape == want["source"].shape, (what, src.shape, want["source"].shape)
    assert (src == want["source"]).all(), what
    assert (rgb == want["rgb"]).all(), what
    err = np.abs(xyz - want["xyz"]) / np.maximum(1.0, np.abs(want["xyz"]))
    assert err.size == 0 or err.max() <= 1e-12, (what, err.max())
    return len(src)
