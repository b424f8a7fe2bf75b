"""TEST INFRASTRUCTURE -- numpy restatement of the point-to-plane PSNR definition (DESIGN.md, "Point-to-plane PSNR";
csrc/normals.cu).  NOT product code.

Both clouds are range images over one ray table; a cloud's points are the pixels with x+y+z != 0 (f32, as
utils/evaluate_metrics.py:14-15).  Distances are the chamfer kernel's f32 expression fma(z,z, fma(x,x, y*y)) on b - a,
restated here with an exactly rounded f32 fma.

  neighbourhood  the knn nearest points of the point's own cloud, itself included, restricted to d <= radius^2 (f32);
                 ties to the smaller flat pixel index.  Brute force, or -- for large images -- scipy cKDTree candidates
                 (knn + 8) re-ranked with the exact f32 distance, brute force wherever the candidates' margin is unclear.
  normal         f64 two-pass covariance (/ n), numpy.linalg.eigh; the eigenvector of the smallest eigenvalue, oriented
                 so that n . p <= 0.  None (0,0,0) when n < 3, lambda2 == 0 or lambda1 - lambda0 <= 1e-6 lambda2.
  error          for a of one cloud, b = its nearest point of the other (first minimum, smallest pixel index):
                 ((a - b) . n(b))^2 in f64, or the f32 squared distance when b has no normal.
"""
import numpy as np

F32, F64 = np.float32, np.float64


def fmaf(a, b, c):
    """Exactly rounded f32 fused multiply-add of f32 arrays (a*b is exact in f64; the one sum that f64 can round onto an
    f32 rounding midpoint is settled by its exact error term)."""
    a, b, c = (np.asarray(x, F32) for x in (a, b, c))
    p = a.astype(F64) * b.astype(F64)
    c64 = c.astype(F64)
    s = p + c64
    bb = s - p
    e = (p - (s - bb)) + (c64 - bb)                  # TwoSum: p + c == s + e exactly
    r = s.astype(F32)
    rd = r.astype(F64)
    with np.errstate(invalid="ignore", over="ignore"):
        other = np.nextafter(r, np.where(s > rd, F32(np.inf), F32(-np.inf)).astype(F32))
        mid = (rd + other.astype(F64)) * 0.5
        flip = (s == mid) & (e != 0) & (rd != s) & (np.sign(e) == np.sign(other.astype(F64) - s))
    return np.where(flip, other, r)


def cham_d(q, pts):
    """f32 squared distances from q (...,3) to pts (...,3), the chamfer kernel's expression on pts - q."""
    x = (pts[..., 0] - q[..., 0]).astype(F32)
    y = (pts[..., 1] - q[..., 1]).astype(F32)
    z = (pts[..., 2] - q[..., 2]).astype(F32)
    return fmaf(z, z, fmaf(x, x, (y * y).astype(F32)))


def cloud(range_image, lut):
    """-> (points (HW,3) f32, valid (HW,) bool) of a range image (PCTransformer.range_image_to_point_cloud)."""
    pts = (np.asarray(range_image, F32).reshape(-1)[:, None] * np.asarray(lut, F32).reshape(-1, 3)).astype(F32)
    valid = (pts[:, 0] + pts[:, 1]) + pts[:, 2] != 0
    return pts, valid


def _ranked(d, idx, k):
    """Sort candidates (rows) by (distance, index) and keep k."""
    order = np.lexsort((idx, d), axis=-1) if d.ndim == 1 else np.array([np.lexsort((i, x)) for x, i in zip(d, idx)])
    d = np.take_along_axis(d, order, -1)[..., :k]
    idx = np.take_along_axis(idx, order, -1)[..., :k]
    return d, idx


def knn_sets(range_image, lut, knn, radius, brute=None):
    """Neighbourhoods of every point -> (idx (HW, knn) int64 flat pixel indices, -1 padded; count (HW,) int)."""
    pts, valid = cloud(range_image, lut)
    HW = pts.shape[0]
    vid = np.flatnonzero(valid)
    vpts = pts[vid]
    rad2 = F32(F32(radius) * F32(radius))
    idx = np.full((HW, knn), -1, np.int64)
    cnt = np.zeros(HW, np.int64)
    if vid.size == 0:
        return idx, cnt
    brute = vid.size <= 20000 if brute is None else brute

    def exact(i):
        d = cham_d(pts[i], vpts)
        keep = d <= rad2
        dd, ii = _ranked(d[keep], vid[keep], knn)
        idx[i, :ii.size] = ii
        cnt[i] = ii.size

    if brute:
        for i in vid:
            exact(i)
        return idx, cnt
    from scipy.spatial import cKDTree
    tree = cKDTree(vpts.astype(F64))
    kc = min(knn + 8, vid.size)
    D, J = tree.query(vpts.astype(F64), k=kc)
    D, J = D.reshape(vid.size, kc), J.reshape(vid.size, kc)
    cand = vid[J]
    d = cham_d(vpts[:, None, :], pts[cand])
    order = np.lexsort((cand, d), axis=-1)
    d = np.take_along_axis(d, order, -1)
    cand = np.take_along_axis(cand, order, -1)
    within = d <= rad2
    m = np.minimum(within.sum(1), knn)
    kth = np.where(m >= knn, d[:, knn - 1] if kc >= knn else np.inf, rad2).astype(F64)
    # every point outside the candidates is at least D[:, -1] away in f64; the f32 distance is within 1e-6 of it
    clear = (kc == vid.size) | (kth * (1 + 1e-5) < D[:, -1] ** 2 * (1 - 1e-5))
    for r in range(vid.size):
        i = vid[r]
        if not clear[r]:
            exact(i)
            continue
        sel = cand[r][within[r]][:knn]
        idx[i, :sel.size] = sel
        cnt[i] = sel.size
    return idx, cnt


def normals(range_image, lut, knn=16, radius=1.0, brute=None):
    """-> dict(normals (HW,3) f64, 0 where there is no normal; has (HW,) bool; lam (HW,3) f64 ascending eigenvalues (0
    where fewer than 3 neighbours); count (HW,) neighbourhood sizes)."""
    pts, valid = cloud(range_image, lut)
    idx, cnt = knn_sets(range_image, lut, knn, radius, brute)
    HW = pts.shape[0]
    out = np.zeros((HW, 3), F64)
    lam = np.zeros((HW, 3), F64)
    has = np.zeros(HW, bool)
    rows = np.flatnonzero(valid & (cnt >= 3))
    if rows.size:
        nb = pts[np.maximum(idx[rows], 0)].astype(F64)
        mask = (np.arange(knn)[None, :] < cnt[rows][:, None]).astype(F64)[..., None]
        n = cnt[rows].astype(F64)[:, None]
        mean = (nb * mask).sum(1) / n
        dev = (nb - mean[:, None, :]) * mask
        cov = np.einsum("nki,nkj->nij", dev, dev) / n[:, :, None]
        w, v = np.linalg.eigh(cov)
        lam[rows] = w
        ok = ~((w[:, 2] == 0) | (w[:, 1] - w[:, 0] <= 1e-6 * w[:, 2]))
        e = v[:, :, 0] / np.linalg.norm(v[:, :, 0], axis=1, keepdims=True)
        flip = (e * pts[rows].astype(F64)).sum(1) > 0
        e[flip] = -e[flip]
        out[rows[ok]] = e[ok]
        has[rows[ok]] = True
    return dict(normals=out, has=has, lam=lam, count=cnt)


def nearest(q_pts, q_valid, o_pts, o_valid, brute=None):
    """Nearest point of the other cloud for every valid query point -> (idx (HW,) int64, -1 if none; d (HW,) f32)."""
    HW = q_pts.shape[0]
    idx = np.full(HW, -1, np.int64)
    dist = np.full(HW, np.inf, F32)
    qv, ov = np.flatnonzero(q_valid), np.flatnonzero(o_valid)
    if qv.size == 0 or ov.size == 0:
        return idx, dist
    brute = ov.size <= 20000 if brute is None else brute

    def exact(i):
        d = cham_d(q_pts[i], o_pts[ov])
        j = int(np.argmin(d))                        # first minimum: smallest index among equals
        idx[i], dist[i] = ov[j], d[j]

    if brute:
        for i in qv:
            exact(i)
        return idx, dist
    from scipy.spatial import cKDTree
    tree = cKDTree(o_pts[ov].astype(F64))
    kc = min(4, ov.size)
    D, J = tree.query(q_pts[qv].astype(F64), k=kc)
    D, J = D.reshape(qv.size, kc), J.reshape(qv.size, kc)
    cand = ov[J]
    d = cham_d(q_pts[qv][:, None, :], o_pts[cand])
    order = np.lexsort((cand, d), axis=-1)
    d0 = np.take_along_axis(d, order, -1)[:, 0]
    c0 = np.take_along_axis(cand, order, -1)[:, 0]
    clear = (kc == ov.size) | (d0.astype(F64) * (1 + 1e-5) < D[:, -1] ** 2 * (1 - 1e-5))
    idx[qv], dist[qv] = c0, d0
    for r in np.flatnonzero(~clear):
        exact(qv[r])
    return idx, dist


def p2plane(range_ref, range_rec, lut, normals_ref, normals_rec, brute=None):
    """The 7 columns of rpcc_p2plane_batch for one pair, given both clouds' normals ((HW,3), f32 as the device stores
    them; (0,0,0) = no normal).  Column 6 (whole-image scans of the device search) is returned as 0."""
    pa, va = cloud(range_ref, lut)
    pb, vb = cloud(range_rec, lut)
    na = np.asarray(normals_ref, F32).reshape(-1, 3)
    nb = np.asarray(normals_rec, F32).reshape(-1, 3)
    out = np.zeros(7, F64)
    for col, (q, qv, o, ov, no) in enumerate(((pa, va, pb, vb, nb), (pb, vb, pa, va, na))):
        j, d = nearest(q, qv, o, ov, brute)
        sel = np.flatnonzero(qv)
        out[3 * col] = sel.size
        if sel.size == 0:
            continue
        jj = j[sel]
        if (jj < 0).any():
            out[3 * col + 1] = np.inf
            continue
        n = no[jj].astype(F64)
        none = (n == 0).all(1)
        a, b = q[sel].astype(F64), o[jj].astype(F64)
        e = ((a[:, 0] - b[:, 0]) * n[:, 0] + (a[:, 1] - b[:, 1]) * n[:, 1]) + (a[:, 2] - b[:, 2]) * n[:, 2]
        err = np.where(none, d[sel].astype(F64), e * e)
        out[3 * col + 1] = err.sum()
        out[3 * col + 2] = none.sum()
    return out
