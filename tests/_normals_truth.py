"""An fp64 ground truth for NormalEstimation outputs and a checker that holds every row to it.

The truth does not restate PCL's algorithm: it takes the neighbour lists a search returned, builds a two-pass covariance
in float64 and solves it with LAPACK (`np.linalg.eigh`: eigenvalues l0 <= l1 <= l2, eigenvectors v0, v1, v2).  A normal
estimator is then judged row by row, with no percentile anywhere:

* NaN pattern: a row is NaN (all four fields) iff its query is not finite or it has fewer than 3 neighbours; the
  returned is_dense flag is true iff no row is NaN (normal_3d.hpp:62-69).
* unit length: | |n| - 1 | <= 1e-6.
* orientation, exactly: with v = vp - p in float32, ((vx*nx + vy*ny) + vz*nz) >= 0 in float32 -- the expression
  flipNormalTowardsViewpoint evaluates before it flips, so a correct estimator meets it bit for bit.
* direction: sin(n, v0) * g <= tau_n, g = (l1 - l0) / l2.  The error of any eigenvector solver grows like 1 / gap, so the
  product is what a solver can guarantee; it is ~0 when the normal is ill defined (l0 = l1) and any answer is right.
* curvature: | c - l0 / (l0 + l1 + l2) | <= tau_c.
* degenerate neighbourhoods, exactly: all neighbours identical (l2 = 0) -> n = +-(1, 0, 0) and c = 0 (eigen33's
  "all three equal" branch); neighbours that differ in one coordinate only (a line parallel to an axis, whose float
  covariance is exactly rank 1) -> n perpendicular to that axis to 1e-6 and c = 0.  A line in any other direction is not
  exactly collinear once its points are rounded to float, and the tiers below cover it.

tau_n and tau_c are tiered by the row's spectral gap g: PCL's fp32 closed-form cubic loses accuracy when the smallest
root has a close neighbour (near-isotropic rows, and nearly collinear ones where l0 ~ l1 ~ 0), and that is also where
the device's atan2f / cosf / sinf differ from the host's libm.  Rows with g < GAP_SPLIT get the looser bounds.  The
bounds leave >= 4x margin over the worst row of the CPU oracle (PCL's own algorithm) on every scene of `scenes()` for
k = 3 ... 100 and three radii; tests/test_normals_truth.py checks that margin and that the checker rejects a set of
plausible kernel mistakes.
"""
import numpy as np

GAP_SPLIT = 0.1          # g = (l1 - l0) / l2 at or above it: the tight tier
# (quantity, tier) -> bound.  Worst oracle rows on scenes() (k = 3 ... 100, three radii): direction 2.1e-5 / 2.7e-3,
# curvature 1.0e-5 / 4.9e-4 on the wide / narrow-gap rows.
TAU = {("direction", "wide"): 3e-4, ("direction", "narrow"): 1.2e-2,
       ("curvature", "wide"): 3e-4, ("curvature", "narrow"): 2e-3}
UNIT_TOL = 1e-6
COLLINEAR_TOL = 1e-6


def knn_to_csr(idx):
    """(nq, k) neighbour lists, -1 for a missing neighbour (only at the end of a row) -> (offsets, flat indices)."""
    idx = np.asarray(idx)
    ok = idx >= 0
    offs = np.zeros(idx.shape[0] + 1, dtype=np.int64)
    np.cumsum(ok.sum(1), out=offs[1:])
    return offs, idx[ok].astype(np.int64)


def truth(cloud, offs, nbr):
    """fp64 two-pass covariance of every neighbour list and its eigen-decomposition.
    Returns (count, lam (nq, 3) ascending, vec (nq, 3, 3) with the eigenvectors in columns, axes (nq, 3): the coordinates
    in which some neighbour differs from the first one); rows with < 3 neighbours hold NaN / False."""
    offs = np.asarray(offs, dtype=np.int64)
    nq = offs.size - 1
    cnt = np.diff(offs)
    lam = np.full((nq, 3), np.nan)
    vec = np.full((nq, 3, 3), np.nan)
    axes = np.zeros((nq, 3), bool)
    rows = np.nonzero(cnt >= 3)[0]
    if rows.size == 0:
        return cnt, lam, vec, axes
    # the neighbours of the rows that have >= 3 of them, in row order
    keep = np.repeat(cnt >= 3, cnt)
    p32 = np.asarray(cloud)[np.asarray(nbr)[keep], :3]
    starts = np.r_[0, np.cumsum(cnt[rows])[:-1]]
    axes[rows] = np.logical_or.reduceat(p32 != np.repeat(p32[starts], cnt[rows], axis=0), starts, axis=0)
    p = p32.astype(np.float64)
    c = cnt[rows].astype(np.float64)
    mean = np.add.reduceat(p, starts, axis=0) / c[:, None]
    d = p - np.repeat(mean, cnt[rows], axis=0)
    C = np.empty((rows.size, 3, 3))
    for a in range(3):
        for b in range(a, 3):
            C[:, a, b] = C[:, b, a] = np.add.reduceat(d[:, a] * d[:, b], starts) / c
    w, v = np.linalg.eigh(C)
    lam[rows], vec[rows] = w, v
    return cnt, lam, vec, axes


class Report:
    """What `check` found: `bad` maps a check's name to the rows that fail it, `worst` holds the largest error of each
    bounded quantity per tier and `ratio` the largest error / bound (< 0.25 means a 4x margin)."""

    def __init__(self):
        self.bad = {}
        self.worst = {}
        self.ratio = {}
        self.rows = 0

    @property
    def ok(self):
        return not any(len(v) for v in self.bad.values())

    def merge(self, other):
        for k, v in other.bad.items():
            self.bad[k] = np.r_[self.bad.get(k, np.zeros(0, np.int64)), v + self.rows]
        for d, o in ((self.worst, other.worst), (self.ratio, other.ratio)):
            for k, v in o.items():
                d[k] = max(d.get(k, 0.0), v)
        self.rows += other.rows
        return self

    def summary(self):
        bad = {k: (len(v), v[:5].tolist()) for k, v in self.bad.items() if len(v)}
        return dict(rows=self.rows, bad=bad, worst={k: float(f"{v:.3g}") for k, v in self.worst.items()},
                    ratio={k: float(f"{v:.3g}") for k, v in self.ratio.items()})


def _f32(a):
    return np.asarray(a, dtype=np.float32)


def check(cloud, queries, offs, nbr, viewpoint, out, dense_flag=None, tau=None):
    """Holds every row of `out` ((nq, >= 4): nx ny nz curvature) to the fp64 truth of the neighbour lists (offs, nbr)
    (indices into `cloud`); `queries` (nq, >= 3) are the points the normals belong to (the flip's p).  `tau` overrides
    entries of TAU."""
    tau = {**TAU, **(tau or {})}
    rep = Report()
    out = np.asarray(out)[:, :4]
    q = _f32(np.asarray(queries)[:, :3])
    nq = q.shape[0]
    rep.rows = nq
    cnt, lam, vec, axes = truth(cloud, offs, nbr)
    finite_q = np.isfinite(q).all(1)
    want_nan = (cnt < 3) | ~finite_q
    all_nan = np.isnan(out).all(1)
    all_fin = np.isfinite(out).all(1)
    bad = rep.bad
    bad["nan_pattern"] = np.nonzero((want_nan & ~all_nan) | (~want_nan & ~all_fin))[0]
    if dense_flag is not None:
        bad["is_dense_flag"] = np.zeros(0, np.int64) if bool(dense_flag) == (not want_nan.any()) else np.array([-1])
    r = np.nonzero(~want_nan & all_fin)[0]
    n32 = _f32(out[r, :3])
    n = n32.astype(np.float64)
    c = out[r, 3].astype(np.float64)
    nn = np.linalg.norm(n, axis=1)
    bad["unit_length"] = r[np.abs(nn - 1.0) > UNIT_TOL]
    rep.worst["unit_length"] = float(np.abs(nn - 1.0).max(initial=0.0))
    # the flip's own expression, in float32 (numpy does not contract to fma)
    v = _f32(viewpoint)[None, :] - q[r]
    dot = (v[:, 0] * n32[:, 0] + v[:, 1] * n32[:, 1]) + v[:, 2] * n32[:, 2]
    bad["orientation"] = r[~(dot >= np.float32(0))]
    L, V = lam[r], vec[r]
    l0, l1, l2 = L[:, 0], L[:, 1], L[:, 2]
    ident = l2 == 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        line = axes[r]
        colin = ~ident & (line.sum(1) == 1)
        nh = n / nn[:, None]
        sin = np.linalg.norm(np.cross(nh, V[:, :, 0]), axis=1)
        e_n = np.where(ident, 0.0, sin * (l1 - l0) / l2)
        e_c = np.where(ident, 0.0, np.abs(c - np.maximum(l0, 0.0) / (l0 + l1 + l2)))
        narrow = np.where(ident, 1.0, (l1 - l0) / l2) < GAP_SPLIT
    # eigen33's "all three equal" branch: (1, 0, 0), flipped by the viewpoint; curvature 0 (zero trace)
    bad["identical"] = r[ident & ~((np.abs(n32[:, 0]) == 1) & (n32[:, 1] == 0) & (n32[:, 2] == 0) & (c == 0))]
    bad["collinear"] = r[colin & ~((np.abs((nh * line).sum(1)) <= COLLINEAR_TOL) & (c == 0))]
    for name, e in (("direction", e_n), ("curvature", e_c)):
        for tier, m in (("wide", ~narrow), ("narrow", narrow)):
            key, t = f"{name}_{tier}", tau[(name, tier)]
            bad[key] = r[m & ~(e <= t)]
            w = float(e[m].max(initial=0.0))
            rep.worst[key] = w
            rep.ratio[key] = w / t
    rep.worst["rows_narrow_gap"] = int(narrow.sum())
    rep.worst["rows_identical"] = int(ident.sum())
    rep.worst["rows_collinear"] = int(colin.sum())
    return rep


def check_chunked(cloud, queries, offs, nbr, viewpoint, out, dense_flag=None, chunk=1_000_000):
    """`check` over row blocks of `chunk` rows (bounded memory at 10 M rows); the flag is checked on the whole."""
    offs = np.asarray(offs, dtype=np.int64)
    rep = Report()
    for b in range(0, offs.size - 1, chunk):
        e = min(b + chunk, offs.size - 1)
        o = offs[b:e + 1]
        rep.merge(check(cloud, np.asarray(queries)[b:e], o - o[0], np.asarray(nbr)[o[0]:o[-1]], viewpoint, out[b:e]))
    if dense_flag is not None:
        want = (np.diff(offs) >= 3) & np.isfinite(np.asarray(queries)[:, :3]).all(1)
        rep.bad["is_dense_flag"] = np.zeros(0, np.int64) if bool(dense_flag) == bool(want.all()) else np.array([-1])
    return rep


# ---------------------------------------------------------------------------------------------------------------------
# the scenes the checker is calibrated on (CPU oracle) and the device is held to
# ---------------------------------------------------------------------------------------------------------------------
class Scene:
    """cloud: float32 rows (4 or 12 floats: PointXYZ / PointNormal), the index holds `subset` of it (None: all),
    queries are cloud[indices] (None: the whole cloud)."""

    def __init__(self, name, xyz, viewpoint=(0.5, 0.5, 5.0), is_dense=True, subset=None, indices=None, width=4):
        self.name = name
        self.cloud = np.zeros((xyz.shape[0], width), np.float32)
        self.cloud[:, :3] = xyz
        self.cloud[:, 3] = 1.0
        self.viewpoint = tuple(float(v) for v in viewpoint)
        self.is_dense = is_dense
        self.subset = subset
        self.indices = indices

    @property
    def queries(self):
        return self.cloud if self.indices is None else self.cloud[self.indices]

    def __repr__(self):
        return self.name


def _sine(rng, n):
    p = rng.random((n, 3), dtype=np.float32)
    p[:, 2] = np.float32(0.1) * np.sin(np.float32(6) * p[:, 0])
    return p


def scenes(n=20000, seed=5):
    """Surfaces, planes, a line, identical points, shifted and rescaled copies, a volume, NaN holes, an index subset, the
    PointNormal stride and a viewpoint on the surface."""
    rng = np.random.default_rng(seed)
    s = _sine(rng, n)
    out = [Scene("sine", s)]
    # an exactly representable tilted plane z = 0.5 x + 0.25 y (dyadic x, y)
    xy = rng.integers(0, 4096, (n, 2)).astype(np.float32) / np.float32(2048)
    out.append(Scene("tilted_plane", np.c_[xy, np.float32(0.5) * xy[:, 0] + np.float32(0.25) * xy[:, 1]]))
    # axis-aligned plane: exact zeros in the covariance (eigen33's |c0| < FLT_EPSILON branch)
    out.append(Scene("axis_plane", np.c_[rng.random((n, 2), dtype=np.float32), np.full(n, 0.5, np.float32)]))
    # a line along z: exactly collinear neighbourhoods (eigen33's l0 = l1 branch)
    out.append(Scene("line_z", np.c_[np.full((n, 2), 0.3, np.float32), rng.random(n, dtype=np.float32)]))
    # 128 identical copies of each of n / 128 points: all-identical neighbourhoods for k <= 128
    base = rng.random((n // 128, 3), dtype=np.float32)
    out.append(Scene("identical_clusters", np.repeat(base, 128, axis=0)[rng.permutation(n // 128 * 128)]))
    out.append(Scene("sine_plus_1e3", s + np.float32(1e3), viewpoint=(1e3 + 0.5, 1e3 + 0.5, 1e3 + 5)))
    out.append(Scene("sine_plus_1e5", s + np.float32(1e5), viewpoint=(1e5 + 0.5, 1e5 + 0.5, 1e5 + 5)))
    out.append(Scene("sine_extent_1e-3", s * np.float32(1e-3), viewpoint=(5e-4, 5e-4, 5e-3)))
    out.append(Scene("sine_extent_1e3", s * np.float32(1e3), viewpoint=(500, 500, 5000)))
    out.append(Scene("volume", rng.random((n, 3), dtype=np.float32)))
    holes = s.copy()
    holes[::301, 1] = np.nan
    holes[7::503, 0] = np.inf
    out.append(Scene("nan_holes", holes, is_dense=False))
    sub = np.sort(rng.choice(n, n // 2, replace=False)).astype(np.int32)
    out.append(Scene("subset", s, subset=sub, indices=np.sort(rng.choice(n, n // 3, replace=False)).astype(np.int32)))
    out.append(Scene("point_normal_stride", s, width=12))
    # a viewpoint on the surface: rows whose flip sees dot = 0 exactly (the axis plane through the viewpoint)
    ap = out[2].cloud[:, :3]
    out.append(Scene("viewpoint_on_plane", ap, viewpoint=(0.25, 0.75, 0.5)))
    out.append(Scene("viewpoint_on_sine", s, viewpoint=tuple(s[0].tolist())))
    return out


def radii(scene, oracle_index, targets=(4, 20, 200), nthreads=8):
    """Radii whose balls hold about `targets` neighbours in `scene`: the median distance of neighbour t - 1 (half the
    smallest positive distance where that median is 0, i.e. among identical points)."""
    q = np.ascontiguousarray(scene.queries)
    _, d2, keff = oracle_index.knn(q, max(targets), nthreads=nthreads)
    fin = np.isfinite(q[:, :3]).all(1)
    out = []
    for t in targets:
        col = d2[fin, min(t, keff) - 1]
        r = float(np.sqrt(np.median(col)))
        if r == 0.0:
            r = 0.5 * float(np.sqrt(d2[fin][d2[fin] > 0].min()))
        out.append(r)
    return out


def truth_normals(cloud, queries, offs, nbr, viewpoint):
    """The truth as a normals array: v0 rounded to float32 and oriented by the flip's float32 rule, curvature
    l0 / (l0 + l1 + l2); NaN rows where the truth has fewer than 3 neighbours or the query is not finite."""
    cnt, lam, vec, _ = truth(cloud, offs, nbr)
    q = _f32(np.asarray(queries)[:, :3])
    n = vec[:, :, 0].astype(np.float32)
    v = _f32(viewpoint)[None, :] - q
    flip = ((v[:, 0] * n[:, 0] + v[:, 1] * n[:, 1]) + v[:, 2] * n[:, 2]) < 0
    n[flip] *= -1
    with np.errstate(divide="ignore", invalid="ignore"):
        c = np.where(lam[:, 2] > 0, np.maximum(lam[:, 0], 0.0) / lam.sum(1), 0.0)
    out = np.c_[n, c].astype(np.float32)
    out[(cnt < 3) | ~np.isfinite(q).all(1)] = np.nan
    return out
