"""The fp64 normals checker (tests/_normals_truth.py) on the CPU: PCL's own algorithm (the oracle) meets every bound on
every row with a 4x margin, and the checker rejects plausible kernel mistakes."""
import os

import numpy as np
import pytest

import _normals_truth as T

KS = (3, 5, 10, 12, 16, 20, 24, 32, 40, 64, 100)
NT = os.cpu_count() or 8
SCENES = T.scenes()


def _oracle_knn_case(orc, sc, k):
    oidx = orc.Index(sc.cloud, subset=sc.subset)
    q = np.ascontiguousarray(sc.queries)
    li, _, _ = oidx.knn(q, k, nthreads=NT)
    li[~np.isfinite(q[:, :3]).all(1)] = -1   # a non-finite query has no neighbours
    out, dense = oidx.normals_knn(sc.cloud, k, viewpoint=sc.viewpoint, indices=sc.indices, is_dense=sc.is_dense,
                                  nthreads=NT)
    offs, nbr = T.knn_to_csr(li)
    return q, li, offs, nbr, out, dense


@pytest.mark.parametrize("sc", SCENES, ids=[s.name for s in SCENES])
def test_oracle_meets_every_bound_with_margin(orc, sc):
    rep = T.Report()
    oidx = orc.Index(sc.cloud, subset=sc.subset)
    for k in KS:
        q, _, offs, nbr, out, dense = _oracle_knn_case(orc, sc, k)
        rep.merge(T.check(sc.cloud, q, offs, nbr, sc.viewpoint, out, dense))
    q = np.ascontiguousarray(sc.queries)
    for r in T.radii(sc, oidx, nthreads=NT):
        offs, nbr, _ = oidx.radius(q, r, nthreads=NT)
        out, dense = oidx.normals_radius(sc.cloud, r, viewpoint=sc.viewpoint, indices=sc.indices,
                                         is_dense=sc.is_dense, nthreads=NT)
        rep.merge(T.check(sc.cloud, q, offs, nbr, sc.viewpoint, out, dense))
    assert rep.ok, rep.summary()
    assert max(rep.ratio.values()) <= 0.25, rep.summary()


def test_degenerate_branches_are_exercised(orc):
    """The scenes reach eigen33's exact branches, so the checker's exact rules are not vacuous."""
    by = {s.name: s for s in SCENES}
    for name, key in (("identical_clusters", "rows_identical"), ("line_z", "rows_collinear")):
        sc = by[name]
        q, _, offs, nbr, out, dense = _oracle_knn_case(orc, sc, 16)
        rep = T.check(sc.cloud, q, offs, nbr, sc.viewpoint, out, dense)
        assert rep.ok and rep.worst[key] == q.shape[0], (name, rep.summary())
    sc = by["viewpoint_on_plane"]
    _, _, _, _, out, _ = _oracle_knn_case(orc, sc, 16)
    v = np.asarray(sc.viewpoint, np.float32) - sc.cloud[:, :3]
    assert np.any(((v[:, 0] * out[:, 0] + v[:, 1] * out[:, 1]) + v[:, 2] * out[:, 2]) == 0)


# ---------------------------------------------------------------------------------------------------------------------
# the checker has teeth
# ---------------------------------------------------------------------------------------------------------------------
def restated_normals(cloud, li, queries, viewpoint, use=None, divide_by=None, curvature_over_l2=False):
    """A numpy fp32 restatement of NormalEstimation over dense k-lists: PCL's shifted single-pass moments in list order,
    a float32 LAPACK eigensolve, curvature l0 / trace, the viewpoint flip.  `use` = neighbours per row to fold,
    `divide_by` = the count the moments are divided by, `curvature_over_l2` = l0 / l2 instead of l0 / trace."""
    k = li.shape[1] if use is None else use
    p = cloud[li[:, :k], :3].astype(np.float32)
    K = p[:, 0, :]
    acc = np.zeros((li.shape[0], 9), np.float32)
    for j in range(k):
        x = p[:, j, :] - K
        acc += np.stack([x[:, 0] * x[:, 0], x[:, 0] * x[:, 1], x[:, 0] * x[:, 2], x[:, 1] * x[:, 1],
                         x[:, 1] * x[:, 2], x[:, 2] * x[:, 2], x[:, 0], x[:, 1], x[:, 2]], 1)
    acc /= np.float32(k if divide_by is None else divide_by)
    m = acc[:, 6:]
    C = np.empty((li.shape[0], 3, 3), np.float32)
    C[:, 0, 0] = acc[:, 0] - m[:, 0] * m[:, 0]
    C[:, 0, 1] = C[:, 1, 0] = acc[:, 1] - m[:, 0] * m[:, 1]
    C[:, 0, 2] = C[:, 2, 0] = acc[:, 2] - m[:, 0] * m[:, 2]
    C[:, 1, 1] = acc[:, 3] - m[:, 1] * m[:, 1]
    C[:, 1, 2] = C[:, 2, 1] = acc[:, 4] - m[:, 1] * m[:, 2]
    C[:, 2, 2] = acc[:, 5] - m[:, 2] * m[:, 2]
    w, v = np.linalg.eigh(C)
    n = v[:, :, 0].astype(np.float32)
    den = w[:, 2] if curvature_over_l2 else (C[:, 0, 0] + C[:, 1, 1]) + C[:, 2, 2]
    curv = np.abs(w[:, 0] / den).astype(np.float32)
    vv = np.asarray(viewpoint, np.float32)[None, :] - queries[:, :3]
    flip = ((vv[:, 0] * n[:, 0] + vv[:, 1] * n[:, 1]) + vv[:, 2] * n[:, 2]) < 0
    n[flip] *= -1
    return np.c_[n, curv]


MUTATION_SCENES = ("sine", "volume", "tilted_plane")


def _mutation_cases(orc):
    by = {s.name: s for s in SCENES}
    for name in MUTATION_SCENES:
        for k in (5, 16, 40):
            sc = by[name]
            q, li, offs, nbr, out, dense = _oracle_knn_case(orc, sc, k)
            yield sc, k, q, li, offs, nbr, out


def _rejected(orc, mutate):
    """Runs `mutate` on every mutation case; returns the names of the checks that rejected a row."""
    fired = set()
    for sc, k, q, li, offs, nbr, out in _mutation_cases(orc):
        bad = mutate(sc, k, q, li, out)
        rep = T.check(sc.cloud, q, offs, nbr, sc.viewpoint, bad)
        fired |= {n for n, v in rep.bad.items() if len(v)}
    return fired


def test_restatement_control_passes(orc):
    """The unmutated restatement passes, so each rejection below is the mutation's doing."""
    assert not _rejected(orc, lambda sc, k, q, li, out: restated_normals(sc.cloud, li, q, sc.viewpoint))


# each mutation and the check that must catch it on the well-conditioned rows (or exactly)
MUTATIONS = {"first_k_minus_1": "direction_wide", "count_plus_1": "direction_wide", "count_minus_1": "direction_wide",
             "missing_flip": "orientation", "curvature_over_l2": "curvature_wide", "row_is_v1": "direction_wide"}


@pytest.mark.parametrize("mutation", sorted(MUTATIONS))
def test_checker_rejects_mutation(orc, mutation):
    def mutate(sc, k, q, li, out):
        if mutation == "first_k_minus_1":
            return restated_normals(sc.cloud, li, q, sc.viewpoint, use=k - 1)
        if mutation == "count_plus_1":
            return restated_normals(sc.cloud, li, q, sc.viewpoint, divide_by=k + 1)
        if mutation == "count_minus_1":
            return restated_normals(sc.cloud, li, q, sc.viewpoint, divide_by=k - 1)
        if mutation == "curvature_over_l2":
            return restated_normals(sc.cloud, li, q, sc.viewpoint, curvature_over_l2=True)
        bad = out.copy()
        v = np.asarray(sc.viewpoint, np.float32)[None, :] - q[:, :3]
        dot = (v[:, 0] * out[:, 0] + v[:, 1] * out[:, 1]) + v[:, 2] * out[:, 2]
        if mutation == "missing_flip":   # one row in 10^4 left on the wrong side
            rows = np.nonzero(dot > 0)[0][::10_000]
            bad[rows, :3] *= -1
            return bad
        # one well-conditioned row replaced by its middle eigenvector, oriented like a normal
        offs, nbr = T.knn_to_csr(li)
        _, lam, vec, _ = T.truth(sc.cloud, offs, nbr)
        i = int(np.nanargmax((lam[:, 1] - lam[:, 0]) / lam[:, 2]))
        v1 = vec[i, :, 1].astype(np.float32)
        bad[i, :3] = v1 if (v[i] * v1).sum() >= 0 else -v1
        return bad

    fired = _rejected(orc, mutate)
    assert MUTATIONS[mutation] in fired, (mutation, sorted(fired))
