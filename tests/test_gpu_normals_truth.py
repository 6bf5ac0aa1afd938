"""Every device normal, row by row, against the fp64 truth of tests/_normals_truth.py, on all five normals paths of
launch_normals / launch_normals_radius (search.cu):
  1. k_normals<K> per thread: k < 12, and any k <= 32 on an index without a cell table (< 256 points);
  2. k_knn_warp<true> for 12 <= k <= 32;
  3. k_normals<K> redoing the rows the warp kernel hands back (mixed density, queries off the cloud);
  4. launch_knn lists, then k_normals_from_lists, for k > 32;
  5. k_normals_from_csr for radius normals.
The truth is built on the device's own neighbour lists, and the same test asserts that those lists equal the oracle's.
Each test prints one JSON line with the worst direction (sin * gap) and curvature error per tier.  Needs a B200."""
import json
import os
import time

import numpy as np
import pytest

import _normals_truth as T

pytestmark = pytest.mark.gpu

NT = os.cpu_count() or 8
SCENES = T.scenes()


@pytest.fixture(scope="module")
def gpu():
    import pcl_b200
    pcl_b200.lib()
    ctx = pcl_b200.Context(0)
    yield pcl_b200, ctx
    ctx.close()


def _finish(path, rep, t0):
    s = rep.summary()
    print(json.dumps({"path": path, "seconds": round(time.time() - t0, 1), "rows": s["rows"], "worst": s["worst"]}))
    assert rep.ok, (path, s)


def _knn_case(gidx, oidx, cloud, q, k, viewpoint, indices=None, is_dense=True):
    """Device k-lists == oracle k-lists on every finite query; the device normals checked on the device lists."""
    q = np.ascontiguousarray(q)
    gi, gd, gk = gidx.knn(q, k)
    oi, od, ok = oidx.knn(q, k, nthreads=NT)
    fin = np.isfinite(q[:, :3]).all(1)
    assert gk == ok and np.array_equal(gi[fin], oi[fin]) and np.array_equal(gd[fin], od[fin]), k
    assert np.all(gi[~fin] == -1)
    out, dense = gidx.normals_knn(cloud, k, viewpoint=viewpoint, indices=indices, is_dense=is_dense)
    offs, nbr = T.knn_to_csr(gi)
    return T.check(cloud, q, offs, nbr, viewpoint, out, dense)


def _scenes_knn(P, ctx, orc, scenes, ks):
    rep = T.Report()
    for sc in scenes:
        gidx, oidx = P.Index(ctx, sc.cloud, subset=sc.subset), orc.Index(sc.cloud, subset=sc.subset)
        for k in ks:
            r = _knn_case(gidx, oidx, sc.cloud, sc.queries, k, sc.viewpoint, sc.indices, sc.is_dense)
            assert r.ok, (sc.name, k, r.summary())
            rep.merge(r)
        gidx.close()
    return rep


def test_path1_per_thread_small_k(gpu, orc):
    P, ctx = gpu
    t0 = time.time()
    rep = _scenes_knn(P, ctx, orc, SCENES, (3, 5, 8, 10))
    # an index of < 256 points has no cell table: k >= 12 runs the per-thread kernel too
    small = T.scenes(n=200, seed=9)
    assert all(s.cloud.shape[0] < 256 for s in small)
    rep.merge(_scenes_knn(P, ctx, orc, small, (12, 16, 32)))
    _finish("1 k_normals<K>", rep, t0)


def test_path2_warp_kernel(gpu, orc):
    P, ctx = gpu
    t0 = time.time()
    _finish("2 k_knn_warp<true>", _scenes_knn(P, ctx, orc, SCENES, (12, 16, 24, 32)), t0)


def test_path3_warp_kernel_redo_rows(gpu, orc):
    """The scene of test_knn_warp_kernel_mixed_density_every_query: a dense sheet inside a sparse volume, every point
    as a query plus queries off the cloud, so the warp kernel hands rows back to the per-thread kernel."""
    P, ctx = gpu
    t0 = time.time()
    rng = np.random.default_rng(77)
    n_sheet, n_vol = 340_000, 60_000
    sheet = rng.random((n_sheet, 3), dtype=np.float32) * np.float32(2.0)
    sheet[:, 2] = np.float32(0.3) * np.sin(np.float32(3) * sheet[:, 0]) * np.cos(np.float32(2) * sheet[:, 1]) + \
        np.float32(0.001) * rng.standard_normal(n_sheet).astype(np.float32)
    vol = (rng.random((n_vol, 3), dtype=np.float32) * np.float32(2.0))
    vol[:, 2] = vol[:, 2] - np.float32(1.0)
    pts = np.concatenate([sheet, vol])[rng.permutation(n_sheet + n_vol)]
    cloud = orc.to_xyz1(pts)
    off = orc.to_xyz1((rng.random((50_000, 3), dtype=np.float32) * np.float32(2.4) - np.float32(0.2)))
    q = np.concatenate([cloud, off])
    gidx, oidx = P.Index(ctx, cloud), orc.Index(cloud)
    rep = T.Report()
    for k in (12, 16, 24, 32):
        r = _knn_case(gidx, oidx, q, q, k, (1.0, 1.0, 5.0))
        assert r.ok, (k, r.summary())
        rep.merge(r)
    _finish("3 k_normals<K> redo", rep, t0)


def test_path4_lists_then_fold(gpu, orc):
    P, ctx = gpu
    t0 = time.time()
    _finish("4 k_normals_from_lists", _scenes_knn(P, ctx, orc, SCENES, (33, 40, 64, 100)), t0)


def test_path5_radius(gpu, orc):
    """Radii holding ~4, ~20 and ~200 neighbours per scene; device radius lists == oracle lists."""
    P, ctx = gpu
    t0 = time.time()
    rep = T.Report()
    for sc in SCENES:
        gidx, oidx = P.Index(ctx, sc.cloud, subset=sc.subset), orc.Index(sc.cloud, subset=sc.subset)
        q = np.ascontiguousarray(sc.queries)
        for r in T.radii(sc, oidx, nthreads=NT):
            goffs, gi, gd = gidx.radius(q, r)
            ooffs, oi, od = oidx.radius(q, r, nthreads=NT)
            assert np.array_equal(goffs, ooffs) and np.array_equal(gi, oi) and np.array_equal(gd, od), (sc.name, r)
            out, dense = gidx.normals_radius(sc.cloud, r, viewpoint=sc.viewpoint, indices=sc.indices,
                                             is_dense=sc.is_dense)
            one = T.check(sc.cloud, q, goffs, gi, sc.viewpoint, out, dense)
            assert one.ok, (sc.name, r, one.summary())
            rep.merge(one)
        gidx.close()
    _finish("5 k_normals_from_csr", rep, t0)


def test_bench_scale_every_row_k16(gpu, orc):
    """bench.py's target (10 M points), k = 16, viewpoint (5, 5, 10): every row against the fp64 truth of the device's
    lists, in 1 M-row chunks; the lists themselves against the oracle on a 100 k-row sample."""
    import bench
    P, ctx = gpu
    t0 = time.time()
    tgt = bench.make_target(10_000_000)
    idx = P.Index(ctx, tgt)
    vp = (5.0, 5.0, 10.0)
    out, dense = idx.normals_knn(tgt, 16, viewpoint=vp)
    gi, gd, gk = idx.knn(tgt, 16)
    assert gk == 16
    sample = np.sort(np.random.default_rng(3).choice(tgt.shape[0], 100_000, replace=False))
    oi, od, _ = orc.Index(tgt).knn(np.ascontiguousarray(tgt[sample]), 16, nthreads=NT)
    assert np.array_equal(gi[sample], oi) and np.array_equal(gd[sample], od)
    del gd
    offs = np.arange(0, 16 * tgt.shape[0] + 1, 16, dtype=np.int64)
    rep = T.check_chunked(tgt, tgt, offs, gi.reshape(-1), vp, out, dense)
    _finish("2 k_knn_warp<true> at 10 M", rep, t0)


def test_icp_point_to_plane_each_side_own_normals(gpu, orc):
    """test_icp_point_to_plane_vs_oracle's registration, but each side with its OWN k = 16 normals.  The tolerance
    comes from the CPU: the oracle ICP with its own normals and with the fp64-truth normals rounded to float differ by
    d; the device with its own normals may differ from the oracle by 4 d more than it does when both sides use the
    oracle's normals (the registration path alone, which test_icp_point_to_plane_vs_oracle holds to 1e-5)."""
    P, ctx = gpu
    n = 40000

    def surf(m, seed):
        r = np.random.default_rng(seed)
        xy = r.random((m, 2)) * 10
        z = 0.5 * np.sin(xy[:, 0]) * np.cos(0.7 * xy[:, 1]) + r.normal(0, 0.002, m)
        return np.column_stack([xy, z])

    a = np.deg2rad(2.0)
    R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
    tgt = np.zeros((n, 12), np.float32)
    tgt[:, :3], tgt[:, 3] = surf(n, 7).astype(np.float32), 1
    src = np.zeros((n, 12), np.float32)
    src[:, :3], src[:, 3] = (surf(n, 8) @ R.T + np.array([0.02, 0.01, -0.01])).astype(np.float32), 1
    vp = (5, 5, 10)
    kw = dict(max_iterations=30, max_correspondence_distance=0.05)
    oidx = orc.Index(tgt)
    on, _ = oidx.normals_knn(tgt, 16, viewpoint=vp, nthreads=NT)
    li, _, _ = oidx.knn(tgt, 16, nthreads=NT)
    offs, nbr = T.knn_to_csr(li)
    tn = T.truth_normals(tgt, tgt, offs, nbr, vp)
    t_own, t_truth = tgt.copy(), tgt.copy()
    t_own[:, 4:8], t_truth[:, 4:8] = on, tn
    o = orc.icp_align(src, t_own, estimator=1, with_normals_transform=True, nthreads=NT, **kw)
    o_truth = orc.icp_align(src, t_truth, estimator=1, with_normals_transform=True, nthreads=NT, **kw)
    tol = 4 * float(np.linalg.norm(o["final"] - o_truth["final"]))
    assert o["iterations"] == o_truth["iterations"]
    tidx = P.Index(ctx, tgt)
    gn, _ = tidx.normals_knn(tgt, 16, viewpoint=vp)
    t_dev = tgt.copy()
    t_dev[:, 4:8] = gn
    r = P.icp_align(ctx, src, tidx, tgt_normals=P.Field(t_dev, 4), estimator=P.EST_POINT_TO_PLANE_LLS,
                    with_normals_transform=1, **kw)
    err = float(np.linalg.norm(r["final"] - o["final"]))
    r_same = P.icp_align(ctx, src, tidx, tgt_normals=P.Field(t_own, 4), estimator=P.EST_POINT_TO_PLANE_LLS,
                         with_normals_transform=1, **kw)
    err_same = float(np.linalg.norm(r_same["final"] - o["final"]))
    print(json.dumps({"icp_own_normals": {"err": err, "err_same_normals": err_same, "tol": tol,
                                          "iterations": r["iterations"]}}))
    assert r["iterations"] == o["iterations"] and r["state"] == o["state"], (r, o)
    assert err <= err_same + tol, (err, err_same, tol)
