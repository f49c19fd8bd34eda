"""GPU parity tests: the CUDA path (through the C ABI, via ctypes) against the CPU oracle on the same
seeded inputs.  Bars (BASELINE.json north_star): neighbour index sets and correspondence lists
bit-exact; descriptors within 1e-4 L2 per descriptor; poses within 1e-4 m and 0.01 degrees.
"""
import numpy as np

import eps
import pytest

pytestmark = pytest.mark.gpu


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


@pytest.fixture(scope="module")
def ctx(b200):
    c = b200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small(synth):
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 40000, scene_id=1)
    return model, scene


def _rot_angle_deg(Ra, Rb):
    # chord form ||Ra - Rb||_F = 2 sqrt(2) sin(angle / 2): unlike arccos((trace - 1) / 2) it is well
    # conditioned near zero (float32 matrices are orthonormal only to ~1e-7)
    return np.degrees(2 * np.arcsin(min(1.0, np.linalg.norm(Ra - Rb) / (2 * np.sqrt(2)))))


# ------------------------------------------------------------------------------------------ search
def test_radius_search_bit_exact(ctx, orc, small):
    model, scene = small
    q = scene[::17]
    for cloud_np, r in ((scene, 0.02), (model, 0.015)):
        qq = q if cloud_np is scene else model[::5]
        cl = ctx.cloud(cloud_np)
        off, idx, d2 = ctx.radius_search(cl, qq, r)
        ooff, oidx, od2 = orc.radius_search(cloud_np, qq, r)
        assert np.array_equal(off, ooff)
        assert np.array_equal(idx, oidx)
        assert np.array_equal(d2, od2)
        cl.close()


def test_radius_search_degenerate(ctx, orc, synth):
    # radius 50 on a small model: the support is the whole cloud (SHOT_demo.cpp:498)
    model = synth.make_model("diagonal", 3000)
    cl = ctx.cloud(model)
    q = model[::300]
    off, idx, d2 = ctx.radius_search(cl, q, 50.0)
    ooff, oidx, od2 = orc.radius_search(model, q, 50.0)
    assert off[-1] == len(q) * 3000
    assert np.array_equal(off, ooff) and np.array_equal(idx, oidx) and np.array_equal(d2, od2)
    # NaN rows in the surface are skipped but keep their index; NaN / far queries return nothing
    s = model.copy()
    s[10] = np.nan
    s[500, 1] = np.inf
    cl2 = ctx.cloud(s)
    q2 = np.concatenate([s[:50], [[np.nan, 0, 0]], [[9, 9, 9]]]).astype(np.float32)
    off, idx, d2 = ctx.radius_search(cl2, q2, 0.03)
    ooff, oidx, od2 = orc.radius_search(s, q2, 0.03)
    assert np.array_equal(off, ooff) and np.array_equal(idx, oidx) and np.array_equal(d2, od2)
    assert off[-1] == off[-3]
    # empty query set
    off, idx, d2 = ctx.radius_search(cl2, np.zeros((0, 3), np.float32), 0.03)
    assert off.tolist() == [0] and len(idx) == 0


@pytest.mark.parametrize("k", [1, 10, 50])
def test_knn_search_parity(ctx, orc, small, k):
    _, scene = small
    cl = ctx.cloud(scene)
    q = scene[::23]
    idx, d2, kf = ctx.knn_search(cl, q, k)
    oidx, od2, okf = orc.knn_search(scene, q, k)
    assert kf == okf == k
    assert np.array_equal(d2, od2)
    assert np.array_equal(idx, oidx)
    # queries that are not surface points, including one far outside the bounding box
    q2 = (q[:200] + np.float32(0.003)).astype(np.float32)
    q2[0] = [5, -4, 3]
    idx, d2, _ = ctx.knn_search(cl, q2, k)
    oidx, od2, _ = orc.knn_search(scene, q2, k)
    assert np.array_equal(d2, od2) and np.array_equal(idx, oidx)


def test_knn_clamps(ctx, orc):
    s = _rng(1).normal(size=(7, 3)).astype(np.float32)
    cl = ctx.cloud(s)
    idx, d2, kf = ctx.knn_search(cl, s, 10)
    oidx, od2, okf = orc.knn_search(s, s, 10)
    assert kf == okf == 7
    assert np.array_equal(idx, oidx) and np.array_equal(d2, od2)


def test_radius_search_warp_kernel_equals_cta_kernel(ctx, synth):
    """radiusSearch lists: the one-query-per-warp fill kernel (up to 512 neighbours, longer lists handed to the CTA
    kernel) writes the same CSR — indices and squared distances — as the CTA kernel."""
    import os
    scene = synth.make_scene(("y",), 80000, scene_id=12)
    q = scene[::13].copy()
    q[3] = np.nan
    cl = ctx.cloud(scene)
    sizes = []
    for r in (0.01, 0.03, 0.08):
        a = ctx.radius_search(cl, q, r)
        os.environ["B200_RADIUS_FILL"] = "cta"
        try:
            b = ctx.radius_search(cl, q, r)
        finally:
            os.environ.pop("B200_RADIUS_FILL", None)
        for x, y in zip(a, b):
            assert x.tobytes() == y.tobytes(), r
        sizes.append(int(np.diff(a[0]).max()))
    assert min(sizes) <= 512 < max(sizes), sizes
    cl.close()


# ------------------------------------------------------------------------------------------ normals
@pytest.mark.parametrize("k", [10, 20, 50])
def test_normals_knn_parity(ctx, orc, small, k):
    model, scene = small
    for cloud_np in (model, scene):
        cl = ctx.cloud(cloud_np)
        got = ctx.normals(cl, k=k)
        ref = orc.normals(cloud_np, k=k)
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        err = np.abs(got - ref)
        assert np.nanmedian(err[:, :3]) < 1e-6
        # float32 covariance sums are bit-identical; only the libm calls in eigen33 differ by an ulp: every row
        # whose eigenvector is stable under a 2-ulp perturbation of theta agrees to 1e-5, the ill-conditioned
        # rest differs by no more than that perturbation explains (tests/eps.py)
        st = eps.normals_check(orc, got, cloud_np, k=k, label="normals k=%d" % k)
        print("normals k=%d: %s" % (k, st))


def test_normals_knn_lattice_nan_pattern(ctx, orc):
    """An exact planar lattice (many ties at the k-th distance, degenerate covariances): the rows without a normal are
    the reference's."""
    g = np.arange(40, dtype=np.float32) * 0.01
    lattice = np.stack(np.meshgrid(g, g, np.zeros(1, np.float32), indexing="ij"), -1).reshape(-1, 3)
    ref = orc.normals(lattice, k=20)
    got = ctx.normals(ctx.cloud(lattice), k=20)
    assert np.array_equal(np.isnan(got), np.isnan(ref))


def test_normals_radius_and_nan(ctx, orc, synth):
    scene = synth.make_scene(("horizontal",), 20000, scene_id=2)
    kp = synth.voxel_grid(scene, 0.03)
    cl = ctx.cloud(kp)
    got = ctx.normals(cl, radius=0.15)          # FPFH_demo.cpp:416-420: normals on the keypoints
    eps.normals_check(orc, got, kp, radius=0.15, label="normals r=0.15")
    s = scene[:5000].copy()
    s[7] = np.nan
    cl2 = ctx.cloud(s)
    got = ctx.normals(cl2, k=10)
    assert np.all(np.isnan(got[7]))
    eps.normals_check(orc, got, s, k=10, label="normals with a NaN row")
    # explicit query cloud (input != surface) and a non-default viewpoint
    q = s[100:400]
    got = ctx.normals(cl2, q=q, k=15, viewpoint=(0.5, 0.5, 3.0))
    eps.normals_check(orc, got, s, k=15, q=q, viewpoint=(0.5, 0.5, 3.0), label="normals, explicit queries")
    # Feature::initCompute: k and radius are exclusive
    with pytest.raises(Exception):
        ctx.normals(cl2, k=10, radius=0.1)
    with pytest.raises(Exception):
        ctx.normals(cl2, k=0, radius=0.0)


def test_normals_radius_warp_kernel_equals_cta_kernel(ctx, orc, synth):
    """Radius normals: the one-query-per-warp kernel (neighbourhoods of up to 256 points; the three shared-memory
    sizes 64 / 128 / 256 and the hand-over of larger neighbourhoods to the CTA kernel) gives the CTA kernel's
    result bit for bit — both run PCL's nine sums in (d2, index) order — and both stand against the restatement."""
    import os
    scene = synth.make_scene(("y",), 60000, scene_id=4)
    s = scene[:30000].copy()
    s[11] = np.nan
    kp = synth.voxel_grid(scene, 0.01)
    cases = [(kp, 0.02, None), (kp, 0.05, None), (kp, 0.08, None), (s, 0.03, None), (s, 0.12, None), (s, 0.05, s[200:900])]
    seen_max = []
    for cloud_np, r, q in cases:
        cl = ctx.cloud(cloud_np)
        os.environ.pop("B200_NORMALS_RADIUS", None)
        got = ctx.normals(cl, q=q, radius=r)
        seen_max.append(ctx.neighbor_stats()[1])
        os.environ["B200_NORMALS_RADIUS"] = "cta"
        try:
            ref = ctx.normals(cl, q=q, radius=r)
        finally:
            os.environ.pop("B200_NORMALS_RADIUS", None)
        assert got.tobytes() == ref.tobytes(), (len(cloud_np), r)
        cl.close()
    print("largest neighbourhoods of the cases:", seen_max)
    # the cases cross the size classes of the warp kernel and the hand-over to the CTA kernel
    assert min(seen_max) <= 128 and any(128 < m <= 256 for m in seen_max) and max(seen_max) > 256, seen_max
    cl = ctx.cloud(kp)
    eps.normals_check(orc, ctx.normals(cl, radius=0.05), kp, radius=0.05, label="normals r=0.05 (warp kernel)")
    cl.close()


# ------------------------------------------------------------------------------------------ SHOT
def _desc_check(got, ref, tol=1e-4):
    assert np.array_equal(np.isnan(got[:, 0]), np.isnan(ref[:, 0]))
    ok = ~np.isnan(ref[:, 0])
    err = np.linalg.norm(got[ok].astype(np.float64) - ref[ok].astype(np.float64), axis=1)
    return err


def test_shot_parity(ctx, orc, synth, small):
    model, scene = small
    for cloud_np, kp, r in ((model, synth.voxel_grid(model, 0.02), 0.02),
                            (scene, synth.voxel_grid(scene, 0.03), 0.02),
                            (scene, synth.uniform_sampling(scene, 0.04), 0.035)):
        nrm = orc.normals(cloud_np, k=10)
        cl = ctx.cloud(cloud_np)
        lrf = ctx.shot_lrf(cl, kp, r)
        olrf = orc.shot_lrf(cloud_np, kp, r)
        assert np.array_equal(np.isnan(lrf), np.isnan(olrf))
        assert np.nanmax(np.abs(lrf - olrf)) < 1e-5
        desc, rf = ctx.shot352(cl, nrm, kp, r)
        odesc, orf = orc.shot352(cloud_np, nrm, kp, r)
        err = _desc_check(desc, odesc)
        assert err.max() < 1e-4, err.max()
        assert np.array_equal(np.isnan(rf), np.isnan(orf))
        assert np.nanmax(np.abs(rf - orf)) < 1e-5
        ok = ~np.isnan(desc[:, 0])
        np.testing.assert_allclose(np.linalg.norm(desc[ok], axis=1), 1.0, atol=1e-5)


def test_shot_whole_model_support(ctx, orc, synth):
    # SHOT_demo.cpp:497-502: model descriptors with radius 50 (every point is a neighbour)
    model = synth.make_model("y", 6000)
    kp = synth.voxel_grid(model, 0.04)
    nrm = orc.normals(model, k=20)
    cl = ctx.cloud(model)
    desc, rf = ctx.shot352(cl, nrm, kp, 50.0)
    odesc, orf = orc.shot352(model, nrm, kp, 50.0)
    err = _desc_check(desc, odesc)
    assert err.max() < 1e-4, err.max()


def test_shot_nan_rows(ctx, orc):
    s = _rng(9).uniform(-1, 1, (300, 3)).astype(np.float32)
    nrm = orc.normals(s, k=5)
    nrm[5] = np.nan                                  # a NaN normal is skipped, not fatal
    kp = np.concatenate([s[:20], [[10, 10, 10]], [[np.nan, 0, 0]]]).astype(np.float32)
    cl = ctx.cloud(s)
    desc, rf = ctx.shot352(cl, nrm, kp, 0.4)
    odesc, orf = orc.shot352(s, nrm, kp, 0.4)
    assert np.array_equal(np.isnan(desc), np.isnan(odesc))
    assert np.all(np.isnan(desc[-2:])) and np.all(np.isnan(rf[-2:]))
    ok = ~np.isnan(odesc[:, 0])
    assert np.linalg.norm(desc[ok] - odesc[ok], axis=1).max() < 1e-4
    d0, _ = ctx.shot352(cl, nrm, np.zeros((0, 3), np.float32), 0.4)
    assert d0.shape == (0, 352)


# ------------------------------------------------------------------------------------------ FPFH
def test_fpfh_parity(ctx, orc, synth, small):
    model, scene = small
    for cloud_np, leaf, r in ((model, 0.01, 0.05), (scene, 0.03, 0.15)):
        kp = synth.voxel_grid(cloud_np, leaf)
        nrm = orc.normals(kp, radius=r)
        cl = ctx.cloud(kp)
        got = ctx.fpfh33(cl, nrm, r)
        ref = orc.fpfh33(kp, nrm, r)
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref[:, 0])
        # ABSOLUTE 1e-4 L2 per descriptor (north star) on every row no atan2f bin-border case can reach; the
        # border rows differ by at most what their border cases move (tests/eps.py)
        st = eps.fpfh_check(orc, got, kp, nrm, r, label="fpfh r=%g" % r)
        print("fpfh r=%g: %s" % (r, st))
        np.testing.assert_allclose(got[ok].reshape(-1, 3, 11).sum(2), 100.0, atol=2e-3)
        # explicit query set (input != surface)
        got_q = ctx.fpfh33(cl, nrm, r, q=kp[::9])
        ref_q = orc.fpfh33(kp, nrm, r, q=kp[::9])
        eps.fpfh_check(orc, got_q, kp, nrm, r, q=kp[::9], label="fpfh queries r=%g" % r)


def test_fpfh_warp_kernels_equal_cta_kernels(ctx, orc, synth):
    """FPFH: the one-point-per-warp kernels (neighbourhoods of up to 256 points, larger ones handed to the CTA kernels)
    give the CTA kernels' descriptors bit for bit, with input == surface (rows written at the original index, a NaN row
    for a point that is not in the grid) and with an explicit query set."""
    import os
    scene = synth.make_scene(("diagonal",), 50000, scene_id=6)
    seen = []
    for leaf, r in ((0.01, 0.03), (0.01, 0.06), (0.008, 0.13)):
        kp = synth.voxel_grid(scene, leaf)[:20000].copy()
        kp[5] = np.nan
        nrm = orc.normals(kp, radius=r)
        cl = ctx.cloud(kp)
        res = {}
        for mode in ("warp", "cta"):
            if mode == "cta":
                os.environ["B200_FPFH"] = "cta"
            try:
                res[mode] = (ctx.fpfh33(cl, nrm, r), ctx.fpfh33(cl, nrm, r, q=kp[3::7]))
            finally:
                os.environ.pop("B200_FPFH", None)
        seen.append(ctx.neighbor_stats()[1])
        assert np.all(np.isnan(res["warp"][0][5]))
        assert res["warp"][0].tobytes() == res["cta"][0].tobytes(), (leaf, r)
        assert res["warp"][1].tobytes() == res["cta"][1].tobytes(), (leaf, r)
        cl.close()
    print("largest neighbourhoods:", seen)
    assert min(seen) <= 256 < max(seen), seen


# ------------------------------------------------------------------------------------------ matching
def test_match_bit_exact(ctx, orc):
    rng = _rng(11)
    for D, Km, Ks in ((352, 700, 1500), (33, 257, 999), (352, 1, 10)):
        a = rng.uniform(0, 1, (Km, D)).astype(np.float32)
        a /= np.linalg.norm(a, axis=1, keepdims=True)
        b = a[rng.integers(0, Km, Ks)] + rng.normal(0, 0.03, (Ks, D)).astype(np.float32)
        b[3, 0] = np.nan
        if Km > 5:
            a[4, D - 1] = np.inf
            b[5] = a[2]                   # exact duplicate → distance 0
        for mode, thr in ((1, 0.25), (1, 0.05), (2, 0.0)):
            got = ctx.match(a, b, mode, thr)
            ref = orc.match(a, b, mode, thr)
            assert np.array_equal(got["index_query"], ref["index_query"])
            assert np.array_equal(got["index_match"], ref["index_match"])
            assert np.array_equal(got["distance"], ref["distance"])
    assert len(ctx.match(np.zeros((0, 352), np.float32), np.ones((5, 352), np.float32))) == 0
    assert len(ctx.match(np.ones((5, 352), np.float32), np.zeros((0, 352), np.float32))) == 0


def test_match_real_descriptors(ctx, orc, synth, small):
    model, scene = small
    kpm, kps = synth.voxel_grid(model, 0.02), synth.voxel_grid(scene, 0.03)
    dm, _ = orc.shot352(model, orc.normals(model, k=10), kpm, 0.02)
    ds, _ = orc.shot352(scene, orc.normals(scene, k=10), kps, 0.02)
    for mode in (1, 2):
        got = ctx.match(dm, ds, mode, 0.25)
        ref = orc.match(dm, ds, mode, 0.25)
        assert len(ref) > 0
        assert got.tobytes() == ref.tobytes()


# ------------------------------------------------------------------------------------------ grouping
def _gc_case(seed, n_model=80, n_in=60, n_out=50):
    from scipy.spatial.transform import Rotation
    rng = _rng(seed)
    R = Rotation.random(random_state=seed).as_matrix()
    t = rng.uniform(-1, 1, 3)
    model = rng.uniform(-0.3, 0.3, (n_model, 3)).astype(np.float32)
    scene_in = (model.astype(np.float64) @ R.T + t + rng.normal(0, 0.0005, (n_model, 3))).astype(np.float32)
    clutter = rng.uniform(-2, 2, (100, 3)).astype(np.float32)
    scene = np.concatenate([scene_in, clutter])
    return rng, R, t, model, scene


def test_gc_parity(ctx, orc, b200):
    for seed in (21, 22, 23):
        rng, R, t, model, scene = _gc_case(seed)
        C = 110
        corrs = np.zeros(C, dtype=b200.CORR_DTYPE)
        corrs["index_query"][:60] = rng.permutation(80)[:60]
        corrs["index_match"][:60] = corrs["index_query"][:60]
        corrs["index_query"][60:] = rng.integers(0, 80, C - 60)      # outliers, duplicate model indices
        corrs["index_match"][60:] = rng.integers(80, 180, C - 60)
        corrs["distance"] = rng.uniform(0, 0.2, C).astype(np.float32)
        corrs["distance"][5] = corrs["distance"][6]                    # a distance tie
        corrs = corrs[rng.permutation(C)]
        for thr in (2, 5):
            T, inst, n = ctx.gc_recognize(model, scene, corrs, 0.01, thr)
            oT, oinst = orc.gc_recognize(model, scene, corrs, 0.01, thr)
            assert n == len(oT)
            assert [len(i) for i in inst] == [len(i) for i in oinst]
            for a, b in zip(inst, oinst):
                assert a.tobytes() == b.tobytes()
            for A, B in zip(T, oT):
                assert np.abs(A[:3, 3] - B[:3, 3]).max() < 1e-4
                assert _rot_angle_deg(A[:3, :3].astype(np.float64), B[:3, :3].astype(np.float64)) < 0.01
            b = int(np.argmax([len(i) for i in inst]))
            assert np.abs(T[b][:3, 3] - t).max() < 5e-3
    # empty / tiny inputs
    T, inst, n = ctx.gc_recognize(model, scene, corrs[:0], 0.01, 2)
    assert n == 0
    T, inst, n = ctx.gc_recognize(model, scene, corrs[:2], 0.01, 2)
    assert n == 0


def test_gc_many_small_instances(ctx, orc, synth, small, b200):
    # gc_threshold = 2 on noisy descriptor matches yields hundreds of 3-4 element instances
    model, scene = small
    kpm, kps = synth.voxel_grid(model, 0.02), synth.voxel_grid(scene, 0.03)
    dm, _ = orc.shot352(model, orc.normals(model, k=10), kpm, 0.02)
    ds, _ = orc.shot352(scene, orc.normals(scene, k=10), kps, 0.02)
    corrs = orc.match(dm, ds, 1, 0.25)
    assert len(corrs) > 100
    T, inst, n = ctx.gc_recognize(kpm, kps, corrs, 0.02, 2, max_inst=2048)
    oT, oinst = orc.gc_recognize(kpm, kps, corrs, 0.02, 2, max_inst=2048)
    assert n == len(oT) and n > 0
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    dT = max(np.abs(A - B).max() for A, B in zip(T, oT))
    assert dT < 1e-4


def test_gc_large_instances(ctx, orc, b200):
    """Sets far larger than the grouping kernel's shared-memory member cache (64) and candidate lists longer than
    its per-seed list (1024): two rigid instances with 1500 / 700 inliers plus outliers."""
    from scipy.spatial.transform import Rotation
    rng = _rng(77)
    model = rng.uniform(-0.3, 0.3, (2500, 3)).astype(np.float32)
    parts, corr_parts = [], []
    base = 0
    for seed, n_in in ((1, 1500), (2, 700)):
        R = Rotation.random(random_state=seed).as_matrix()
        t = rng.uniform(-1, 1, 3) + 3 * seed
        sel = rng.permutation(2500)[:n_in]
        pts = (model[sel].astype(np.float64) @ R.T + t + rng.normal(0, 0.0005, (n_in, 3))).astype(np.float32)
        parts.append(pts)
        c = np.zeros(n_in, dtype=b200.CORR_DTYPE)
        c["index_query"], c["index_match"] = sel, base + np.arange(n_in)
        corr_parts.append(c)
        base += n_in
    clutter = rng.uniform(-2, 8, (600, 3)).astype(np.float32)
    parts.append(clutter)
    c = np.zeros(600, dtype=b200.CORR_DTYPE)
    c["index_query"], c["index_match"] = rng.integers(0, 2500, 600), base + np.arange(600)
    corr_parts.append(c)
    scene = np.concatenate(parts)
    corrs = np.concatenate(corr_parts)
    corrs["distance"] = rng.uniform(0, 0.25, len(corrs)).astype(np.float32)
    corrs = corrs[rng.permutation(len(corrs))]
    T, inst, n = ctx.gc_recognize(model, scene, corrs, 0.01, 3, max_inst=256)
    oT, oinst = orc.gc_recognize(model, scene, corrs, 0.01, 3, max_inst=256)
    assert n == len(oT) and n >= 2
    assert max(len(i) for i in inst) > 1024
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    for A, B in zip(T, oT):
        assert np.abs(A[:3, 3] - B[:3, 3]).max() < 1e-4
        assert _rot_angle_deg(A[:3, :3].astype(np.float64), B[:3, :3].astype(np.float64)) < 0.01


def _rigid_instances_case(b200, sizes, n_model, n_clutter, seed):
    from scipy.spatial.transform import Rotation
    rng = _rng(seed)
    model = rng.uniform(-0.3, 0.3, (n_model, 3)).astype(np.float32)
    parts, corr_parts = [], []
    base = 0
    for k, n_in in enumerate(sizes):
        R = Rotation.random(random_state=seed + k).as_matrix()
        t = rng.uniform(-1, 1, 3) + 3 * (k + 1)
        sel = rng.permutation(n_model)[:n_in]
        pts = (model[sel].astype(np.float64) @ R.T + t + rng.normal(0, 0.0005, (n_in, 3))).astype(np.float32)
        parts.append(pts)
        c = np.zeros(n_in, dtype=b200.CORR_DTYPE)
        c["index_query"], c["index_match"] = sel, base + np.arange(n_in)
        corr_parts.append(c)
        base += n_in
    parts.append(rng.uniform(-2, 3 * len(sizes) + 2, (n_clutter, 3)).astype(np.float32))
    c = np.zeros(n_clutter, dtype=b200.CORR_DTYPE)
    c["index_query"], c["index_match"] = rng.integers(0, n_model, n_clutter), base + np.arange(n_clutter)
    corr_parts.append(c)
    corrs = np.concatenate(corr_parts)
    corrs["distance"] = rng.uniform(0, 0.25, len(corrs)).astype(np.float32)
    return model, np.concatenate(parts), corrs[rng.permutation(len(corrs))]


def test_gc_grouping_and_order_match_restatement(ctx, orc, synth, small, b200, monkeypatch):
    """Grouping (the cluster kernel) returns the sequential algorithm's instance lists byte for byte, and so does every
    way of putting the correspondences in (distance, position) order."""
    cases = []
    # (a) two large sets, far beyond the 64 members kept in shared memory, in clutter
    cases.append(_rigid_instances_case(b200, (2600, 900), 4000, 800, 5) + (0.01, 3, 256))
    # (b) sets far beyond 64 members
    cases.append(_rigid_instances_case(b200, (1900, 40, 300), 2500, 1500, 6) + (0.01, 3, 512))
    # (c) hundreds of 3-4 element instances on noisy descriptor matches (threshold 2), failed seeds in between
    model, scene = small
    kpm, kps = synth.voxel_grid(model, 0.02), synth.voxel_grid(scene, 0.03)
    dm, _ = orc.shot352(model, orc.normals(model, k=10), kpm, 0.02)
    ds, _ = orc.shot352(scene, orc.normals(scene, k=10), kps, 0.02)
    cases.append((kpm, kps, orc.match(dm, ds, 1, 0.25), 0.02, 2, 2048))
    for m, sc, corrs, size, thr, max_inst in cases:
        oT, oinst = orc.gc_recognize(m, sc, corrs, size, thr, max_inst=max_inst)
        assert len(oT) > 0
        T, inst, n = ctx.gc_recognize(m, sc, corrs, size, thr, max_inst=max_inst)
        assert n == len(oT), (n, len(oT))
        assert [len(i) for i in inst] == [len(i) for i in oinst]
        for a, b in zip(inst, oinst):
            assert a.tobytes() == b.tobytes()
    # the (distance, position) order: bucket sort (default), its hand-over to the counting kernel when a bucket is too
    # large (here: 3 000 equal distances), and the counting kernel alone
    m, sc, corrs, size, thr, max_inst = cases[1]
    tied = corrs.copy()
    tied["distance"][:3000] = np.float32(0.125)
    for c in (corrs, tied):
        oT, oinst = orc.gc_recognize(m, sc, c, size, thr, max_inst=max_inst)
        for sel in (None, "count"):
            if sel is None:
                monkeypatch.delenv("B200_GC_SORT", raising=False)
            else:
                monkeypatch.setenv("B200_GC_SORT", sel)
            T, inst, n = ctx.gc_recognize(m, sc, c, size, thr, max_inst=max_inst)
            assert n == len(oT), (sel, n, len(oT))
            for a, b in zip(inst, oinst):
                assert a.tobytes() == b.tobytes(), sel
    monkeypatch.delenv("B200_GC_SORT", raising=False)


def test_gc_ransac_rare_good_samples(ctx, orc, b200):
    """Instances in which almost every 3-sample is rejected by isSampleGood (many scene points matched to one model
    point): RANSAC redraws hundreds of times, past the first 624 outputs of the mt19937 stream.  One instance
    has no good sample at all (identity transform, unfiltered correspondences)."""
    from scipy.spatial.transform import Rotation
    rng = _rng(91)
    model = np.array([[0, 0, 0], [0.3, 0, 0], [0, 0.25, 0.1], [2, 2, 2], [2.2, 2, 2]], np.float32)
    R = Rotation.random(random_state=3).as_matrix()
    base = (model.astype(np.float64) @ R.T + [0.5, -0.2, 1.0]).astype(np.float32)
    scene, corr = [], []

    def add(mi, pt, d):
        corr.append((mi, len(scene), d))
        scene.append(pt)
    add(0, base[0], 0.01)
    add(1, base[1], 0.02)
    for i in range(38):                                  # 38 scene points matched to model point 2
        add(2, base[2] + rng.uniform(-0.002, 0.002, 3).astype(np.float32), 0.03 + 0.001 * i)
    for i in range(5):                                   # second instance: every member shares model point 3
        add(3, base[3] + np.float32([1, 0, 0]) + rng.uniform(-0.002, 0.002, 3).astype(np.float32), 0.1 + 0.001 * i)
    scene = np.array(scene, np.float32)
    corrs = np.zeros(len(corr), dtype=b200.CORR_DTYPE)
    corrs["index_query"] = [c[0] for c in corr]
    corrs["index_match"] = [c[1] for c in corr]
    corrs["distance"] = np.array([c[2] for c in corr], np.float32)
    T, inst, n = ctx.gc_recognize(model, scene, corrs, 0.01, 2, max_inst=16)
    oT, oinst = orc.gc_recognize(model, scene, corrs, 0.01, 2, max_inst=16)
    assert n == len(oT) == 2
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    assert max(np.abs(A - B).max() for A, B in zip(T, oT)) < 1e-4
    assert np.array_equal(T[1], np.eye(4, dtype=np.float32)) and len(inst[1]) == 5
    assert np.abs(T[0][:3, :3] - R).max() < 0.05


# ------------------------------------------------------------------------------------------ pipeline
def test_register_scene_pipeline(ctx, orc, synth, b200):
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 60000, scene_id=0)
    kpm, kps = synth.voxel_grid(model, 0.02), synth.voxel_grid(scene, 0.03)
    p = b200.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                         max_instances=2048)
    m = ctx.model_create_shot(model, kpm, p)
    dm, kk = m.download()
    odm, _ = orc.shot352(model, orc.normals(model, k=10), kpm, 0.02)
    assert np.array_equal(kk, kpm)
    assert _desc_check(dm, odm).max() < 1e-4
    res = ctx.register_scene_shot(m, scene, kps, p)
    ods, _ = orc.shot352(scene, orc.normals(scene, k=10), kps, 0.02)
    # oracle chain on the oracle's own descriptors; correspondence lists must agree except where a
    # descriptor distance sits within 1e-5 of the threshold / of the runner-up
    oc = orc.match(odm, ods, 1, 0.25)
    gc_ = res["corrs"]
    # every differing entry must sit within the descriptor tolerance of the threshold or of a runner-up tie
    st = eps.corr_check(odm, ods, gc_, oc, 0.25, label="pipeline correspondences")
    print("pipeline correspondences: %s" % st)
    # grouping parity on identical correspondences
    T, inst, n = ctx.gc_recognize(kpm, kps, gc_, 0.02, 2, max_inst=2048)
    assert n == res["n_instances"]
    for a, b in zip(inst, res["instances"]):
        assert a.tobytes() == b.tobytes()
    oT, oinst = orc.gc_recognize(kpm, kps, gc_, 0.02, 2, max_inst=2048)
    assert n == len(oT)
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    assert max(np.abs(A - B).max() for A, B in zip(res["transforms"], oT)) < 1e-4
    assert ctx.launches > 0
    m.close()


# ------------------------------------------------------------------------------------------ descriptor index
def test_desc_index_knn_bit_exact(ctx, orc):
    """KdTreeFLANN<SHOT352>::setInputCloud + nearestKSearch per query (SHOT.cpp:405-417, SHOT_demo.cpp:508-521):
    distances are FLANN's sequential float32 L2_Simple sums, order (distance, index)."""
    rng = _rng(41)
    for D, Km, nq in ((352, 300, 40), (33, 500, 64)):
        a = rng.uniform(0, 1, (Km, D)).astype(np.float32)
        q = (a[rng.integers(0, Km, nq)] + rng.normal(0, 0.05, (nq, D))).astype(np.float32)
        a[7, 3] = np.nan                     # dropped from the index, position kept
        a[11] = a[10]                        # duplicate rows: tie broken by index
        q[0] = a[10]
        ix = ctx.desc_index(a)
        assert ix.size == Km - 1
        valid = np.isfinite(a).all(1)
        diff = (q[:, None, :] - a[None, :, :]).astype(np.float32)
        d2_all = np.cumsum(diff * diff, axis=2, dtype=np.float32)[:, :, -1]     # sequential float32 sum
        d2_all[:, ~valid] = np.inf
        for k in (1, 2, 5, 16):
            idx, d2, kf = ix.knn(q, k)
            assert kf == k
            order = np.lexsort((np.broadcast_to(np.arange(Km), d2_all.shape), d2_all), axis=1)[:, :k]
            assert np.array_equal(idx, order.astype(np.int32))
            assert np.array_equal(d2, np.take_along_axis(d2_all, order, 1))
        # k = 1 / 2 agree with the correspondence oracle (same arg-min, same distance)
        ref = orc.match(a, q, 1, 1e30)
        idx, d2, _ = ix.knn(q, 1)
        assert np.array_equal(ref["index_query"], idx[:, 0]) and np.array_equal(ref["distance"], d2[:, 0])
        ix.close()
    small = ctx.desc_index(rng.uniform(0, 1, (3, 33)).astype(np.float32))
    idx, d2, kf = small.knn(rng.uniform(0, 1, (2, 33)).astype(np.float32), 5)
    assert kf == 3 and np.all(idx[:, 3:] == -1) and np.all(np.isinf(d2[:, 3:]))
    small.close()


# ------------------------------------------------------------------------------------------ keypoints
def test_keypoint_extraction_parity(ctx, orc, synth, b200):
    """UniformSampling (SHOT.cpp:314-323): same points and rows, bit for bit.  VoxelGrid (SHOT_demo.cpp:413-417):
    same voxels in the same order, centroids to 1 ulp (float64 sums whose order is not fixed on the device)."""
    for cloud, leaf in ((synth.make_model("y", 20000), 0.005), (synth.make_scene(("y",), 80000, scene_id=9), 0.01),
                        (synth.make_scene(("horizontal",), 30000, scene_id=2), 0.03)):
        cloud = cloud.copy()
        cloud[5] = np.nan
        us, idx = ctx.uniform_sampling(cloud, leaf, return_index=True)
        ous, oidx = orc.uniform_sampling(cloud, leaf, return_index=True)
        assert np.array_equal(idx, oidx) and np.array_equal(us, ous)
        vg = ctx.voxel_grid(cloud, leaf)
        ovg = orc.voxel_grid(cloud, leaf)
        assert vg.shape == ovg.shape
        assert np.abs(vg - ovg).max() <= 2.4e-7 * max(1.0, np.abs(ovg).max())
    vg = ctx.voxel_grid(cloud, (0.03, 0.05, 0.02))
    assert vg.shape == orc.voxel_grid(cloud, (0.03, 0.05, 0.02)).shape
    assert len(ctx.uniform_sampling(np.zeros((0, 3), np.float32), 0.01)) == 0
    with pytest.raises(b200.B200Error):
        ctx.uniform_sampling(cloud, 1e-5)


# ------------------------------------------------------------------------------------------ multi-view library
def test_multiview_library_registration(ctx, orc, synth, b200):
    """BASELINE.json config 4 (scaled down): a descriptor library over partial views of the three CAD joints
    (CAD_desc.cpp:231-370) and one scene matched against every view (the per-view loop of SHOT.cpp:243-483), the
    scene's normals and descriptors computed once.  Per view the result must equal the single-model pipeline
    and, on the same correspondences, the oracle's grouping."""
    p = b200.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                         max_instances=512)
    scene = synth.make_scene(("y", "horizontal"), 50000, scene_id=4)
    kps = synth.uniform_sampling(scene, 0.03)
    lib = b200.Library(ctx)
    views = []
    for joint in ("y", "diagonal", "horizontal"):
        for v in (3, 20, 41):
            cloud = synth.make_partial_view(joint, v, 6000)
            kp = synth.uniform_sampling(cloud, 0.02)
            assert lib.add_view(cloud, kp, p) == len(views)
            views.append((cloud, kp))
    assert lib.views == 9 and lib.view_size(4) == len(views[4][1])
    res = lib.register_scene(scene, kps, p, max_inst=4096)
    assert res["n_instances"] == len(res["view"]) == len(res["instances"])
    assert np.all(np.diff(res["view"]) >= 0)
    total = 0
    for v, (cloud, kp) in enumerate(views):
        m = ctx.model_create_shot(cloud, kp, p)
        single = ctx.register_scene_shot(m, scene, kps, p)
        mine = [i for i in range(res["n_instances"]) if res["view"][i] == v]
        assert len(mine) == single["n_instances"] and res["view_n_corrs"][v] == len(single["corrs"])
        for i, ins in zip(mine, single["instances"]):
            assert res["instances"][i].tobytes() == ins.tobytes()
        if mine:
            assert np.array_equal(res["transforms"][mine], single["transforms"])
        # oracle grouping on the view's correspondences
        oT, oinst = orc.gc_recognize(kp, kps, single["corrs"], 0.02, 2, max_inst=512)
        assert len(oT) == len(mine)
        for i, oi in zip(mine, oinst):
            assert res["instances"][i].tobytes() == oi.tobytes()
        # the library's descriptors are the single-model ones
        dl, kl = lib.download_view(v)
        dm, km = m.download()
        assert np.array_equal(dl, dm, equal_nan=True) and np.array_equal(kl, km)
        total += len(mine)
        m.close()
    assert total == res["n_instances"] and total > 0
    lib.close()


def test_scene_batch_sharding(ctx, orc, synth, b200, pkg):
    """BASELINE.json config 5 (scaled down): a batch of scenes registered against one model; on one rank the
    sharded driver must return every scene's correspondences, identical to direct calls."""
    import importlib
    sharding = importlib.import_module(pkg.__name__ + ".sharding")
    p = b200.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                         max_instances=512)
    model = synth.make_model("y", 5000)
    m = ctx.model_create_shot(model, synth.uniform_sampling(model, 0.02), p)
    scenes = [synth.make_scene(("y",), 20000 + 3000 * s, scene_id=20 + s) for s in range(3)]
    kps = [synth.uniform_sampling(s, 0.03) for s in scenes]
    local, gathered = sharding.register_scene_batch(ctx, m, scenes, kps, p)
    assert sorted(local) == sorted(gathered) == [0, 1, 2]
    for s in range(3):
        direct = ctx.register_scene_shot(m, scenes[s], kps[s], p)
        assert gathered[s].tobytes() == direct["corrs"].tobytes()
        assert local[s]["n_instances"] == direct["n_instances"]
    m.close()


# ------------------------------------------------------------------------------------------ Hough grouping
def test_hough3d_parity(ctx, orc, synth, small):
    """Hough3DGrouping (the reference's default grouping, SHOT.cpp:433-470) with SHOT reference frames: same
    instances in the same order, voters bit-exact, poses within 1e-4, against the restatement."""
    model, scene = small
    kpm, kps = synth.uniform_sampling(model, 0.02), synth.uniform_sampling(scene, 0.03)
    dm, mrf = orc.shot352(model, orc.normals(model, k=10), kpm, 0.02)
    ds, srf = orc.shot352(scene, orc.normals(scene, k=10), kps, 0.02)
    corrs = orc.match(dm, ds, 1, 0.25)
    assert len(corrs) > 100
    for bin_size, thr in ((0.02, 2.0), (0.03, 3.0), (0.05, -0.5)):
        T, inst, n = ctx.hough3d_recognize(kpm, mrf, kps, srf, corrs, bin_size, thr, max_inst=4096)
        oT, oinst = orc.hough3d_recognize(kpm, mrf, kps, srf, corrs, bin_size, thr, max_inst=4096)
        assert n == len(oT) and (n > 0 or thr > 2)
        for a, b in zip(inst, oinst):
            assert a.tobytes() == b.tobytes()
        if n:
            assert max(np.abs(A - B).max() for A, B in zip(T, oT)) < 1e-4
    # NaN frames are skipped, empty input gives nothing
    srf2 = srf.copy()
    srf2[corrs["index_match"][:5]] = np.nan
    T, inst, n = ctx.hough3d_recognize(kpm, mrf, kps, srf2, corrs, 0.03, 2.0, max_inst=4096)
    oT, oinst = orc.hough3d_recognize(kpm, mrf, kps, srf2, corrs, 0.03, 2.0, max_inst=4096)
    assert n == len(oT)
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    assert ctx.hough3d_recognize(kpm, mrf, kps, srf, corrs[:0], 0.03, 2.0)[2] == 0


# ------------------------------------------------------------------------------------------ ICP
def test_icp_parity(ctx, orc, synth, small):
    """IterativeClosestPoint::align / getFitnessScore (SHOT.cpp:177-192: the model placed by a grouped pose is
    refined against the scene).  Same iteration counts and convergence flags as the restatement, final transforms
    within 1e-4 m / 0.01 degrees, fitness within 1e-4 relative (the rigid fit is float64 on both sides; the
    nearest-neighbour sets are exact, so the iterates agree to float32 rounding)."""
    from scipy.spatial.transform import Rotation
    model, scene = small
    _, poses = synth.make_scene(("y",), 40000, scene_id=1, return_poses=True)
    Tgt = np.asarray(poses[0], dtype=np.float64)
    # perturb the true pose the way a grouped pose is off: ~1 degree, a few millimetres
    dR = Rotation.from_rotvec([0.012, -0.015, 0.01]).as_matrix()
    G = Tgt.copy()
    G[:3, :3] = dR @ Tgt[:3, :3]
    G[:3, 3] = dR @ Tgt[:3, 3] + [0.003, -0.002, 0.002]
    placed = (model.astype(np.float64) @ G[:3, :3].T + G[:3, 3]).astype(np.float32)
    tgt = ctx.cloud(scene)
    for iters in (1, 5, 30):
        a = ctx.icp_align(placed, tgt, max_iterations=iters)
        b = orc.icp_align(placed, scene, max_iterations=iters)
        assert a["iterations"] == b["iterations"] and a["converged"] == b["converged"]
        assert np.abs(a["final_transform"][:3, 3] - b["final_transform"][:3, 3]).max() < 1e-4
        assert _rot_angle_deg(a["final_transform"][:3, :3], b["final_transform"][:3, :3]) < 0.01
        assert abs(a["fitness"] - b["fitness"]) <= 1e-4 * b["fitness"]
        assert np.abs(a["aligned"] - b["aligned"]).max() < 2e-4
    # refinement reduces the error of the perturbed pose
    err0 = np.abs(placed - (model.astype(np.float64) @ Tgt[:3, :3].T + Tgt[:3, 3])).max()
    err1 = np.abs(a["aligned"] - (model.astype(np.float64) @ Tgt[:3, :3].T + Tgt[:3, 3])).max()
    assert err1 < err0
    # guess = the pose itself, source = the untransformed model (what the adapters' align(output, guess) does)
    a = ctx.icp_align(model, tgt, max_iterations=5, guess=G.astype(np.float32))
    b = orc.icp_align(model, scene, max_iterations=5, guess=G.astype(np.float32))
    assert a["iterations"] == b["iterations"] == 5
    assert np.abs(a["final_transform"] - b["final_transform"]).max() < 1e-4
    # distance gate: only pairs within 5 mm are used; a gate nothing passes ends unconverged with the guess
    a = ctx.icp_align(placed, tgt, max_iterations=5, max_corr_dist=0.005)
    b = orc.icp_align(placed, scene, max_iterations=5, max_corr_dist=0.005)
    assert a["iterations"] == b["iterations"]
    assert np.abs(a["final_transform"] - b["final_transform"]).max() < 1e-4
    far = ctx.icp_align(placed + 10.0, tgt, max_iterations=5, max_corr_dist=0.01)
    assert not far["converged"] and far["iterations"] == 0 and np.array_equal(far["final_transform"], np.eye(4))
    # NaN source rows are ignored and stay NaN in the aligned cloud; an empty source is a no-op
    p2 = placed.copy()
    p2[7] = np.nan
    a = ctx.icp_align(p2, tgt, max_iterations=3)
    b = orc.icp_align(p2, scene, max_iterations=3)
    assert np.isnan(a["aligned"][7]).all() and np.abs(a["final_transform"] - b["final_transform"]).max() < 1e-4
    e = ctx.icp_align(np.zeros((0, 3), np.float32), tgt, max_iterations=3)
    assert e["iterations"] == 0 and np.array_equal(e["final_transform"], np.eye(4))
    tgt.close()


# ------------------------------------------------------------------------------------------ BOARD
def test_board_lrf_parity(ctx, orc, synth, small, b200):
    """BOARDLocalReferenceFrameEstimation (SHOT.cpp:441-453: find_holes, keypoints on the full cloud).  Same NaN rows;
    frames within 1e-5 of the restatement on every keypoint whose frame does not change when the support directions'
    angles are perturbed by 2 ulp (acosf differs in the last bit between the device and glibc, and an angle within
    an ulp of a sector border then lands in the other sector) — the border cases are identified, not counted.  The
    rand() stream continues across calls (model, then scene) like PCL's two compute() calls."""
    model, scene = small
    kpm, kps = synth.uniform_sampling(model, 0.02), synth.uniform_sampling(scene, 0.03)
    nm, ns = orc.normals(model, k=10), orc.normals(scene, k=10)
    cm, cs = ctx.cloud(model), ctx.cloud(scene)

    def compare(a, b, variants):
        """variants: the restatement's frames under the +2 ulp / -2 ulp angle perturbation."""
        assert np.array_equal(np.isnan(a), np.isnan(b))
        ok = ~np.isnan(b[:, 0])
        stable = ok.copy()
        for v in variants:
            stable &= np.nan_to_num(np.abs(v - b)).max(axis=1) <= 5e-6   # continuous effect of 2 ulp on the angles: ~3e-6
        assert stable.sum() >= 0.98 * ok.sum(), (int(stable.sum()), int(ok.sum()))
        err = np.abs(a - b).max(axis=1)
        assert err[stable].max() <= 1e-5, float(err[stable].max())
        print("BOARD: %d frames, %d stable under the 2-ulp angle perturbation (max err %.2e), %d border cases of which "
              "%d differ" % (ok.sum(), stable.sum(), err[stable].max(), (ok & ~stable).sum(),
                             (err[ok & ~stable] > 1e-5).sum()))
        f = a[ok].reshape(-1, 3, 3)
        assert np.abs(np.einsum("nij,nkj->nik", f, f) - np.eye(3)).max() < 1e-4

    def oracle_variants(cloud, nrm, kp, r, **kw):
        out = []
        for name in ("board_angle_up", "board_angle_down"):
            with orc.variant(name):
                out.append(orc.board_lrf(cloud, nrm, kp, r, **kw)[0])
        return out

    ctx.srand(1)
    a_m = ctx.board_lrf(cm, nm, kpm, 0.015)
    a_s = ctx.board_lrf(cs, ns, kps, 0.015)
    o_m, used = orc.board_lrf(model, nm, kpm, 0.015)
    o_s, used2 = orc.board_lrf(scene, ns, kps, 0.015, rand_skip=used)
    assert used > 0 and used2 > 0
    compare(a_m, o_m, oracle_variants(model, nm, kpm, 0.015))
    compare(a_s, o_s, oracle_variants(scene, ns, kps, 0.015, rand_skip=used))
    # reseeding reproduces the first call
    ctx.srand(1)
    assert np.array_equal(ctx.board_lrf(cm, nm, kpm, 0.015), a_m, equal_nan=True)
    # parameter variants: no hole search; ring between 0.85 r and r (tangent radius = support radius); 12 sectors
    for kw in (dict(find_holes=False), dict(tangent_radius=0.02), dict(check_margin_array_size=12, steep_thresh=0.0)):
        r = 0.02
        ctx.srand(7)
        a = ctx.board_lrf(cs, ns, kps, r, b200.board_params(**kw))
        o, _ = orc.board_lrf(scene, ns, kps, r, orc.board_params(**kw), rand_seed=7)
        compare(a, o, oracle_variants(scene, ns, kps, r, params=orc.board_params(**kw), rand_seed=7))
    # NaN normals and a far keypoint
    ns2 = ns.copy()
    ns2[::7] = np.nan
    kp2 = np.concatenate([kps[:200], [[9.0, 9.0, 9.0]]]).astype(np.float32)
    ctx.srand(3)
    a = ctx.board_lrf(cs, ns2, kp2, 0.02)
    o, _ = orc.board_lrf(scene, ns2, kp2, 0.02, rand_seed=3)
    assert np.isnan(a[-1]).all()
    compare(a, o, oracle_variants(scene, ns2, kp2, 0.02, rand_seed=3))
    cm.close()
    cs.close()


def test_board_warp_kernel_equals_cta_kernel(ctx, orc, synth, b200):
    """BOARD frames: the one-keypoint-per-warp kernel (supports of up to 512 points, larger ones handed to the CTA
    kernel) against the CTA kernel on the same rand() stream.  Both run the same float32 sequence after the z axis; the
    float64 plane-fit sums are grouped differently (32 partials instead of 128), so a frame may differ in the last
    bits: 1e-6 is the bar, and nearly every frame is identical."""
    import os
    scene = synth.make_scene(("y",), 120000, scene_id=9)
    kp = synth.uniform_sampling(scene, 0.03)
    nrm = orc.normals(scene, k=10)
    cl = ctx.cloud(scene)
    seen = []
    for r, kw in ((0.01, {}), (0.02, {}), (0.07, {}), (0.02, dict(find_holes=False)), (0.02, dict(check_margin_array_size=40))):
        res = {}
        for mode in ("warp", "cta"):
            ctx.srand(5)
            if mode == "cta":
                os.environ["B200_BOARD"] = "cta"
            try:
                res[mode] = ctx.board_lrf(cl, nrm, kp, r, b200.board_params(**kw))
            finally:
                os.environ.pop("B200_BOARD", None)
        off = ctx.radius_search(cl, kp, r)[0]
        seen.append(int(np.diff(off).max()))
        a, b = res["warp"], res["cta"]
        assert np.array_equal(np.isnan(a), np.isnan(b))
        ok = ~np.isnan(b[:, 0])
        same = (a[ok] == b[ok]).all(axis=1).mean()
        assert np.abs(a[ok] - b[ok]).max() < 1e-6 and same > 0.999, (r, kw, float(np.abs(a[ok] - b[ok]).max()), same)
    print("largest supports:", seen)
    assert min(seen) <= 512 < max(seen), seen
    cl.close()


# ------------------------------------------------------------------------------------------ library file
def test_library_file_roundtrip(ctx, orc, synth, b200, tmp_path):
    """The binary descriptor library (replaces the reference's Partial_View<l>.txt dumps, CAD_desc.cpp:354-370): save →
    load in a second context → identical descriptors, keypoints, pose table and registration results; a view built
    from the reference's text format equals the original to the 6 digits the text keeps; damaged files are refused."""
    p = b200.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                         max_instances=512)
    scene = synth.make_scene(("y",), 40000, scene_id=1)
    kps = synth.uniform_sampling(scene, 0.03)
    lib = b200.Library(ctx)
    for joint, v in (("y", 3), ("y", 20), ("diagonal", 7)):
        cloud = synth.make_partial_view(joint, v, 5000)
        lib.add_view(cloud, synth.uniform_sampling(cloud, 0.02), p)
    pose = np.eye(4, dtype=np.float32)
    pose[:3, 3] = [0.1, -0.2, 0.3]
    lib.set_view_pose(1, pose)
    path = str(tmp_path / "joints.b200lib")
    lib.save(path)
    raw = open(path, "rb").read()
    assert raw[:8] == b"B200LIB1" and np.frombuffer(raw[8:16], "<u4").tolist() == [3, 352]
    assert len(raw) == 16 + sum(4 + 64 + lib.view_size(v) * (3 + 352) * 4 for v in range(3)) + 8
    ctx2 = b200.Context(0)
    lib2 = b200.Library.load(ctx2, path)
    assert lib2.views == 3
    for v in range(3):
        d1, k1 = lib.download_view(v)
        d2, k2 = lib2.download_view(v)
        assert np.array_equal(d1, d2, equal_nan=True) and np.array_equal(k1, k2)
        assert np.array_equal(lib2.view_pose(v), pose if v == 1 else np.eye(4))
    r1 = lib.register_scene(scene, kps, p)
    r2 = lib2.register_scene(scene, kps, p)
    assert r1["n_instances"] == r2["n_instances"] > 0 and np.array_equal(r1["transforms"], r2["transforms"])
    assert all(a.tobytes() == b.tobytes() for a, b in zip(r1["instances"], r2["instances"]))
    # the reference's text dump: one float per line, 6 significant digits
    d0, k0 = lib.download_view(0)
    txt = str(tmp_path / "Partial_View0.txt")
    ok = ~np.isnan(d0[:, 0])
    b200.write_partial_view_text(txt, d0[ok])
    dt = b200.read_partial_view_text(txt)
    assert dt.shape == d0[ok].shape and np.abs(dt - d0[ok]).max() < 1e-5
    lib3 = b200.Library(ctx2)
    assert lib3.add_view_descriptors(dt, k0[ok]) == 0
    r3 = lib3.register_scene(scene, kps, p)
    n0 = int((r1["view"] == 0).sum())
    assert abs(r3["n_instances"] - n0) <= max(1, n0 // 10)
    # damaged files
    for name, data in (("trunc", raw[:len(raw) // 2]), ("magic", b"X" + raw[1:]),
                       ("flip", raw[:4000] + bytes([raw[4000] ^ 1]) + raw[4001:])):
        bad = str(tmp_path / (name + ".b200lib"))
        open(bad, "wb").write(data)
        with pytest.raises(b200.B200Error):
            b200.Library.load(ctx2, bad)
    with pytest.raises(b200.B200Error):
        b200.Library.load(ctx2, str(tmp_path / "missing.b200lib"))
    lib3.close()
    lib2.close()
    ctx2.close()
    lib.close()


# ------------------------------------------------------------------------------------------ cloud utilities
def test_remove_nan_and_transform_bit_exact(ctx, orc, synth):
    """removeNaNFromPointCloud (SHOT.cpp:298-299) and transformPointCloud with a 4x4 (model placed by a pose before
    ICP): bit-exact against the restatement, including non-finite rows, strided input and empty clouds."""
    from scipy.spatial.transform import Rotation
    rng = _rng(21)
    c = synth.make_scene(("y",), 20000, scene_id=2)
    c = np.concatenate([c, rng.uniform(0, 1, (len(c), 5)).astype(np.float32)], axis=1)   # stride 8, like PointXYZRGBA
    bad = rng.choice(len(c), 300, replace=False)
    c[bad[:100], 0] = np.nan
    c[bad[100:200], 1] = np.inf
    c[bad[200:], 2] = -np.inf
    kept, idx = ctx.remove_nan(c)
    okept, oidx = orc.remove_nan(c)
    assert np.array_equal(idx, oidx) and kept.tobytes() == okept.tobytes() and len(kept) == len(c) - 300
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = Rotation.from_rotvec([0.7, -0.4, 1.1]).as_matrix()
    T[:3, 3] = [0.31, -1.2, 0.77]
    a, b = ctx.transform_points(c, T), orc.transform_points(c, T)
    assert a.tobytes() == b.tobytes()
    assert len(ctx.remove_nan(np.zeros((0, 3), np.float32))[0]) == 0
    assert len(ctx.transform_points(np.zeros((0, 3), np.float32), T)) == 0


def test_resident_fpfh_pipeline(ctx, orc, synth, b200):
    """b200_model_create_fpfh + b200_register_scene_fpfh (FPFH_demo.cpp:405-538 with the model resident): equals the
    per-call API bit for bit; normals and descriptors hold the stage bars against the restatement (tests/eps.py)."""
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 30000, scene_id=4)
    kpm, kps = synth.voxel_grid(model, 0.01), synth.voxel_grid(scene, 0.02)
    r = 0.05
    p = b200.shot_params(normal_k=0, normal_radius=r, descr_radius=r, match_mode=2, match_thr=0.0, gc_size=0.02,
                         gc_threshold=3, max_instances=2048)
    m = ctx.model_create_fpfh(kpm, p)
    dm, kk = m.download()
    assert dm.shape == (len(kpm), 33) and np.array_equal(kk, kpm)
    res = ctx.register_scene_fpfh(m, kps, p, want_desc=True)
    # per-call API, same stages
    cm, cs = ctx.cloud(kpm), ctx.cloud(kps)
    nm, ns = ctx.normals(cm, radius=r), ctx.normals(cs, radius=r)
    fm, fs = ctx.fpfh33(cm, nm, r), ctx.fpfh33(cs, ns, r)
    assert np.array_equal(dm, fm, equal_nan=True) and np.array_equal(res["desc"], fs, equal_nan=True)
    c = ctx.match(fm, fs, 2, 0.0)
    assert c.tobytes() == res["corrs"].tobytes() and len(c) > 100
    T, inst, n = ctx.gc_recognize(kpm, kps, c, 0.02, 3, max_inst=2048)
    assert n == res["n_instances"] and all(a.tobytes() == b.tobytes() for a, b in zip(inst, res["instances"]))
    # against the restatement, stage by stage from identical inputs
    eps.normals_check(orc, ns, kps, radius=r, label="resident fpfh: normals")
    eps.fpfh_check(orc, fs, kps, ns, r, label="resident fpfh: descriptors")
    oc = orc.match(fm, fs, 2, 0.0)
    assert oc.tobytes() == c.tobytes()
    cm.close()
    cs.close()
    m.close()


def test_desc_index_batched_k1_equals_single_queries(ctx, orc):
    """b200_desc_index_knn with a batch of k = 1 queries goes through the correspondence-search machinery (tensor-core
    filter + exact rescoring for large indices); the per-query call goes through the per-query kernel.  Same answers,
    bit for bit, including rows with non-finite values on either side."""
    rng = np.random.Generator(np.random.PCG64(9))
    for K, D in ((3000, 352), (500, 352), (2000, 33)):
        centres = rng.gamma(0.3, 1.0, (100, D)).astype(np.float32)
        model = (centres[rng.integers(0, 100, K)] + 0.05 * rng.gamma(0.3, 1.0, (K, D))).astype(np.float32)
        model /= np.linalg.norm(model, axis=1, keepdims=True)
        q = (model[rng.integers(0, K, 300)] * rng.uniform(0.99, 1.01, (300, D))).astype(np.float32)
        model[7, 3] = np.nan
        q[11, 0] = np.inf
        ix = ctx.desc_index(model)
        bi, bd, kf = ix.knn(q, 1)
        assert kf == 1
        for r in (0, 5, 11, 42, 123, 299):
            si, sd, _ = ix.knn(q[r:r + 1], 1)
            if r == 11:
                assert bi[r, 0] == -1
                continue
            assert si[0, 0] == bi[r, 0] and sd[0, 0].tobytes() == bd[r, 0].tobytes(), (K, D, r)
        # and against the restatement's search on the valid rows
        oc = orc.match(model, q, 1, 1e30, omp=True)
        ok = oc["index_match"]
        assert np.array_equal(bi[ok, 0], oc["index_query"]) and np.array_equal(bd[ok, 0], oc["distance"])
        ix.close()


def test_new_entry_points_edge_cases(ctx, b200, synth):
    """Empty and degenerate inputs through the round-2 entry points: nothing crashes, nothing is invented."""
    p = b200.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                         max_instances=64)
    model = synth.make_model("y", 3000)
    kpm = synth.voxel_grid(model, 0.02)
    m = ctx.model_create_shot(model, kpm, p)
    scene = synth.make_scene(("y",), 8000, scene_id=3)
    # sharded call without a communicator (world 1): no keypoints, then keypoints far away from the scene
    r = ctx.register_scene_shot_sharded(m, p, scene, np.zeros((0, 3), np.float32))
    assert r["n_instances"] == 0 and len(r["corrs"]) == 0
    far = np.full((5, 3), 50.0, np.float32)
    r = ctx.register_scene_shot_sharded(m, p, scene, far)
    assert r["n_instances"] == 0 and len(r["corrs"]) == 0
    m.close()
    # FPFH pipeline: a model of three isolated points (no neighbour within the radius: PCL's histograms stay all zero)
    pf = b200.shot_params(normal_k=0, normal_radius=0.05, descr_radius=0.05, match_mode=2, match_thr=0.0, gc_size=0.02,
                          gc_threshold=3, max_instances=64)
    tiny = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    mf = ctx.model_create_fpfh(tiny, pf)
    dm, _ = mf.download()
    assert dm.shape == (3, 33)
    from oracle import pcl_oracle as orc_
    assert np.array_equal(dm, orc_.fpfh33(tiny, orc_.normals(tiny, radius=0.05), 0.05), equal_nan=True)
    kq = synth.voxel_grid(scene, 0.03)
    r = ctx.register_scene_fpfh(mf, kq, pf, want_desc=True)
    assert r["corrs"].tobytes() == orc_.match(dm, r["desc"], 2, 0.0).tobytes()
    r = ctx.register_scene_fpfh(mf, np.zeros((0, 3), np.float32), pf)
    assert r["n_instances"] == 0 and len(r["corrs"]) == 0
    mf.close()
    # a SHOT model cannot be used with the FPFH scene call
    m = ctx.model_create_shot(model, kpm, p)
    with pytest.raises(Exception):
        ctx.register_scene_fpfh(m, kq, pf)
    m.close()
    # batched k = 1 index queries on an index without a single valid row
    ix = ctx.desc_index(np.full((40, 352), np.nan, np.float32))
    bi, bd, kf = ix.knn(np.ones((64, 352), np.float32), 1)
    assert kf == 0 and np.all(bi == -1)
    ix.close()
