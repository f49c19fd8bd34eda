"""The FPFH pipeline's Hough branch (b200_model_create_fpfh_hough, b200_register_scene_fpfh_hough): FPFH33 on the
keypoint clouds, k = 2 ratio matching, BOARD frames over the dense clouds and Hough3DGrouping, as FPFH_demo.cpp:405-585
runs them.  Checked against the per-call chain on the same rand() stream (byte for byte), against the CPU oracle chain,
for determinism across scene order, on its edge cases, and against apps/fpfh_recognition --hough.  Also: a model of
the wrong descriptor length is refused by the SHOT registrations before anything is launched."""
import os
import subprocess

import numpy as np

import eps
import pytest

from conftest import PKG_NAME

pytestmark = pytest.mark.gpu

SEED = 11
R = 0.05           # FPFH and keypoint-normal radius of BASELINE config 2
SURFACE_K = 50     # normals of the dense clouds (FPFH_demo.cpp:405-409)
MAX_INST = 1 << 15


@pytest.fixture(scope="module")
def small(synth):
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 30000, scene_id=4)
    return model, synth.voxel_grid(model, 0.01), scene, synth.voxel_grid(scene, 0.02)


@pytest.fixture(scope="module")
def config2(synth):
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 100000, scene_id=1)
    return model, synth.voxel_grid(model, 0.01), scene, synth.voxel_grid(scene, 0.01)


def _params(b200, **kw):
    p = dict(normal_k=0, normal_radius=R, descr_radius=R, match_mode=2, match_thr=0.0, gc_size=0.02, gc_threshold=3,
             max_instances=MAX_INST)
    p.update(kw)
    return b200.shot_params(**p)


def _hough(b200, **kw):
    h = dict(rf_radius=0.02, bin_size=0.02, threshold=2.0)
    h.update(kw)
    return b200.hough_params(**h)


def _chain_frames(b200, model, kpm, scene, kps, h, seed=SEED):
    """srand(seed) -> board_lrf(dense model) -> board_lrf(dense scene) on a fresh context, each over its cloud's k = 50
    normals; then a further call, to show where the stream went on."""
    c = b200.Context(0)
    c.srand(seed)
    cm, cs = c.cloud(model), c.cloud(scene)
    mrf = c.board_lrf(cm, c.normals(cm, k=SURFACE_K), kpm, h.rf_radius, h.board)
    srf = c.board_lrf(cs, c.normals(cs, k=SURFACE_K), kps, h.rf_radius, h.board)
    after = c.board_lrf(cs, c.normals(cs, k=SURFACE_K), kps[:50], h.rf_radius, h.board)
    cm.close()
    cs.close()
    c.close()
    return mrf, srf, after


def _chain_descriptors(ctx, kpm, kps):
    """Per-call descriptor side: radius normals and FPFH33 on each keypoint cloud (input = surface)."""
    cm, cs = ctx.cloud(kpm), ctx.cloud(kps)
    nm, ns = ctx.normals(cm, radius=R), ctx.normals(cs, radius=R)
    fm, fs = ctx.fpfh33(cm, nm, R), ctx.fpfh33(cs, ns, R)
    cm.close()
    cs.close()
    return fm, fs, ns


def _same_result(a, b):
    assert a["n_instances"] == b["n_instances"]
    assert a["corrs"].tobytes() == b["corrs"].tobytes()
    assert np.array_equal(a["transforms"], b["transforms"])
    assert len(a["instances"]) == len(b["instances"])
    for x, y in zip(a["instances"], b["instances"]):
        assert x.tobytes() == y.tobytes()


def test_model_descriptors_and_frames(b200, small):
    """Descriptors = b200_model_create_fpfh's; frames = srand(s) + board_lrf(dense model, its k = 50 normals, keypoints)
    on a fresh context; the creating context's stream then continues as after that per-call BOARD."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    plain = c.model_create_fpfh(kpm, p)
    (d, k), (d0, k0) = m.download(), plain.download()
    assert d.shape == (len(kpm), 33) and d.tobytes() == d0.tobytes() and k.tobytes() == k0.tobytes()
    rf = m.download_frames()
    mrf, _, _ = _chain_frames(b200, model, kpm, scene, kps, h)
    assert rf.shape == (len(kpm), 9) and np.isfinite(rf).any()
    assert np.array_equal(rf, mrf, equal_nan=True)
    ref = b200.Context(0)
    ref.srand(SEED)
    rm, rs = ref.cloud(model), ref.cloud(scene)
    ref.board_lrf(rm, ref.normals(rm, k=SURFACE_K), kpm, h.rf_radius, h.board)
    cs = c.cloud(scene)
    a = c.board_lrf(cs, c.normals(cs, k=SURFACE_K), kps, h.rf_radius, h.board)
    b = ref.board_lrf(rs, ref.normals(rs, k=SURFACE_K), kps, h.rf_radius, h.board)
    assert np.array_equal(a, b, equal_nan=True)
    for x in (m, plain, cs, rm, rs):
        x.close()
    c.close()
    ref.close()


@pytest.mark.parametrize("which", ["small", "config2"])
def test_pipeline_equals_per_call_chain(b200, small, config2, which):
    """Descriptors = fpfh33 on the keypoint cloud; correspondences = match(..., 2, 0.0) and register_scene_fpfh's;
    scene frames = the chain's board_lrf(scene) after the model's; instances and transforms = hough3d_recognize on
    those correspondences and frames."""
    model, kpm, scene, kps = small if which == "small" else config2
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    res = c.register_scene_fpfh_hough(m, scene, kps, p, h, surface_normal_k=SURFACE_K, want_desc=True)
    assert res["status"] == b200.OK
    fm, fs, _ = _chain_descriptors(c, kpm, kps)
    assert np.array_equal(res["desc"], fs, equal_nan=True)
    corrs = c.match(fm, fs, 2, 0.0)
    assert res["corrs"].tobytes() == corrs.tobytes() and len(corrs) > 100
    gc = c.register_scene_fpfh(m, kps, p)
    assert gc["corrs"].tobytes() == corrs.tobytes()
    mrf, srf, _ = _chain_frames(b200, model, kpm, scene, kps, h)
    assert np.array_equal(res["rf"], srf, equal_nan=True)
    T, inst, n = c.hough3d_recognize(kpm, mrf, kps, srf, corrs, h.bin_size, h.threshold, max_inst=MAX_INST)
    assert n == res["n_instances"] and n > 0
    assert np.array_equal(T, res["transforms"])
    assert len(inst) == len(res["instances"])
    for a, b in zip(inst, res["instances"]):
        assert a.tobytes() == b.tobytes()
    print(which, "keypoints", len(kpm), len(kps), "correspondences", len(corrs), "instances", n)
    m.close()
    c.close()


def test_pipeline_against_oracle_chain(b200, orc, small):
    """Oracle chain stage by stage from identical inputs: normals and FPFH through the stage bars of tests/eps.py,
    correspondences equal to the oracle's search on the same descriptors, frames within 1e-5 on the rows stable under
    the 2-ulp angle variants (the oracle's BOARD fed the dense normals the pipeline computed), and, on the pipeline's
    own correspondences and frames, the same instances byte for byte and poses within 1e-4."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    res = c.register_scene_fpfh_hough(m, scene, kps, p, h, surface_normal_k=SURFACE_K, want_desc=True)
    fm, fs, ns = _chain_descriptors(c, kpm, kps)
    eps.normals_check(orc, ns, kps, radius=R, label="fpfh hough: keypoint normals")
    eps.fpfh_check(orc, res["desc"], kps, ns, R, label="fpfh hough: descriptors")
    assert orc.match(fm, res["desc"], 2, 0.0).tobytes() == res["corrs"].tobytes()
    ob = orc.board_params()
    cm, cs = c.cloud(model), c.cloud(scene)
    nm, nsd = c.normals(cm, k=SURFACE_K), c.normals(cs, k=SURFACE_K)   # what dev_normals gave the pipeline
    cm.close()
    cs.close()
    o_m, used = orc.board_lrf(model, nm, kpm, h.rf_radius, ob, rand_seed=SEED)
    o_s, _ = orc.board_lrf(scene, nsd, kps, h.rf_radius, ob, rand_seed=SEED, rand_skip=used)

    def variants(cloud, nrm, kp, **kw):
        out = []
        for name in ("board_angle_up", "board_angle_down"):
            with orc.variant(name):
                out.append(orc.board_lrf(cloud, nrm, kp, h.rf_radius, ob, rand_seed=SEED, **kw)[0])
        return out

    for got, ref, var in ((m.download_frames(), o_m, variants(model, nm, kpm)),
                          (res["rf"], o_s, variants(scene, nsd, kps, rand_skip=used))):
        assert np.array_equal(np.isnan(got[:, 0]), np.isnan(ref[:, 0]))
        ok = ~np.isnan(ref[:, 0])
        stable = ok.copy()
        for v in var:
            stable &= np.nan_to_num(np.abs(v - ref)).max(axis=1) <= 5e-6
        assert stable.sum() >= 0.95 * ok.sum(), (int(stable.sum()), int(ok.sum()))
        err = np.abs(got - ref).max(axis=1)
        assert err[stable].max() <= 1e-5, float(err[stable].max())
    oT, oinst = orc.hough3d_recognize(kpm, m.download_frames(), kps, res["rf"], res["corrs"], h.bin_size, h.threshold,
                                      max_inst=MAX_INST)
    assert res["n_instances"] == len(oT) > 0
    for a, b in zip(res["instances"], oinst):
        assert a.tobytes() == b.tobytes()
    assert max(np.abs(A - B).max() for A, B in zip(res["transforms"], oT)) < 1e-4
    m.close()
    c.close()


def test_determinism_scene_order(b200, synth, small):
    """Scenes A, B, A: every scene draws its frames from the model's recorded stream state, so both A results are
    identical, frames included."""
    model, kpm, sa, ka = small
    sb = synth.make_scene(("y",), 40000, scene_id=1)
    kb = synth.voxel_grid(sb, 0.02)
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    a1 = c.register_scene_fpfh_hough(m, sa, ka, p, h, surface_normal_k=SURFACE_K)
    b1 = c.register_scene_fpfh_hough(m, sb, kb, p, h, surface_normal_k=SURFACE_K)
    a2 = c.register_scene_fpfh_hough(m, sa, ka, p, h, surface_normal_k=SURFACE_K)
    assert a1["status"] == b1["status"] == a2["status"] == b200.OK
    assert a1["n_instances"] > 0 and b1["n_instances"] > 0
    _same_result(a1, a2)
    assert np.array_equal(a1["rf"], a2["rf"], equal_nan=True)
    m.close()
    c.close()


def test_pipeline_edge_cases(b200, small):
    """Bin-size overflow (B200_ERR_CAPACITY, correspondences kept), max_instances overflow (the first one kept), no
    scene keypoints, the surface normal settings, and models the call does not take."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)

    def reg(mm, pp=p, hh=h, kp=kps, surface_normal_k=SURFACE_K, surface_normal_radius=0.0):
        return c.register_scene_fpfh_hough(mm, scene, kp, pp, hh, surface_normal_k=surface_normal_k,
                                           surface_normal_radius=surface_normal_radius)

    full = reg(m)
    assert full["status"] == b200.OK and full["n_instances"] >= 2
    over = reg(m, hh=_hough(b200, bin_size=1e-4))
    assert over["status"] == b200.ERR_CAPACITY and over["n_instances"] == 0 and len(over["instances"]) == 0
    assert over["corrs"].tobytes() == full["corrs"].tobytes()
    one = reg(m, pp=_params(b200, max_instances=1))
    assert one["status"] == b200.ERR_CAPACITY and one["n_instances"] == full["n_instances"]
    assert len(one["instances"]) == 1 and one["instances"][0].tobytes() == full["instances"][0].tobytes()
    assert np.array_equal(one["transforms"][0], full["transforms"][0])
    empty = reg(m, kp=kps[:0])
    assert empty["status"] == b200.OK and empty["n_instances"] == 0 and len(empty["corrs"]) == 0
    # exactly one of surface_normal_k / surface_normal_radius
    for k, r in ((0, 0.0), (SURFACE_K, 0.03)):
        with pytest.raises(b200.B200Error) as e:
            reg(m, surface_normal_k=k, surface_normal_radius=r)
        assert e.value.code == b200.ERR_INVALID
        with pytest.raises(b200.B200Error) as e:
            c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=k, surface_normal_radius=r)
        assert e.value.code == b200.ERR_INVALID
    # the radius setting is a surface normal setting too
    rad = reg(m, surface_normal_k=0, surface_normal_radius=0.03)
    assert rad["status"] == b200.OK and rad["corrs"].tobytes() == full["corrs"].tobytes()
    # a SHOT model (with or without frames) and an FPFH model without frames
    shot_p = b200.shot_params(normal_k=10, descr_radius=0.02, max_instances=64)
    for other in (c.model_create_shot(model, kpm, shot_p), c.model_create_shot_hough(model, kpm, shot_p, h),
                  c.model_create_fpfh(kpm, p)):
        with pytest.raises(b200.B200Error) as e:
            reg(other)
        assert e.value.code == b200.ERR_INVALID
        other.close()
    m.close()
    c.close()


def test_fpfh_model_refused_by_shot_registrations(b200, small):
    """An FPFH model (33-float descriptors, with frames) into the SHOT registrations: B200_ERR_INVALID before anything
    is launched; into register_scene_fpfh (GC): the plain FPFH model's result."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    shot_p = b200.shot_params(normal_k=10, descr_radius=0.02, max_instances=64)
    c = b200.Context(0)
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    c.sync()
    for call in (lambda: c.register_scene_shot(m, scene, kps, shot_p),
                 lambda: c.register_scene_shot_hough(m, scene, kps, shot_p, h)):
        before = c.launches
        with pytest.raises(b200.B200Error) as e:
            call()
        assert e.value.code == b200.ERR_INVALID
        assert c.launches == before
    for hough in (None, h):
        with pytest.raises(b200.B200Error) as e:
            b200.register_scene_batch(m, [scene, scene], [kps, kps], shot_p, lanes=2, hough=hough)
        assert e.value.code == b200.ERR_INVALID
    plain = c.model_create_fpfh(kpm, p)
    _same_result(c.register_scene_fpfh(m, kps, p), c.register_scene_fpfh(plain, kps, p))
    plain.close()
    m.close()
    c.close()


def test_fpfh_recognition_app_hough(b200, synth, small, tmp_path):
    """apps/fpfh_recognition --hough (FPFH_demo's grouping block through the PCL-style adapters) writes the .corr, .T
    and .rf of the pipeline on a fresh context (srand(1)), byte for byte."""
    import importlib
    apps = {os.path.basename(x): x for x in importlib.import_module(PKG_NAME + ".build").build_apps()}
    model, kpm, scene, kps = small
    w = lambda name, a: np.ascontiguousarray(a[:, :3], dtype=np.float32).tofile(str(tmp_path / name))
    for name, a in (("m.f32", model), ("s.f32", scene), ("mk.f32", kpm), ("sk.f32", kps)):
        w(name, a)
    prefix = str(tmp_path / "out")
    r = subprocess.run([apps["fpfh_recognition"], "--hough", str(tmp_path / "m.f32"), str(tmp_path / "s.f32"),
                        str(tmp_path / "mk.f32"), str(tmp_path / "sk.f32"), prefix, str(R), "0.02", "2"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)   # a fresh context: srand(1), as the app's
    m = c.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    res = c.register_scene_fpfh_hough(m, scene, kps, p, h, surface_normal_k=SURFACE_K)
    assert res["status"] == b200.OK and res["n_instances"] > 0
    corr = np.fromfile(prefix + ".corr", dtype=b200.CORR_DTYPE)
    T = np.fromfile(prefix + ".T", dtype=np.float32).reshape(-1, 4, 4)
    rf = np.fromfile(prefix + ".rf", dtype=np.float32).reshape(-1, 9)
    assert corr.tobytes() == res["corrs"].tobytes()
    assert np.array_equal(T, res["transforms"])
    assert np.array_equal(rf, np.concatenate([m.download_frames(), res["rf"]]), equal_nan=True)
    assert "Model instances found: %d" % res["n_instances"] in r.stdout
    m.close()
    c.close()
