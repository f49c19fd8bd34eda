"""The resident Hough branch (b200_model_create_shot_hough, b200_register_scene_shot_hough and its device and lanes
forms): BOARD frames and Hough3DGrouping inside scene registration.  Checked against the per-call chain on the same
rand() stream (byte for byte), against the CPU oracle chain, for determinism across scene order / lanes / forms, and on
the Hough corner cases of the device-side grouping."""
import ctypes as C
import os
import subprocess

import numpy as np

import eps
import pytest

from conftest import PKG_NAME

pytestmark = pytest.mark.gpu

SEED = 11


@pytest.fixture(scope="module")
def ctx(b200):
    c = b200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def small(synth):
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 40000, scene_id=1)
    return model, synth.uniform_sampling(model, 0.02), scene, synth.uniform_sampling(scene, 0.03)


@pytest.fixture(scope="module")
def mid(synth):
    model = synth.make_model("y", 20000)
    scene = synth.make_scene(("y", "diagonal"), 60000, scene_id=30)
    return model, synth.uniform_sampling(model, 0.005), scene, synth.uniform_sampling(scene, 0.02)


def _params(b200, **kw):
    p = dict(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, max_instances=4096)
    p.update(kw)
    return b200.shot_params(**p)


def _hough(b200, **kw):
    h = dict(rf_radius=0.015, bin_size=0.02, threshold=2.0)
    h.update(kw)
    return b200.hough_params(**h)


def _chain_frames(b200, model, kpm, scene, kps, h, seed=SEED, k=10):
    """srand(seed) -> board_lrf(model) -> board_lrf(scene) on a fresh context, normals from the same dev_normals call
    as the pipeline."""
    c = b200.Context(0)
    c.srand(seed)
    cm, cs = c.cloud(model), c.cloud(scene)
    mrf = c.board_lrf(cm, c.normals(cm, k=k), kpm, h.rf_radius, h.board)
    srf = c.board_lrf(cs, c.normals(cs, k=k), kps, h.rf_radius, h.board)
    after = c.board_lrf(cs, c.normals(cs, k=k), kps[:50], h.rf_radius, h.board)   # where the stream went on
    cm.close()
    cs.close()
    c.close()
    return mrf, srf, after


def _same_result(a, b):
    assert a["n_instances"] == b["n_instances"]
    assert a["corrs"].tobytes() == b["corrs"].tobytes()
    assert np.array_equal(a["transforms"], b["transforms"])
    assert len(a["instances"]) == len(b["instances"])
    for x, y in zip(a["instances"], b["instances"]):
        assert x.tobytes() == y.tobytes()


def test_model_frames_follow_the_context_stream(b200, small):
    """Model frames = srand(s) + board_lrf(model) on a fresh context; the creating context's stream then continues
    as after that call; descriptors as b200_model_create_shot; a model without frames has none to give."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_shot_hough(model, kpm, p, h)
    rf = m.download_frames()
    mrf, _, _ = _chain_frames(b200, model, kpm, scene, kps, h)
    assert rf.shape == (len(kpm), 9) and np.isfinite(rf).any()
    assert np.array_equal(rf, mrf, equal_nan=True)
    # the context's stream continues exactly as after the per-call model frames
    ref = b200.Context(0)
    ref.srand(SEED)
    rm, rs = ref.cloud(model), ref.cloud(scene)
    ref.board_lrf(rm, ref.normals(rm, k=10), kpm, h.rf_radius, h.board)
    cs = c.cloud(scene)
    a = c.board_lrf(cs, c.normals(cs, k=10), kps, h.rf_radius, h.board)
    b = ref.board_lrf(rs, ref.normals(rs, k=10), kps, h.rf_radius, h.board)
    assert np.array_equal(a, b, equal_nan=True)
    m0 = c.model_create_shot(model, kpm, p)
    assert m.download()[0].tobytes() == m0.download()[0].tobytes()
    with pytest.raises(b200.B200Error) as e:
        m0.download_frames()
    assert e.value.code == b200.ERR_INVALID
    with pytest.raises(b200.B200Error) as e:
        c.register_scene_shot_hough(m0, scene, kps, p, h)
    assert e.value.code == b200.ERR_INVALID
    for x in (m, m0, cs, rm, rs):
        x.close()
    c.close()
    ref.close()


@pytest.mark.parametrize("which", ["small", "mid"])
def test_pipeline_equals_per_call_chain(b200, small, mid, which):
    """Correspondences = register_scene_shot's; scene frames = a fresh context's srand(s) -> board_lrf(model) ->
    board_lrf(scene); instances and transforms = hough3d_recognize on those correspondences and frames."""
    model, kpm, scene, kps = small if which == "small" else mid
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_shot_hough(model, kpm, p, h)
    res = c.register_scene_shot_hough(m, scene, kps, p, h)
    assert res["status"] == b200.OK
    gc = c.register_scene_shot(m, scene, kps, p)
    assert res["corrs"].tobytes() == gc["corrs"].tobytes() and len(res["corrs"]) > 50
    mrf, srf, _ = _chain_frames(b200, model, kpm, scene, kps, h)
    assert np.array_equal(res["rf"], srf, equal_nan=True)
    T, inst, n = c.hough3d_recognize(kpm, mrf, kps, srf, res["corrs"], h.bin_size, h.threshold, max_inst=4096)
    assert n == res["n_instances"] and n > 0
    assert np.array_equal(T, res["transforms"])
    for a, b in zip(inst, res["instances"]):
        assert a.tobytes() == b.tobytes()
    m.close()
    c.close()


def test_pipeline_against_oracle_chain(b200, orc, small):
    """Oracle chain: normals -> SHOT352 -> match -> BOARD (model, then scene on the continued stream) -> Hough.
    Correspondences through eps.corr_check; frames within 1e-5 on the rows stable under the 2-ulp angle variants (as
    test_board_lrf_parity), the oracle's BOARD fed the normals the pipeline computed (normals that differ in the last
    bits, as the oracle's do, move an ill-conditioned frame by more than 1e-5; normals have their own parity tests); on
    the pipeline's own correspondences and frames, the same instances byte for byte and poses within 1e-4."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_shot_hough(model, kpm, p, h)
    res = c.register_scene_shot_hough(m, scene, kps, p, h)
    nm, ns = orc.normals(model, k=10), orc.normals(scene, k=10)
    odm, _ = orc.shot352(model, nm, kpm, 0.02)
    ods, _ = orc.shot352(scene, ns, kps, 0.02)
    eps.corr_check(odm, ods, res["corrs"], orc.match(odm, ods, 1, 0.25), 0.25, label="Hough pipeline correspondences")
    ob = orc.board_params()
    cm, cs = c.cloud(model), c.cloud(scene)
    nm, ns = c.normals(cm, k=10), c.normals(cs, k=10)   # what dev_normals gave the pipeline
    cm.close()
    cs.close()
    o_m, used = orc.board_lrf(model, nm, kpm, h.rf_radius, ob, rand_seed=SEED)
    o_s, _ = orc.board_lrf(scene, ns, kps, h.rf_radius, ob, rand_seed=SEED, rand_skip=used)

    def variants(cloud, nrm, kp, **kw):
        out = []
        for name in ("board_angle_up", "board_angle_down"):
            with orc.variant(name):
                out.append(orc.board_lrf(cloud, nrm, kp, h.rf_radius, ob, rand_seed=SEED, **kw)[0])
        return out

    for got, ref, var in ((m.download_frames(), o_m, variants(model, nm, kpm)),
                          (res["rf"], o_s, variants(scene, ns, kps, rand_skip=used))):
        assert np.array_equal(np.isnan(got[:, 0]), np.isnan(ref[:, 0]))
        ok = ~np.isnan(ref[:, 0])
        stable = ok.copy()
        for v in var:
            stable &= np.nan_to_num(np.abs(v - ref)).max(axis=1) <= 5e-6
        assert stable.sum() >= 0.95 * ok.sum(), (int(stable.sum()), int(ok.sum()))
        err = np.abs(got - ref).max(axis=1)
        assert err[stable].max() <= 1e-5, float(err[stable].max())
    oT, oinst = orc.hough3d_recognize(kpm, m.download_frames(), kps, res["rf"], res["corrs"], h.bin_size, h.threshold,
                                      max_inst=4096)
    assert res["n_instances"] == len(oT) > 0
    for a, b in zip(res["instances"], oinst):
        assert a.tobytes() == b.tobytes()
    assert max(np.abs(A - B).max() for A, B in zip(res["transforms"], oT)) < 1e-4
    m.close()
    c.close()


def test_determinism_order_lanes_and_forms(b200, small, mid):
    """Scenes A, B, A give identical A results (every scene draws from the model's recorded stream state); the batch
    with 1, 3 and 8 lanes equals single calls byte for byte; the device form equals the host form."""
    import torch
    model, kpm, sa, ka = mid
    _, _, sb, kb = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_shot_hough(model, kpm, p, h)
    a1 = c.register_scene_shot_hough(m, sa, ka, p, h)
    b1 = c.register_scene_shot_hough(m, sb, kb, p, h)
    a2 = c.register_scene_shot_hough(m, sa, ka, p, h)
    _same_result(a1, a2)
    assert np.array_equal(a1["rf"], a2["rf"], equal_nan=True)
    scenes, kps = [sa, sb, sa, sb, sb, sa, sb, sa, sa], [ka, kb, ka, kb, kb, ka, kb, ka, ka]
    for lanes in (1, 3, 8):
        out = b200.register_scene_batch(m, scenes, kps, p, lanes=lanes, hough=h)
        for s, r in enumerate(out):
            assert r["status"] == b200.OK
            _same_result(r, a1 if scenes[s] is sa else b1)
    # device form
    dev = torch.device("cuda", 0)
    Ks, mi = len(ka), p.max_instances
    out = {"transforms": torch.zeros(mi * 16, dtype=torch.float32, device=dev),
           "inst_offsets": torch.zeros(mi + 1, dtype=torch.int32, device=dev),
           "inst_counts": torch.zeros(mi, dtype=torch.int32, device=dev),
           "inst_corrs": torch.zeros((Ks, 3), dtype=torch.int32, device=dev), "corr_cap": Ks,
           "n_inst": torch.zeros(1, dtype=torch.int32, device=dev),
           "corrs": torch.zeros((Ks, 3), dtype=torch.int32, device=dev),
           "n_corrs": torch.zeros(1, dtype=torch.int32, device=dev),
           "rf": torch.zeros((Ks, 9), dtype=torch.float32, device=dev),
           "status": torch.full((1,), 7, dtype=torch.int32, device=dev)}
    d_xyz, d_kp = torch.from_numpy(sa).to(dev), torch.from_numpy(ka).to(dev)
    torch.cuda.synchronize()
    c.dev_register_scene_shot_hough(m, d_xyz, len(sa), 3, d_kp, Ks, 3, p, h, out)
    c.sync()
    assert int(out["status"].item()) == b200.OK
    n = int(out["n_inst"].item())
    assert n == a1["n_instances"]
    nc = int(out["n_corrs"].item())
    assert out["corrs"][:nc].cpu().numpy().view(b200.CORR_DTYPE).reshape(-1).tobytes() == a1["corrs"].tobytes()
    assert np.array_equal(out["rf"].cpu().numpy(), a1["rf"], equal_nan=True)
    assert np.array_equal(out["transforms"][:n * 16].cpu().numpy().reshape(n, 4, 4), a1["transforms"])
    offs = out["inst_offsets"][:n + 1].cpu().numpy()
    cnts = out["inst_counts"][:n].cpu().numpy()
    ic = out["inst_corrs"].cpu().numpy().view(b200.CORR_DTYPE).reshape(-1)
    for i in range(n):
        assert ic[offs[i]:offs[i] + cnts[i]].tobytes() == a1["instances"][i].tobytes()
    # bin-size overflow in the device form: *d_status
    c.dev_register_scene_shot_hough(m, d_xyz, len(sa), 3, d_kp, Ks, 3, p, _hough(b200, bin_size=1e-4), out)
    c.sync()
    assert int(out["status"].item()) == b200.ERR_CAPACITY and int(out["n_inst"].item()) == 0
    m.close()
    c.close()


def test_pipeline_edge_cases(b200, small):
    """Bin-size overflow (B200_ERR_CAPACITY, correspondences kept), max_instances overflow (the first ones kept),
    no scene keypoints, no correspondences."""
    model, kpm, scene, kps = small
    p, h = _params(b200), _hough(b200)
    c = b200.Context(0)
    c.srand(SEED)
    m = c.model_create_shot_hough(model, kpm, p, h)
    full = c.register_scene_shot_hough(m, scene, kps, p, h)
    assert full["n_instances"] >= 2
    over = c.register_scene_shot_hough(m, scene, kps, p, _hough(b200, bin_size=1e-4))
    assert over["status"] == b200.ERR_CAPACITY and over["n_instances"] == 0
    assert over["corrs"].tobytes() == full["corrs"].tobytes()
    one = c.register_scene_shot_hough(m, scene, kps, _params(b200, max_instances=1), h)
    assert one["status"] == b200.ERR_CAPACITY and one["n_instances"] == full["n_instances"]
    assert len(one["instances"]) == 1 and one["instances"][0].tobytes() == full["instances"][0].tobytes()
    assert np.array_equal(one["transforms"][0], full["transforms"][0])
    empty = c.register_scene_shot_hough(m, scene, kps[:0], p, h)
    assert empty["status"] == b200.OK and empty["n_instances"] == 0 and len(empty["corrs"]) == 0
    none = c.register_scene_shot_hough(m, scene, kps, _params(b200, match_thr=1e-12), h)
    assert none["status"] == b200.OK and none["n_instances"] == 0 and len(none["corrs"]) == 0
    m.close()
    c.close()


# ------------------------------------------------------------------------------------------ crafted Hough inputs
# Model keypoints on a 1/64 grid (their centroid, the votes and the scene keypoints below are exact in float32) with
# identity frames: correspondence (i, j) with scene keypoint kp_i - centroid + v votes exactly v.
def _crafted(targets, seed=0):
    rng = np.random.Generator(np.random.PCG64(seed))
    kpm = (rng.integers(0, 16, size=(64, 3)) / 64.0).astype(np.float32)
    c = kpm.astype(np.float64).mean(axis=0)
    assert np.array_equal(c.astype(np.float32), kpm.sum(axis=0, dtype=np.float32) / np.float32(64))
    kps, corrs, i = [], [], 0
    for v, count in targets:
        for _ in range(count):
            kps.append(kpm[i % 64].astype(np.float64) - c + np.asarray(v, dtype=np.float64))
            corrs.append((i % 64, len(kps) - 1, 0.1))
            i += 7
    kps = np.asarray(kps, dtype=np.float32)
    corrs = np.array(corrs, dtype=[("index_query", "<i4"), ("index_match", "<i4"), ("distance", "<f4")])
    eye = np.tile(np.eye(3, dtype=np.float32).reshape(1, 9), (1, 1))
    return kpm, np.repeat(eye, len(kpm), 0), kps, np.repeat(eye, len(kps), 0), corrs


def _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, bin_size, thr, expect=None, max_inst=4096):
    T, inst, n = ctx.hough3d_recognize(kpm, mrf, kps, srf, corrs, bin_size, thr, max_inst=max_inst)
    oT, oinst = orc.hough3d_recognize(kpm, mrf, kps, srf, corrs, bin_size, thr, max_inst=4096)
    assert n == len(oT), (n, len(oT))
    if expect is not None:
        assert n == expect
    for a, b in zip(inst, oinst):
        assert a.tobytes() == b.tobytes()
    for A, B in zip(T, oT):
        assert np.abs(A - B).max() < 1e-4
    return n, inst


def test_hough_corner_cases(ctx, orc, b200):
    """The device-side Hough space: all votes on one coordinate (a degenerate axis holds no bin), a vote exactly on
    the upper bound (dropped), NaN frames (skipped), a negative threshold (relative to the largest bin), max_inst
    overflow (B200_ERR_CAPACITY, the first max_inst valid) and a bin size that needs more than 2^27 bins."""
    # one coordinate: every vote has x = 0.5
    kpm, mrf, kps, srf, corrs = _crafted([((0.5, 0.0, 0.0), 5), ((0.5, 0.5, 0.25), 6)])
    _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, 0.25, 2.0, expect=0)
    # span [0, 1] with bin 0.25: 4 bins per axis; the 7 votes at (1, 1, 1) lie on the upper bound and are dropped
    kpm, mrf, kps, srf, corrs = _crafted([((0.0, 0.0, 0.0), 5), ((0.5, 0.5, 0.5), 6), ((1.0, 1.0, 1.0), 7)])
    _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, 0.25, 2.0, expect=2)
    # NaN scene frames: their correspondences do not vote
    srf2 = srf.copy()
    srf2[[0, 1, 2, 6, 7]] = np.nan
    n, inst = _check_against_oracle(ctx, orc, kpm, mrf, kps, srf2, corrs, 0.25, 2.0, expect=2)
    assert not set(inst[0]["index_match"]) & {0, 1, 2}
    # negative threshold: 0.6 of the largest bin (9 votes) keeps the 9-vote bin and the 6-vote bin
    kpm, mrf, kps, srf, corrs = _crafted([((0.0, 0.0, 0.0), 5), ((0.5, 0.5, 0.5), 9), ((0.75, 0.25, 0.5), 6),
                                          ((1.0, 1.0, 1.0), 1)])
    _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, 0.25, -0.6, expect=2)
    # max_inst overflow
    targets = [((0.25 * (t % 4), 0.25 * (t // 4), 0.125 * t), 4) for t in range(7)] + [((1.0, 1.0, 1.0), 1)]
    kpm, mrf, kps, srf, corrs = _crafted(targets)
    n_all, inst_all = _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, 0.125, 3.0)
    assert n_all == 7
    T3, inst3, n3 = ctx.hough3d_recognize(kpm, mrf, kps, srf, corrs, 0.125, 3.0, max_inst=3)
    assert n3 == 7 and len(inst3) == 3
    for a, b in zip(inst3, inst_all[:3]):
        assert a.tobytes() == b.tobytes()
    # more than 2^27 bins: B200_ERR_CAPACITY and no instance
    L = b200.lib()
    T = np.zeros((16, 16), np.float32)
    off = np.zeros(17, np.int32)
    oc = np.zeros(len(corrs), dtype=b200.CORR_DTYPE)
    n = C.c_int(-1)
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    rc = L.b200_hough3d_recognize(ctx.h, f(kpm), f(mrf), len(kpm), 3, f(kps), f(srf), len(kps), 3,
                                  corrs.ctypes.data_as(C.POINTER(b200.Corr)), len(corrs), 1e-3, 2.0, f(T), 16,
                                  off.ctypes.data_as(C.POINTER(C.c_int)), oc.ctypes.data_as(C.POINTER(b200.Corr)),
                                  len(corrs), C.byref(n))
    assert rc == b200.ERR_CAPACITY and n.value == 0
    # and the context is fine afterwards
    _check_against_oracle(ctx, orc, kpm, mrf, kps, srf, corrs, 0.125, 3.0, expect=7)


def test_fullsize_lanes_equal_single_calls(b200, synth):
    """Three 1 M-point Kinect-like scenes (about 91 000 keypoints each): the batch with 2 lanes equals single calls
    byte for byte."""
    p = b200.shot_params(normal_k=20, descr_radius=0.02, match_mode=1, match_thr=0.25, max_instances=4096)
    h = b200.hough_params()
    model = synth.make_model("y", 50000)
    kpm = synth.uniform_sampling(model, 0.005)
    scenes = [synth.make_kinect_scene(("y", "diagonal", "horizontal"), target_points=1_000_000, scene_id=s)
              for s in range(3)]
    kps = [synth.uniform_sampling(sc, 0.01) for sc in scenes]
    c = b200.Context(0)
    m = c.model_create_shot_hough(model, kpm, p, h)
    single = [c.register_scene_shot_hough(m, sc, kp, p, h) for sc, kp in zip(scenes, kps)]
    batch = b200.register_scene_batch(m, scenes, kps, p, lanes=2, hough=h)
    for a, b in zip(single, batch):
        assert b["status"] == a["status"]
        _same_result(a, b)
    print("full size:", [(len(k), len(r["corrs"]), r["n_instances"]) for k, r in zip(kps, single)])
    assert all(r["n_instances"] > 0 for r in single)
    m.close()
    c.close()


def test_batch_recognition_app_hough(b200, synth, tmp_path):
    """apps/batch_recognition --hough writes the same .T and .corr as the Python batch call."""
    import importlib
    apps = {os.path.basename(x): x for x in importlib.import_module(PKG_NAME + ".build").build_apps()}
    model = synth.make_model("y", 20000)
    kpm = synth.uniform_sampling(model, 0.005)
    w = lambda path, a: np.ascontiguousarray(a[:, :3], dtype=np.float32).tofile(path)
    w(tmp_path / "m.f32", model)
    w(tmp_path / "mk.f32", kpm)
    args, scenes, kps = [], [], []
    for s in range(3):
        sc = synth.make_scene(("y", "diagonal"), 60000, scene_id=30 + s)
        kp = synth.uniform_sampling(sc, 0.02)
        w(tmp_path / ("s%d.f32" % s), sc)
        w(tmp_path / ("k%d.f32" % s), kp)
        args += [str(tmp_path / ("s%d.f32" % s)), str(tmp_path / ("k%d.f32" % s))]
        scenes.append(sc)
        kps.append(kp)
    prefix = str(tmp_path / "out")
    r = subprocess.run([apps["batch_recognition"], "--hough", str(tmp_path / "m.f32"), str(tmp_path / "mk.f32"), prefix,
                        "2"] + args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    p = b200.shot_params(normal_k=20, descr_radius=0.02, match_mode=1, match_thr=0.25, max_instances=4096)
    h = b200.hough_params(rf_radius=0.02, bin_size=0.02, threshold=2.0)
    c = b200.Context(0)   # a fresh context: srand(1), as the app's
    m = c.model_create_shot_hough(model, kpm, p, h)
    ref = b200.register_scene_batch(m, scenes, kps, p, lanes=2, hough=h)
    for s in range(3):
        corr = np.fromfile("%s.%d.corr" % (prefix, s), dtype=b200.CORR_DTYPE)
        T = np.fromfile("%s.%d.T" % (prefix, s), dtype=np.float32).reshape(-1, 4, 4)
        assert corr.tobytes() == ref[s]["corrs"].tobytes() and np.array_equal(T, ref[s]["transforms"])
        assert "scene %d: %d correspondences, %d instances" % (s, len(ref[s]["corrs"]), ref[s]["n_instances"]) in r.stdout
    assert any(x["n_instances"] > 0 for x in ref)
    m.close()
    c.close()
