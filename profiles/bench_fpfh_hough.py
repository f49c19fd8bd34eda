"""Figures of the FPFH pipeline's Hough branch (b200_model_create_fpfh_hough + b200_register_scene_fpfh_hough).

Workload: BASELINE config 2 (bench.py `other_configs.config2_fpfh_demo`): the 5 000-point Y-joint model and
100 000-point scenes (synth.make_scene(("y",), 100000, scene_id=s); s = 1 is config 2's scene, the pool adds s = 2, 3,
...), keypoints voxel_grid(0.01), radius normals and FPFH33 at r = 0.05 on the keypoint clouds, the k = 2 ratio test;
the reference's Hough settings (SURVEY §2c: BOARD radius 0.02 with find_holes, bin 0.02, threshold 2) over the dense
clouds with k = 50 normals (FPFH_demo.cpp:405-409).  In one run:
  - FPFH-GC (b200_register_scene_fpfh, GC 0.02 / 3 as bench.py) and FPFH-Hough registrations, alternating scene by
    scene, host buffers in and out, a host clock around each call (every call ends in a synchronise);
  - per-stage device times of both from b200_ctx_set_profiling, in a pass of their own;
  - the per-call chain a caller had to run before this branch existed (host clock; every call synchronises):
    b200_cloud_create + b200_normals + b200_fpfh33 of the scene keypoints, b200_match, b200_cloud_create +
    b200_normals of the dense scene, b200_board_lrf of the model keypoints over the dense model (whose normals are
    computed once, outside the clock) and of the scene keypoints, b200_hough3d_recognize;
  - the pipeline's outputs against that chain on every scene: descriptors, correspondences, scene frames, instances
    and transforms, byte for byte.  A mismatch sets the exit code.
The clouds fit in L2 (126 MB) and are not flushed between calls: these are warm-cache figures.  Writes one JSON file.

usage: python profiles/bench_fpfh_hough.py [--pool 4] [--rounds 5] [--out profiles/r03/bench_fpfh_hough.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "3d-object-detection-of-industrial-joints_b200"
R = 0.05
SURFACE_K = 50


def device_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else None
    except (OSError, subprocess.SubprocessError, IndexError):
        info["nvidia_smi"] = None
    return info


def stats(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "n": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pool", type=int, default=4, help="distinct scenes (scene ids 1 .. pool)")
    ap.add_argument("--rounds", type=int, default=5, help="timed passes over the pool")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "bench_fpfh_hough.json"))
    args = ap.parse_args()

    synth = importlib.import_module(PKG + ".synth")
    binding = importlib.import_module(PKG + ".binding")
    model = synth.make_model("y", 5000)
    kpm = synth.voxel_grid(model, 0.01)
    scenes = [synth.make_scene(("y",), 100000, scene_id=s) for s in range(1, args.pool + 1)]
    kps = [synth.voxel_grid(s, 0.01) for s in scenes]
    p = binding.shot_params(normal_k=0, normal_radius=R, descr_radius=R, match_mode=2, match_thr=0.0, gc_size=0.02,
                            gc_threshold=3, max_instances=1 << 16)
    h = binding.hough_params(rf_radius=0.02, bin_size=0.02, threshold=2.0)

    ctx = binding.Context(0)   # a fresh context: the model's frames draw after srand(1)
    m_gc = ctx.model_create_fpfh(kpm, p)
    m_h = ctx.model_create_fpfh_hough(model, kpm, p, h, surface_normal_k=SURFACE_K)
    run = {"gc": lambda i: ctx.register_scene_fpfh(m_gc, kps[i], p, want_desc=True),
           "hough": lambda i: ctx.register_scene_fpfh_hough(m_h, scenes[i], kps[i], p, h, surface_normal_k=SURFACE_K,
                                                            want_desc=True)}
    for i in range(args.pool):   # warm-up: every scene with both branches
        for kind in ("gc", "hough"):
            run[kind](i)

    # ---- host clock around each call, alternating the branches scene by scene
    lat = {"gc": [], "hough": []}
    for r in range(args.rounds):
        for i in range(args.pool):
            for kind in (("gc", "hough") if (r + i) % 2 == 0 else ("hough", "gc")):
                t0 = time.perf_counter()
                run[kind](i)
                lat[kind].append((time.perf_counter() - t0) * 1e3)

    # ---- stage times, a pass of their own
    stages = {}
    ctx.set_profiling(True)
    for kind in ("gc", "hough"):
        ctx.reset_profiling()
        for i in range(args.pool):
            run[kind](i)
        stages[kind] = {n: ms / args.pool for n, (ms, c) in ctx.stage_times().items() if c > 0}
    ctx.set_profiling(False)

    # ---- the per-call chain, and the pipeline's outputs against it on every scene
    fm = m_h.download()[0]
    cc = binding.Context(0)
    cm = cc.cloud(model)
    nm = cc.normals(cm, k=SURFACE_K)

    def chain(i):
        cc.srand(1)
        ck = cc.cloud(kps[i])
        fs = cc.fpfh33(ck, cc.normals(ck, radius=R), R)
        corrs = cc.match(fm, fs, 2, 0.0)
        cs = cc.cloud(scenes[i])
        ns = cc.normals(cs, k=SURFACE_K)
        mrf = cc.board_lrf(cm, nm, kpm, h.rf_radius, h.board)
        srf = cc.board_lrf(cs, ns, kps[i], h.rf_radius, h.board)
        T, inst, n = cc.hough3d_recognize(kpm, mrf, kps[i], srf, corrs, h.bin_size, h.threshold, max_inst=p.max_instances)
        ck.close()
        cs.close()
        return fs, corrs, srf, T, inst, n

    for i in range(args.pool):   # warm-up
        chain(i)
    chain_ms, parity = [], []
    for r in range(args.rounds):
        for i in range(args.pool):
            t0 = time.perf_counter()
            out = chain(i)
            chain_ms.append((time.perf_counter() - t0) * 1e3)
            if r == 0:
                fs, corrs, srf, T, inst, n = out
                res = run["hough"](i)
                check = {"status": res["status"] == binding.OK,
                         "desc": np.array_equal(res["desc"], fs, equal_nan=True),
                         "corrs": res["corrs"].tobytes() == corrs.tobytes(),
                         "rf": np.array_equal(res["rf"], srf, equal_nan=True),
                         "n_instances": res["n_instances"] == n,
                         "transforms": res["transforms"].shape == T.shape and np.array_equal(res["transforms"], T),
                         "instances": len(res["instances"]) == len(inst) and
                                      all(a.tobytes() == b.tobytes() for a, b in zip(res["instances"], inst))}
                same_rf = (res["rf"] == srf) | (np.isnan(res["rf"]) & np.isnan(srf))
                parity.append({"scene_id": i + 1, "points": len(scenes[i]), "K_scene": len(kps[i]),
                               "correspondences": len(corrs), "instances": int(n),
                               "equal_to_chain": all(check.values()), "checks": check,
                               "rf_rows_differing": int((~same_rf).any(axis=1).sum()) if same_rf.ndim == 2 else -1})

    res = {
        "device": device_info(),
        "workload": "BASELINE config 2: %d-pt Y-joint model (%d keypoints), %d scenes of %d points (scene ids 1-%d, "
                    "%d-%d keypoints), voxel_grid 0.01, radius normals + FPFH33 r=%.2f on the keypoint clouds, k=2 ratio "
                    "test; Hough: BOARD r=%.2f find_holes over the dense clouds (k=%d normals), bin %.2f, threshold %g; "
                    "GC: 0.02 / 3" % (len(model), len(kpm), args.pool, len(scenes[0]), args.pool,
                                      min(map(len, kps)), max(map(len, kps)), R, h.rf_radius, SURFACE_K, h.bin_size,
                                      h.threshold),
        "clock": "host clock around host-buffer calls that end in a synchronise; L2 not flushed (the clouds fit in it)",
        "ms_per_scene": {k: stats(v) for k, v in lat.items()},
        "stage_ms_per_scene": stages,
        "per_call_chain_ms": stats(chain_ms),
        "pipeline_equals_chain": parity,
    }
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "ms_per_scene", "per_call_chain_ms")}))
    print("stages:", json.dumps(stages))
    ok = all(x["equal_to_chain"] for x in parity)
    print("pipeline == chain:", ok, [(x["scene_id"], x["equal_to_chain"], x["rf_rows_differing"]) for x in parity])
    for c in (cc, ctx):
        c.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
