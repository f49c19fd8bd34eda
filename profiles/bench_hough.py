"""First figures of the resident Hough branch (BOARD frames + Hough3DGrouping inside scene registration).

Workload: bench.py's target scenes, model and PARAMS (1 M-point Kinect-like scenes, about 91 000 keypoints, against
the 50 000-point Y-joint model) with the reference's Hough settings (SHOT_scenes.cpp:54-55: BOARD radius 0.02 with
find_holes, bin 0.02, threshold 2).  In one run, alternating so that both see the same machine state:
  - single-scene latency (one lane, device events, L2 overwritten between scenes) with per-stage device times, for the
    Hough branch and for the geometric-consistency (GC) pipeline;
  - throughput with `--lanes` scenes in flight over `--pool` distinct scenes, a 256 MiB L2 flush before every scene
    inside the timed region (as bench.py), Hough and GC;
  - the per-call chain a caller had to run before this branch existed: b200_register_scene_shot (for the
    correspondences), b200_cloud_create + b200_normals of the scene, b200_board_lrf of the model and of the scene,
    b200_hough3d_recognize (host clock; every call ends in a synchronise).
The pipeline's outputs are checked against that chain on every scene of the pool: correspondences, instances and
transforms byte for byte (the exit code), the scene frames row by row ("rf_rows_differing": BOARD's float64 plane-fit
sums follow the order in which a grid build left the points of a cell, so a frame can differ in its last bit between two
builds of the same cloud, about one row in 50 000 on these scenes; DESIGN §7).  Writes one JSON file (--out).

usage: python profiles/bench_hough.py [--lanes 8] [--pool 8] [--rounds 3] [--steps 4] [--out profiles/r03/bench_hough.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload, PARAMS: the benchmark's own definitions, read only)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=8)
    ap.add_argument("--pool", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3, help="alternating GC / Hough rounds of each measurement")
    ap.add_argument("--steps", type=int, default=4, help="scenes per lane in one throughput round")
    ap.add_argument("--scene-points", type=int, default=1_000_000)
    ap.add_argument("--model-points", type=int, default=50_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "bench_hough.json"))
    args = ap.parse_args()

    import torch
    binding = __import__("importlib").import_module(bench.PKG + ".binding")
    sharding = __import__("importlib").import_module(bench.PKG + ".sharding")
    dev = torch.device("cuda", 0)
    P, L = args.pool, args.lanes
    pool = [bench.workload(i, args.scene_points, args.model_points) for i in range(P)]
    wl = pool[0]
    p = binding.shot_params(**bench.PARAMS)
    h = binding.hough_params(rf_radius=0.02, bin_size=0.02, threshold=2.0)

    streams = [torch.cuda.Stream(device=dev) for _ in range(L)]
    ctxs = [binding.Context(0, stream=st.cuda_stream) for st in streams]
    ctx = ctxs[0]
    model_gc = ctx.model_create_shot(wl["model"], wl["model_kp"], p)
    model_h = ctx.model_create_shot_hough(wl["model"], wl["model_kp"], p, h)   # fresh context: srand(1)
    ctx.sync()
    d_scenes = [torch.from_numpy(w["scene"]).to(dev) for w in pool]
    d_kps = [torch.from_numpy(w["scene_kp"]).to(dev) for w in pool]
    Ns, Kss = [len(w["scene"]) for w in pool], [len(w["scene_kp"]) for w in pool]
    Ks_max, mi = max(Kss), p.max_instances

    def make_out():
        z = lambda *shape, dt=torch.int32: torch.zeros(*shape, dtype=dt, device=dev)
        return {"transforms": z(mi * 16, dt=torch.float32), "inst_offsets": z(mi + 1), "inst_counts": z(mi),
                "inst_corrs": z(Ks_max, 3), "corr_cap": Ks_max, "n_inst": z(1), "corrs": z(Ks_max, 3), "n_corrs": z(1),
                "rf": z(Ks_max, 9, dt=torch.float32), "status": z(1)}

    outs = [make_out() for _ in range(L)]
    flushes = [torch.empty(256 << 20, dtype=torch.uint8, device=dev) for _ in range(L)]
    torch.cuda.synchronize()

    def step(kind, lane, s, flush=False):
        i = s % P
        with torch.cuda.stream(streams[lane]):
            if flush:
                flushes[lane].zero_()
            if kind == "gc":
                ctxs[lane].dev_register_scene_shot(model_gc, d_scenes[i], Ns[i], 3, d_kps[i], Kss[i], 3, p, outs[lane])
            else:
                ctxs[lane].dev_register_scene_shot_hough(model_h, d_scenes[i], Ns[i], 3, d_kps[i], Kss[i], 3, p, h,
                                                         outs[lane])

    # warm-up: every lane meets every scene of the pool with both branches
    for kind in ("gc", "hough"):
        sharding.run_lanes(L, 2 * P * L, lambda lane, s: step(kind, lane, s))
    torch.cuda.synchronize()

    # ---- single-scene latency + stage times, one lane, alternating
    lat = {"gc": [], "hough": []}
    stages = {"gc": {}, "hough": {}}
    ctx.set_profiling(True)
    for r in range(args.rounds):
        for kind in ("gc", "hough"):
            ctx.reset_profiling()
            for s in range(P):
                with torch.cuda.stream(streams[0]):
                    flushes[0].zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(streams[0])
                step(kind, 0, s)
                b.record(streams[0])
                torch.cuda.synchronize()
                lat[kind].append(a.elapsed_time(b))
            for name, (ms, n) in ctx.stage_times().items():
                if n > 0:
                    stages[kind].setdefault(name, []).append(ms / P)
    ctx.set_profiling(False)

    # ---- throughput, L lanes, alternating
    thr = {"gc": [], "hough": []}
    n_steps = args.steps * L
    single = {k: float(np.median(v)) for k, v in lat.items()}
    for r in range(args.rounds):
        for kind in ("gc", "hough"):
            torch.cuda.synchronize()
            ev0 = torch.cuda.Event(enable_timing=True)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(L)]
            ev0.record(streams[0])
            sharding.run_lanes(L, n_steps, lambda lane, s: step(kind, lane, s, flush=True),
                               stagger_s=single[kind] / 1e3 / L)
            for l in range(L):
                evs[l].record(streams[l])
            torch.cuda.synchronize()
            thr[kind].append(max(ev0.elapsed_time(e) for e in evs) / n_steps)

    # ---- per-call chain, and the pipeline's outputs against it on every scene of the pool
    chain_ms, parity = [], []
    cc = binding.Context(0)
    cm = cc.cloud(wl["model"])
    nm = cc.normals(cm, k=bench.PARAMS["normal_k"])
    for s in range(P):
        w = pool[s]
        cc.srand(1)   # the pipeline's model was made on a fresh context: its scenes draw after srand(1) + model frames
        cc.sync()
        t0 = time.perf_counter()
        gc = cc.register_scene_shot(model_gc, w["scene"], w["scene_kp"], p)
        cs = cc.cloud(w["scene"])
        ns = cc.normals(cs, k=bench.PARAMS["normal_k"])
        mrf = cc.board_lrf(cm, nm, w["model_kp"], h.rf_radius, h.board)
        srf = cc.board_lrf(cs, ns, w["scene_kp"], h.rf_radius, h.board)
        T, inst, n = cc.hough3d_recognize(w["model_kp"], mrf, w["scene_kp"], srf, gc["corrs"], h.bin_size, h.threshold,
                                          max_inst=mi)
        chain_ms.append((time.perf_counter() - t0) * 1e3)
        cs.close()
        step("hough", 0, s)
        torch.cuda.synchronize()
        o = outs[0]
        m = min(int(o["n_inst"].item()), mi)
        nc = int(o["n_corrs"].item())
        offs, cnts = o["inst_offsets"][:m + 1].cpu().numpy(), o["inst_counts"][:m].cpu().numpy()
        ic = o["inst_corrs"].cpu().numpy().view(binding.CORR_DTYPE).reshape(-1)
        prf = o["rf"][:Kss[s]].cpu().numpy()
        PT = o["transforms"][:m * 16].cpu().numpy().reshape(m, 4, 4)
        check = {"n_instances": int(o["n_inst"].item()) == n,
                 "corrs": o["corrs"][:nc].cpu().numpy().view(binding.CORR_DTYPE).reshape(-1).tobytes() == gc["corrs"].tobytes(),
                 "rf": np.array_equal(prf, srf, equal_nan=True),
                 "transforms": PT.shape == T.shape and np.array_equal(PT, T),
                 "instances": all(ic[offs[i]:offs[i] + cnts[i]].tobytes() == inst[i].tobytes() for i in range(m))}
        parity.append({"scene": s, "K_scene": Kss[s], "correspondences": nc, "instances": int(o["n_inst"].item()),
                       "equal_to_chain": all(v for k, v in check.items() if k != "rf"), "checks": check,
                       "rf_rows_differing": int((~((prf == srf) | (np.isnan(prf) & np.isnan(srf)))).any(axis=1).sum())
                       if prf.shape == srf.shape else -1})

    res = {
        "device": device_info(),
        "workload": "bench.py target: %d-pt Kinect-like scenes (pool of %d), %d-pt Y-joint model, %d model keypoints, "
                    "%d-%d scene keypoints" % (Ns[0], P, len(wl["model"]), model_h.size, min(Kss), max(Kss)),
        "params": {"shot": bench.PARAMS, "hough": {"rf_radius": h.rf_radius, "find_holes": h.board.find_holes,
                                                   "bin_size": h.bin_size, "threshold": h.threshold}},
        "single_scene_ms": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
                            for k, v in lat.items()},
        "stage_ms_per_scene": {k: {n: float(np.median(v)) for n, v in st.items()} for k, st in stages.items()},
        "lanes": L,
        "throughput_ms_per_scene": {k: {"rounds": v, "median": float(np.median(v))} for k, v in thr.items()},
        "per_call_chain_ms": {"median": float(np.median(chain_ms)), "all": chain_ms},
        "pipeline_equals_chain": parity,
        "l2": "256 MiB written before every scene (inside the timed region in the lanes pass, outside it in the "
              "single-lane pass)",
    }
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "single_scene_ms", "throughput_ms_per_scene", "per_call_chain_ms")}))
    print("stages:", json.dumps(res["stage_ms_per_scene"]))
    print("pipeline == chain:", all(x["equal_to_chain"] for x in parity))
    for c in ctxs + [cc]:
        c.close()
    return 0 if all(x["equal_to_chain"] for x in parity) else 1


if __name__ == "__main__":
    sys.exit(main())
