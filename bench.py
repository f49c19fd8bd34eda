#!/usr/bin/env python
"""bench.py — SHOT registration hot path on B200 (contract: see the task statement / DESIGN.md §5).

A "step" is one pass of the hot path over one scene per rank: normals (k=20) → SHOT352 (r=0.02) at the
scene keypoints → correspondence search against the resident model descriptor library (k=1,
d2<0.25) → geometric-consistency grouping + RANSAC poses (0.02 / 2); parameters of SHOT_scenes.cpp
(:50-55, :286, :360).  Workload = BASELINE.json's target run: a 1 M-point Kinect-like synthetic scene
with three joints against a 50 k-point Y-joint model.

  value  : SHOT descriptors/s through the whole step, inputs resident in HBM (device-timed)
  e2e    : the same through the host-buffer C-ABI call (b200_register_scene_shot), pinned host
           buffers in, host results out, copies inside the timed region
  --impl reference : the CPU restatement of the reference's PCL path (oracle/) on the host cores,
           on a bounded sample of the same workload
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "3d-object-detection-of-industrial-joints_b200"
METRIC = "SHOT descriptors/s + scene registrations/s at 1-8 B200 vs PCL OMP host CPU"

PARAMS = dict(normal_k=20, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
              max_instances=4096)
MODEL_SS, SCENE_SS = 0.005, 0.01


_REAL_STDOUT = None

# DRAM read + write bytes per launch of each stage's main kernel, from the committed `ncu --set full` capture of the
# default workload (profiles/summary_r02.md)
TRAFFIC_NCU = {"match_filter": 83.2e6 + 33.0e6, "gc_group": 25.7e6, "gc_ransac": 2.0e6,
               "match": 83.2e6 + 33.0e6 + 147.8e6 + 6.4e6, "normals": 36.5e6, "shot": 128.1e6, "gc_adjacency": 52.4e6,
               "gc_sort": 1.0e6, "neighbor_count": 17.8e6}


def _emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 62_000_000   # payload of --dump-outputs: with the .npy headers the files stay under 64 MB


def registration_outputs(out, binding):
    """Host copies of what one dev_register_scene_shot call left in `out`, cut to the valid rows.  Correspondences
    are (index_query, index_match, distance) rows in float64, which holds both int32 and float32 exactly."""
    def corr_rows(t, n):
        c = t[:n].cpu().numpy().view(binding.CORR_DTYPE).reshape(-1)
        return np.stack([c["index_query"], c["index_match"], c["distance"]], axis=1).astype(np.float64)

    m = min(int(out["n_inst"].item()), PARAMS["max_instances"])
    off = out["inst_offsets"][:m + 1].cpu().numpy()
    return {"corrs": corr_rows(out["corrs"], int(out["n_corrs"].item())),
            "transforms": out["transforms"][:m * 16].cpu().numpy().reshape(m, 4, 4),
            "inst_offsets": off.astype(np.float64),
            "inst_counts": out["inst_counts"][:m].cpu().numpy().astype(np.float64),
            "inst_corrs": corr_rows(out["inst_corrs"], min(int(off[-1]), out["corr_cap"]))}


def dump_outputs(out_dir, arrays):
    """Writes name -> array as out_dir/<name>.npy.  Above DUMP_BYTES in all, every array keeps the same fraction of
    its rows, picked with a fixed seed, so that two builds with equally long outputs write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    frac = min(1.0, DUMP_BYTES / total) if total else 1.0
    for name, a in arrays.items():
        if frac < 1.0 and len(a) > 1:
            keep = max(1, int(len(a) * frac))
            a = a[np.sort(np.random.Generator(np.random.PCG64(0)).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload(scene_id, scene_points, model_points):
    synth = importlib.import_module(PKG).synth
    model = synth.make_model("y", model_points)
    scene = synth.make_kinect_scene(("y", "diagonal", "horizontal"), target_points=scene_points, scene_id=scene_id)
    return dict(model=model, scene=scene, model_kp=synth.uniform_sampling(model, MODEL_SS),
                scene_kp=synth.uniform_sampling(scene, SCENE_SS))


def config_dict(args, wl, world, scenes_per_step=None):
    synth = importlib.import_module(PKG).synth
    return {
        "workload": "SHOT_scenes pipeline, north-star target: %d-pt Kinect-like scene (Y+diagonal+horizontal joints) "
                    "vs %d-pt Y-joint model; a step = one batch of scene registrations (distinct scenes, round-robin)"
                    % (len(wl["scene"]), len(wl["model"])),
        "params": {"normals_k": 20, "uniform_sampling": {"model": MODEL_SS, "scene": SCENE_SS}, "shot_radius": 0.02,
                   "match": "k=1, d2<0.25", "gc": {"size": 0.02, "threshold": 2}},
        "N_scene": int(len(wl["scene"])), "N_model": int(len(wl["model"])), "K_scene": int(len(wl["scene_kp"])),
        "K_model": int(len(wl["model_kp"])), "shapes": synth.SHAPE_INFO,
        "scenes_per_step": scenes_per_step if scenes_per_step is not None else world,
        "scene_pool_per_rank": getattr(args, "pool", 1),
        "parallelism": "scene-sharded x%d (every rank registers its own distinct scenes), model library replicated, "
                       "NCCL gather of each scene's correspondence list; %d scenes in flight per GPU (lanes)"
                       % (world, args.lanes),
        "lanes_per_gpu": args.lanes,
        "host_waits": "blocking events" if getattr(args, "blocking", False) else "spinning",
        "l2": "256 MiB buffer written on the scene's stream before every scene registration, inside the timed region "
              "(lanes pass); between scenes, outside the timed intervals, in the single-lane pass",
    }


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
def cpu_full_pass(wl, threads=None, serial_sample=1500):
    """The reference path (CPU restatement, oracle/) on ONE COMPLETE scene, nothing sampled: normals of every
    point (OpenMP, as NormalEstimationOMP), SHOT352 at every scene keypoint (OpenMP, as SHOTEstimationOMP), the
    correspondence loop over every scene descriptor against the full model library, geometric-consistency grouping +
    RANSAC.  The reference's matching loop is serial (SHOT.cpp:409-423); run serially it alone takes minutes on this
    workload, so the measured pass parallelises it with OpenMP (faster than the reference, i.e. a stronger baseline)
    and the serial loop is timed on `serial_sample` scene descriptors and extrapolated, labelled as an estimate.
    Returns (measured seconds, detail)."""
    from oracle import pcl_oracle as orc
    orc.set_num_threads(threads or os.cpu_count() or 1)
    scene, kp = wl["scene"], wl["scene_kp"]
    t0 = time.perf_counter()
    nrm = orc.normals(scene, k=PARAMS["normal_k"])
    t1 = time.perf_counter()
    desc, _ = orc.shot352(scene, nrm, kp, PARAMS["descr_radius"])
    t2 = time.perf_counter()
    corr = orc.match(wl["model_desc"], desc, PARAMS["match_mode"], PARAMS["match_thr"], omp=True)
    t3 = time.perf_counter()
    T, _inst = orc.gc_recognize(wl["model_kp"], kp, corr, PARAMS["gc_size"], PARAMS["gc_threshold"],
                                max_inst=PARAMS["max_instances"])
    t4 = time.perf_counter()
    stride = max(1, len(kp) // max(serial_sample, 1))
    sub = np.ascontiguousarray(desc[::stride])
    t5 = time.perf_counter()
    orc.match(wl["model_desc"], sub, PARAMS["match_mode"], PARAMS["match_thr"])  # serial, as SHOT.cpp:409-423
    t6 = time.perf_counter()
    t_serial_est = (t6 - t5) * len(desc) / len(sub)
    measured = t4 - t0
    detail = {"t_normals_s": t1 - t0, "t_shot_s": t2 - t1, "t_match_omp_s": t3 - t2, "t_gc_s": t4 - t3,
              "measured_full_pass_s": measured, "correspondences": int(len(corr)), "instances": int(len(T)),
              "serial_match_sample_rows": int(len(sub)), "t_match_serial_sample_s": t6 - t5,
              "t_match_serial_est_s": t_serial_est,
              "est_full_pass_s_with_serial_matching": measured - (t3 - t2) + t_serial_est}
    return measured, detail


def model_descriptors_cpu(wl):
    from oracle import pcl_oracle as orc
    orc.set_num_threads(os.cpu_count() or 1)
    nrm = orc.normals(wl["model"], k=PARAMS["normal_k"])
    desc, _ = orc.shot352(wl["model"], nrm, wl["model_kp"], PARAMS["descr_radius"])
    return desc


def cpu_baseline_record(wl, measured, detail, cores):
    K = len(wl["scene_kp"])
    return {
        "value": K / measured, "unit": "descriptors/s", "cores": cores, "kind": "port",
        "sample": "ONE complete pass over scene 0 (%d points, %d keypoints vs %d model descriptors), nothing sampled or "
                  "extrapolated: normals + SHOT352 (OpenMP over points / keypoints as PCL's *OMP classes), matching loop "
                  "parallelised with OpenMP (the reference's loop is serial: that variant is estimated below from %d "
                  "rows), GC grouping + RANSAC serial; PCL-semantics restatement (oracle/), not libpcl" %
                  (len(wl["scene"]), K, len(wl["model_kp"]), detail["serial_match_sample_rows"]),
        "measured": True, "detail": detail,
        "value_with_serial_matching_estimate": K / detail["est_full_pass_s_with_serial_matching"],
    }


def run_reference(args, rank, world):
    """CPU arm: rank 0 alone, every host core, one measured un-sampled pass per invocation (a pass takes tens of
    seconds; repeating the identical pass K times would only burn the lease)."""
    if rank != 0:
        return
    from oracle import pcl_oracle as orc
    cores = os.cpu_count() or 1
    orc.set_num_threads(cores)   # explicitly: torchrun exports OMP_NUM_THREADS=1
    wl = workload(0, args.scene_points, args.model_points)
    wl["model_desc"] = model_descriptors_cpu(wl)  # resident library: untimed setup, like the GPU arm
    measured, detail = cpu_full_pass(wl, cores, args.cpu_sample)
    rec = cpu_baseline_record(wl, measured, detail, orc.num_threads())
    line = {
        "impl": "reference", "metric": METRIC, "value": rec["value"], "unit": "descriptors/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": measured * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
        "config": config_dict(args, wl, 1, scenes_per_step=1),
        "registrations_per_s": 1.0 / measured,
        "cpu_passes_timed": 1,
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": "descriptors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "PCL-semantics restatement (oracle/), not libpcl: PCL is neither vendored in the reference nor "
                "installed here or on the GPU box (profiles/pcl_probe_r02.txt).  ms_per_step is one complete scene "
                "registration on the CPU (the GPU arm's step holds several scenes: compare `value`, not ms_per_step); "
                "value uses an OpenMP matching loop, value_with_serial_matching_estimate the reference's serial loop",
    }
    _emit(line)


# --------------------------------------------------------------------------------------------------
# algorithmic bytes / flop per stage (SURVEY.md 8(d)); the kernel that carries the stage
STAGE_KERNEL = {"normals": "normals_knn_kernel", "shot": "shot_warp_kernel", "match_filter": "tc_filter_kernel",
                "gc_adjacency": "gc_adjacency_kernel", "gc_group": "gc_group_cluster_kernel",
                "gc_ransac": "gc_ransac_kernel", "gc_sort": "gc_rank_kernel",
                "neighbor_count": "shot_count_cov_kernel (+ shot_eigen_kernel)",
                "grid_build": "cell_count/scan/scatter kernels", "match": "tc_filter + tc_rescore + prep kernels"}


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module(PKG)
    binding = importlib.import_module(PKG + ".binding")
    sharding = importlib.import_module(PKG + ".sharding")
    binding.lib()  # fail loudly if the CUDA library is missing
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # Workload: every rank owns a pool of DISTINCT synthetic scenes (scene ids rank*P .. rank*P+P-1: different joint
    # poses, clutter and noise, so K_s, the correspondence count and the number of instances differ from scene to
    # scene and from rank to rank) and registers them round-robin against the replicated model library.
    P = max(1, args.pool)
    fixed_total = max(0, args.total_scenes)
    if fixed_total:
        # BASELINE config 5 as written: a fixed batch of scenes sharded over the ranks (scene g -> rank g mod world); the
        # batch cycles through P distinct scenes (generating hundreds of distinct scenes on the host would take minutes);
        # rank r's j-th scene is batch scene r + j * world
        base = [workload(i, args.scene_points, args.model_points) for i in range(P)]
        mine = [(rank + j * world) % P for j in range(P)]
        pool = [base[i] for i in mine]
    else:
        pool = [workload(rank * P + i, args.scene_points, args.model_points) for i in range(P)]
    wl = pool[0]
    p = binding.shot_params(**PARAMS)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    # Lanes: scenes are independent, so a rank keeps L of them in flight, each on its own context + stream +
    # host thread (sharding.run_lanes).  The grouping stage of one scene is a latency-bound chain on 8 SMs; the
    # other lanes' wide stages (normals, SHOT, matching) fill the rest of the GPU meanwhile.
    L = max(1, args.lanes)
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    # more lane threads than cores: the contexts wait on blocking events (the threads sleep) instead of spinning
    blocking = world * L > cores or args.blocking_sync
    args.lanes = L
    args.blocking = blocking
    B = L * max(1, args.scenes_per_lane)   # scene registrations per step and rank
    if fixed_total:
        B = max(1, fixed_total // world)   # this rank's share of the batch (every rank the same: one gather per scene)
    streams = [torch.cuda.Stream(device=dev) for _ in range(L)]
    ctxs = [binding.Context(local_rank, stream=st.cuda_stream) for st in streams]
    if blocking:
        for c in ctxs:
            c.set_blocking_sync(True)
    ctx = ctxs[0]
    with torch.cuda.stream(streams[0]):
        model = ctx.model_create_shot(wl["model"], wl["model_kp"], p)   # resident, replicated library (setup)
    ctx.sync()
    Km = model.size
    d_scenes = [torch.from_numpy(w["scene"]).to(dev) for w in pool]
    d_kps = [torch.from_numpy(w["scene_kp"]).to(dev) for w in pool]
    Ns = [len(w["scene"]) for w in pool]
    Kss = [len(w["scene_kp"]) for w in pool]
    Ks_max = max(Kss)
    mi = PARAMS["max_instances"]
    # the gather needs equally sized correspondence buffers on every rank (scenes differ in K_s)
    corr_cap_all = sharding.common_capacity(Ks_max, device=dev) if world > 1 else Ks_max

    def make_out():
        return {"transforms": torch.zeros(mi * 16, dtype=torch.float32, device=dev),
                "inst_offsets": torch.zeros(mi + 1, dtype=torch.int32, device=dev),
                "inst_counts": torch.zeros(mi, dtype=torch.int32, device=dev),
                "inst_corrs": torch.zeros((Ks_max, 3), dtype=torch.int32, device=dev), "corr_cap": Ks_max,
                "n_inst": torch.zeros(1, dtype=torch.int32, device=dev),
                "corrs": torch.zeros((corr_cap_all, 3), dtype=torch.int32, device=dev),
                "n_corrs": torch.zeros(1, dtype=torch.int32, device=dev)}

    outs = [make_out() for _ in range(L)]
    flushes = [torch.empty(256 << 20, dtype=torch.uint8, device=dev) for _ in range(L)]
    out = outs[0]
    gate = sharding.Turnstile()   # collectives are issued in global step order on every rank
    torch.cuda.synchronize()

    def step(lane, s, flush=False):
        i = s % P
        with torch.cuda.stream(streams[lane]):
            if flush:
                flushes[lane].zero_()
            ctxs[lane].dev_register_scene_shot(model, d_scenes[i], Ns[i], 3, d_kps[i], Kss[i], 3, p, outs[lane])
            if world > 1:   # the path's one exchange: gather the correspondence lists (NCCL over NVLink)
                gate.run(s, lambda: sharding.gather_correspondences(outs[lane]["corrs"], outs[lane]["n_corrs"]))

    # warm-up: every lane meets each of the scenes it will see in the timed passes at least twice (its arena grows to
    # the largest of them), then lane 0 walks the whole pool once for the single-lane pass
    gate.reset()
    sharding.run_lanes(L, max(args.warmup, 3, 2 * P) * L, step)
    torch.cuda.synchronize()
    if world == 1:
        for s in range(P):
            step(0, s)
        torch.cuda.synchronize()

    # ---- pass A, one lane: per-scene latency and the per-stage device times (roofline attribution) ----
    stream = streams[0]
    ctx.set_profiling(True)
    ctx.reset_profiling()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_begin = time.time()
    n_single = max(2 * P, 8)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(n_single)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(n_single)]
    per_scene = {}
    gate.reset()
    for s in range(n_single):
        with torch.cuda.stream(stream):
            flushes[0].zero_()
            starts[s].record(stream)
        step(0, s)
        ends[s].record(stream)
        if s < P:
            torch.cuda.synchronize()
            per_scene[s] = {"N": Ns[s], "K_scene": Kss[s], "correspondences": int(out["n_corrs"].item()),
                            "instances": int(out["n_inst"].item())}
    torch.cuda.synchronize()
    step_ms = [a.elapsed_time(b) for a, b in zip(starts, ends)]
    stages = ctx.stage_times()
    fb_rows, p1_rows = ctx.match_fallback_rows(), ctx.match_pass1_rows()
    ctx.set_profiling(False)
    mean_nbrs, max_nbrs = ctx.neighbor_stats()
    single_ms = float(np.median(step_ms))  # median: one scene of a multi-rank run may wait for a slow peer's gather

    # ---- pass B, L lanes: the throughput the metric is quoted on.  One start event when the device is idle,
    # one end event per lane stream; the L2 flush (256 MiB write) runs before every scene INSIDE the timed region
    n_scene_steps = args.steps * B
    gate.reset()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = sum(c.launches for c in ctxs)
    ev_start = torch.cuda.Event(enable_timing=True)
    ev_ends = [torch.cuda.Event(enable_timing=True) for _ in range(L)]
    ev_start.record(streams[0])
    stagger = single_ms / 1e3 / L   # inside the timed region: lane l starts l/L of a scene latency late
    sharding.run_lanes(L, n_scene_steps, lambda lane, s: step(lane, s, flush=True), stagger_s=stagger)
    for l in range(L):
        ev_ends[l].record(streams[l])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end)
    total_ms = max(ev_start.elapsed_time(e) for e in ev_ends)
    launches = sum(c.launches for c in ctxs) - launches0
    desc_done = float(sum(Kss[s % P] for s in range(n_scene_steps)))
    if args.dump_outputs and rank == 0:
        # lane l ran scenes l, l + L, ... of the timed pass and its buffers hold the last of them; the lanes whose last
        # scene belongs to the last step (all of them when B >= L) hold the last registrations of that step
        last = [l for l in range(L) if l < n_scene_steps and l + L * ((n_scene_steps - 1 - l) // L) >= n_scene_steps - B]
        dump_outputs(args.dump_outputs, {"lane%d_%s" % (l, k): v for l in last
                                         for k, v in registration_outputs(outs[l], binding).items()})

    ms = total_ms / args.steps
    t = torch.tensor([ms, desc_done, single_ms], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_max, total_desc, single_ms_max = float(tmax[0]), float(tsum[1]), float(tmax[2])
    else:
        ms_max, total_desc, single_ms_max = ms, desc_done, single_ms
    total_s = ms_max * args.steps / 1e3

    # ---- end to end through the host-buffer C-ABI call: pinned host buffers, copies timed, same lanes ----
    h_scenes = [torch.from_numpy(w["scene"]).pin_memory() for w in pool]
    h_kps = [torch.from_numpy(w["scene_kp"]).pin_memory() for w in pool]
    hs, hk = [x.numpy() for x in h_scenes], [x.numpy() for x in h_kps]
    results = [None] * L
    truncated = [0]

    def e2e_step(lane, s):
        i = s % P
        results[lane] = ctxs[lane].register_scene_shot(model, hs[i], hk[i], p)
        if results[lane].get("truncated"):
            truncated[0] += 1
        if world > 1:
            with torch.cuda.stream(streams[lane]):
                gate.run(s, lambda: sharding.gather_correspondences(outs[lane]["corrs"], outs[lane]["n_corrs"]))

    gate.reset()
    sharding.run_lanes(L, 2 * L, e2e_step)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    gate.reset()
    t0 = time.perf_counter()
    sharding.run_lanes(L, n_scene_steps, e2e_step, stagger_s=stagger)
    torch.cuda.synchronize()
    e2e_total_s = time.perf_counter() - t0
    h2d = float(sum(hs[s % P].nbytes + hk[s % P].nbytes for s in range(n_scene_steps))) / args.steps
    res = results[0]
    d2h_scene = int(res["transforms"].nbytes + 4 * (len(res["instances"]) + 2) + 12 * len(res["corrs"]) +
                    12 * sum(len(i) for i in res["instances"]))
    te = torch.tensor([e2e_total_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_total_s = float(te[0])

    if rank == 0:
        N, Ks = Ns[0], Kss[0]
        n_corrs, n_inst = per_scene[0]["correspondences"], per_scene[0]["instances"]
        Nm = float(np.mean(Ns))
        Ksm = float(np.mean(Kss))
        Cm = float(np.mean([v["correspondences"] for v in per_scene.values()]))
        work = {
            "normals": ("hbm", 32.0 * Nm, "GB/s"),
            "shot": ("hbm", 1444.0 * Ksm + 32.0 * Nm, "GB/s"),
            "neighbor_count": ("hbm", 16.0 * Nm + 4.0 * Ksm, "GB/s"),
            "grid_build": ("hbm", 40.0 * Nm, "GB/s"),
            "match": ("tensor", 2.0 * Ksm * Km * 352, "TFLOP/s"),
            "match_filter": ("tensor", 2.0 * Ksm * Km * 352, "TFLOP/s"),   # nested in "match": the tcgen05 kernel alone
            "gc_adjacency": ("hbm", 32.0 * Cm + Cm * (Cm / 8.0), "GB/s"),
            "gc_group": ("hbm", 12.0 * Cm + 16.0 * (Ksm + Km), "GB/s"),
            "gc_sort": ("hbm", 12.0 * Cm * 2, "GB/s"),
            "gc_ransac": ("hbm", 12.0 * Cm, "GB/s"),
        }
        stage_ms = {k: (v[0] / n_single, v[1] / n_single) for k, v in stages.items() if v[1] > 0}
        kernel_total = sum(v[0] for k, v in stage_ms.items() if k != "match_filter")

        def roof(k):
            bound, units, unit = work[k]
            dur_s = stage_ms[k][0] / 1e3
            if bound == "hbm":
                achieved, peak = units / dur_s / 1e9, peaks.get("hbm_gbs", 6650.0)
            else:
                achieved, peak = units / dur_s / 1e12, peaks.get("bf16_tflops", 1650.0)
            r = {"kernel": STAGE_KERNEL.get(k, k), "stage": k, "bound": bound, "achieved": achieved, "peak": peak,
                 "unit": unit, "frac": achieved / peak, "traffic": TRAFFIC_NCU.get(k), "algorithmic_units": units,
                 "avg_ms": stage_ms[k][0], "share_of_scene_kernel_time": stage_ms[k][0] / kernel_total}
            if k in ("match", "match_filter"):
                r["note"] = ("algorithmic flop = 2*K_s*K_m*352 per scene; the tcgen05 filter issues one fp16 term for "
                             "every row plus three terms (hi/lo split) for the rows the first pass cannot certify; "
                             "exact FP32 rescoring + certificate make the result bit-identical to the FP32 search")
            return r

        # the roofline line is the kernel with the LARGEST DURATION per scene, whatever it is; the three largest follow
        order = sorted((k for k in stage_ms if k in work and k != "match"), key=lambda k: -stage_ms[k][0])
        roofline = roof(order[0])
        roofline.update({"traffic_source": "ncu --set full, profiles/summary_r02.md, per launch, default workload",
                         "peak_source": ("MEASURED_PEAKS.json (burst figures: kernel timed alone, single-lane pass)"
                                         if peaks else "fallback (B200_PROFILING.md)"),
                         "selection": "largest average duration per scene among all kernels of the step (CUDA-event "
                                      "pair around the stage on the launching stream, single-lane pass)"})
        roofline_top3 = [roof(k) for k in order[:3]]
        roofline_all = [roof(k) for k in sorted((k for k in stage_ms if k in work), key=lambda k: -stage_ms[k][0])]
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            wl["model_desc"], _ = model.download()
            from oracle import pcl_oracle as orc
            measured, detail = cpu_full_pass(wl, os.cpu_count(), args.cpu_sample)
            cpu_baseline = cpu_baseline_record(wl, measured, detail, orc.num_threads())
            # the same scene on both arms: the CPU pass must find what the device found
            cpu_baseline["agrees_with_gpu"] = {"correspondences": detail["correspondences"] == n_corrs,
                                               "instances": detail["instances"] == n_inst}
        line = {
            "metric": METRIC, "value": total_desc / total_s, "unit": "descriptors/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max, "higher_is_better": True,
            "scaling": "strong" if fixed_total else "weak", "vs_baseline": None,
            "dtype": "f32 (f64 for the SHOT frame/bin decisions)",
            "data": "synthetic",
            "config": config_dict(args, wl, world, scenes_per_step=fixed_total if fixed_total else B * world),
            "registrations_per_s": world * n_scene_steps / total_s,
            "timed_region_s": total_s,
            "lanes": L,
            "single_lane": {"ms_per_scene": single_ms_max, "value": Ksm / (single_ms_max / 1e3),
                            "note": "one scene in flight per GPU (per-scene latency, median of the listed scene_ms); stage times and the roofline "
                                    "entries are measured in this pass"},
            "e2e": {"value": total_desc / e2e_total_s, "unit": "descriptors/s",
                    "ms_per_step": e2e_total_s * 1e3 / args.steps, "timed_region_s": e2e_total_s,
                    "registrations_per_s": world * n_scene_steps / e2e_total_s, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h_scene * B), "truncated_results": truncated[0],
                    "api": "b200_register_scene_shot (host buffers, pinned), %d scenes per step" % B},
            "gpu_launches": int(launches),
            "gpu_launches_per_scene": launches / max(n_scene_steps, 1),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_top3": roofline_top3,
            "roofline_all_stages": roofline_all,
            "cpu_baseline": cpu_baseline,
            "stages_ms_per_scene": {k: round(v[0], 4) for k, v in stage_ms.items()},
            "match_filter_rows": {"left_by_one_term_pass": p1_rows, "left_to_exact_kernel": fb_rows},
            "measured": {"N": N, "K_scene": Ks, "K_model": Km, "mean_neighbors": mean_nbrs, "max_neighbors": max_nbrs,
                         "correspondences": n_corrs, "instances": n_inst, "scene_ms": [round(x, 3) for x in step_ms],
                         "pool": per_scene},
        }
        if args.other_configs and world == 1:
            try:
                line["other_configs"] = run_other_configs(ctx, binding, pkg, args)
            except Exception as e:  # the headline line must survive a failure of the side measurements
                line["other_configs"] = {"error": repr(e)}
        _emit(line)
    model.close()
    for c in ctxs:
        c.close()
    if world > 1:
        dist.destroy_process_group()


def run_sharded(args, rank, world, local_rank):
    """Strong scaling of ONE scene stream (north star: "scene keypoints are sharded across the GPUs"): every step is
    one b200_register_scene_shot_sharded call — the root holds the scene in pinned host memory, the library broadcasts
    it over NCCL, every rank computes the normals and its keypoint slab's descriptors + correspondences, the lists are
    gathered on the root, which groups them.  Total work is fixed as N grows.  Wall clock per call on the root
    (host buffers in, host results out), max over ranks."""
    import torch
    import torch.distributed as dist
    binding = importlib.import_module(PKG + ".binding")
    binding.lib()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = workload(0, args.scene_points, args.model_points)
    p = binding.shot_params(**PARAMS)
    ctx = binding.Context(local_rank)
    if world > 1:   # the library's own communicator; torch.distributed only carries the 128-byte token
        tok = [binding.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(tok, src=0)
        ctx.comm_init(tok[0], rank, world)
    model = ctx.model_create_shot(wl["model"], wl["model_kp"], p)
    hs = torch.from_numpy(wl["scene"]).pin_memory().numpy()
    hk = torch.from_numpy(wl["scene_kp"]).pin_memory().numpy()

    def call():
        if rank == 0:
            return ctx.register_scene_shot_sharded(model, p, hs, hk, root=0)
        return ctx.register_scene_shot_sharded(model, p, root=0)

    for _ in range(max(args.warmup, 3)):
        res = call()
    single = ctx.register_scene_shot(model, hs, hk, p) if rank == 0 else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_begin = time.time()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = call()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t[0])
    clocks = sampler.stop(t_begin, time.time())
    if rank == 0:
        same = (res["corrs"].tobytes() == single["corrs"].tobytes() and res["n_instances"] == single["n_instances"] and
                np.array_equal(res["transforms"], single["transforms"]) and
                all(a.tobytes() == b.tobytes() for a, b in zip(res["instances"], single["instances"])))
        Ks = len(wl["scene_kp"])
        _emit({"metric": METRIC, "mode": "sharded", "value": Ks * args.steps / dt, "unit": "descriptors/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3 / args.steps,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32 (f64 for the SHOT frame/bin decisions)", "data": "synthetic",
               "registrations_per_s": args.steps / dt,
               "config": {"workload": "ONE %d-pt scene (%d keypoints) per step vs the %d-descriptor model, keypoint "
                                      "slabs over %d GPU(s): b200_register_scene_shot_sharded, host buffers, one call in "
                                      "flight" % (len(wl["scene"]), Ks, model.size, world),
                          "l2": "inputs larger than L2 are re-uploaded and re-broadcast every step"},
               "identical_to_single_gpu_result": bool(same), "correspondences": int(len(res["corrs"])),
               "instances": int(res["n_instances"]), "clocks": clocks,
               "e2e": {"value": Ks * args.steps / dt, "unit": "descriptors/s",
                       "h2d_bytes_per_step": int(hs.nbytes + hk.nbytes),
                       "d2h_bytes_per_step": int(12 * len(res["corrs"]) + 64 * res["n_instances"])}})
    model.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def _timeit(fn, sync, reps, warm=2):
    for _ in range(warm):
        fn()
    sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        r = fn()
    sync()
    return (time.perf_counter() - t0) / reps, r


def run_other_configs(ctx, binding, pkg, args):
    """BASELINE.json configs 1, 2 and 4 through the host-buffer C ABI (host arrays in, host results out, copies inside
    the timed region), one scene in flight, with the CPU restatement of the same calls timed beside each on every host
    core.  Small cases: each takes a second or two."""
    from oracle import pcl_oracle as orc
    synth = pkg.synth
    orc.set_num_threads(os.cpu_count() or 1)
    out = {}
    model = synth.make_model("y", 5000)
    scene = synth.make_scene(("y",), 100000, scene_id=1)
    # ---- config 1: SHOT_demo pipeline (SHOT_demo.cpp:405-424, 497-531 + GC grouping), normals k=10, SHOT r=0.02
    kpm, kps = synth.voxel_grid(model, 0.02), synth.voxel_grid(scene, 0.03)
    p1 = binding.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=2,
                             max_instances=1024)
    m1 = ctx.model_create_shot(model, kpm, p1)
    t_gpu, res = _timeit(lambda: ctx.register_scene_shot(m1, scene, kps, p1), ctx.sync, 10)
    dm, _ = m1.download()
    m1.close()

    def cpu1():
        nrm = orc.normals(scene, k=10)
        ds, _ = orc.shot352(scene, nrm, kps, 0.02)
        c = orc.match(dm, ds, 1, 0.25)          # serial loop, as the reference
        T, inst = orc.gc_recognize(kpm, kps, c, 0.02, 2, max_inst=1024)
        return c, T
    t_cpu, (c_cpu, T_cpu) = _timeit(cpu1, lambda: None, 2, warm=0)
    out["config1_shot_demo"] = {
        "workload": "5000-pt Y-joint model (%d keypoints) vs 100000-pt scene (%d keypoints), normals k=10, SHOT r=0.02, "
                    "k=1 d2<0.25, GC 0.02/2" % (len(kpm), len(kps)),
        "descriptors_per_s": len(kps) / t_gpu, "registrations_per_s": 1.0 / t_gpu, "ms_per_scene_e2e": t_gpu * 1e3,
        "cpu": {"descriptors_per_s": len(kps) / t_cpu, "ms_per_scene": t_cpu * 1e3, "cores": orc.num_threads(),
                "kind": "port", "measured": True, "matching": "serial loop (as the reference)"},
        "same_correspondence_pairs_as_cpu": bool(
            np.array_equal(res["corrs"]["index_query"], c_cpu["index_query"]) and
            np.array_equal(res["corrs"]["index_match"], c_cpu["index_match"])),
        "same_instance_count_as_cpu": bool(res["n_instances"] == len(T_cpu)),
        "correspondences": int(len(res["corrs"])), "instances": int(res["n_instances"])}
    # ---- config 2: FPFH_demo (FPFH_demo.cpp:416-428, 505-538): radius normals + FPFH33 on the keypoint cloud,
    # k = 2 ratio matching, GC grouping; radius 0.05 as BASELINE.json states
    kq_m, kq_s = synth.voxel_grid(model, 0.01), synth.voxel_grid(scene, 0.01)
    r = 0.05

    p2 = binding.shot_params(normal_k=0, normal_radius=r, descr_radius=r, match_mode=2, match_thr=0.0, gc_size=0.02,
                             gc_threshold=3, max_instances=1024)
    m2 = ctx.model_create_fpfh(kq_m, p2)      # resident model side (b200_model_create_fpfh)

    def gpu2():
        return ctx.register_scene_fpfh(m2, kq_s, p2, want_desc=True)
    t_gpu2, res2 = _timeit(gpu2, ctx.sync, 5)
    fs_gpu, c_gpu, g_gpu = res2["desc"], res2["corrs"], (res2["transforms"],)
    # where the time goes (CUDA-event pairs around the stages of one more pass): the k = 2 ratio test of
    # FPFH_demo.cpp:530-532 accepts every scene descriptor, so the grouping sees one correspondence per scene point
    ctx.set_profiling(True)
    ctx.reset_profiling()
    gpu2()
    stages2 = {k: round(v[0], 3) for k, v in ctx.stage_times().items() if v[1] > 0}
    ctx.set_profiling(False)
    m2.close()

    fm_cpu = orc.fpfh33(kq_m, orc.normals(kq_m, radius=r), r)   # model side: untimed setup on both arms

    def cpu2():
        fs = orc.fpfh33(kq_s, orc.normals(kq_s, radius=r), r)
        c = orc.match(fm_cpu, fs, 2, 0.0)
        return fs, c
    t_cpu2_scene, (fs_cpu, c_cpu2) = _timeit(cpu2, lambda: None, 1, warm=0)
    ok = np.isfinite(fs_cpu[:, 0]) & np.isfinite(fs_gpu[:, 0])
    out["config2_fpfh_demo"] = {
        "workload": "FPFH33 r=%.2f on the voxel-filtered (0.01) clouds: %d model / %d scene points, radius normals, "
                    "k=2 ratio matching, GC 0.02/3" % (r, len(kq_m), len(kq_s)),
        "api": "b200_model_create_fpfh + b200_register_scene_fpfh (resident model, host buffers)",
        "descriptors_per_s": len(kq_s) / t_gpu2, "ms_per_scene_e2e": t_gpu2 * 1e3, "stages_ms": stages2,
        "descriptor_stages_ms": round(sum(stages2.get(k, 0.0) for k in ("grid_build", "normals", "neighbor_count", "fpfh",
                                                                         "match")), 3),
        "cpu": {"descriptors_per_s": len(kq_s) / t_cpu2_scene, "ms_per_scene": t_cpu2_scene * 1e3,
                "cores": orc.num_threads(), "kind": "port", "measured": True,
                "note": "scene side: normals + FPFH + matching (no grouping); FPFH via the OpenMP variant"},
        "descriptor_l2_vs_cpu": {"median": float(np.median(np.linalg.norm(fs_gpu[ok] - fs_cpu[ok], axis=1))),
                                 "max": float(np.linalg.norm(fs_gpu[ok] - fs_cpu[ok], axis=1).max()),
                                 "note": "each arm on its own normals: rows with an atan2f value within an ulp of a bin "
                                         "border move by one vote (tests/eps.py shows every differing row is one)"},
        "correspondences": int(len(c_gpu)), "instances": int(len(g_gpu[0]))}
    # ---- config 4: CAD_desc + partial views: 64 views x 3 joints in one resident library, one scene against all
    p4 = binding.shot_params(normal_k=10, descr_radius=0.02, match_mode=1, match_thr=0.25, gc_size=0.02, gc_threshold=3,
                             max_instances=512)
    lib = binding.Library(ctx)
    t0 = time.perf_counter()
    n_desc = 0
    for joint in ("y", "diagonal", "horizontal"):
        for v in range(64):
            cloud = synth.make_partial_view(joint, v, 4000)
            kp = synth.uniform_sampling(cloud, 0.02)
            lib.add_view(cloud, kp, p4)
            n_desc += len(kp)
    ctx.sync()
    t_build = time.perf_counter() - t0
    scene4 = synth.make_scene(("y", "diagonal", "horizontal"), 150000, scene_id=7)
    kps4 = synth.uniform_sampling(scene4, 0.03)
    t_gpu4, res4 = _timeit(lambda: lib.register_scene(scene4, kps4, p4, max_inst=98304), ctx.sync, 3, warm=1)
    lib.close()
    out["config4_view_library"] = {
        "workload": "192 partial views (64 x Y/diagonal/horizontal, %d library descriptors) vs a 150000-pt scene "
                    "(%d keypoints); scene normals + SHOT once, then per view: matching + GC grouping + poses"
                    % (n_desc, len(kps4)),
        "library_build_s_incl_host_synthesis": t_build, "registrations_per_s": 1.0 / t_gpu4,
        "ms_per_scene_e2e": t_gpu4 * 1e3, "view_matches_per_s": 192.0 / t_gpu4, "instances": int(res4["n_instances"])}
    # ---- the reference's DEFAULT grouping branch on config 1's clouds and correspondences (SHOT.cpp:433-470): BOARD
    # frames (find_holes, rf_rad 0.02) for the model and the scene keypoints, then Hough3DGrouping
    try:
        out["config1_hough_branch"] = run_hough_config(ctx, binding, orc, model, scene, kpm, kps, res["corrs"])
    except Exception as e:
        out["config1_hough_branch"] = {"error": repr(e)}
    # ---- the last gate of the reference's callback: GlobalHypothesesVerification on the registered instances
    # (SHOT_hypothesis.cpp:631-653), host buffers in, mask out, in the reference's call order
    try:
        out["hypothesis_verification"] = run_hv_config(ctx, binding, synth, orc)
    except Exception as e:  # an extra record must not cost the headline line
        out["hypothesis_verification"] = {"error": repr(e)}
    return out


def run_hough_config(ctx, binding, orc, model, scene, kpm, kps, corrs):
    cm, cs = ctx.cloud(model), ctx.cloud(scene)
    nm, ns = ctx.normals(cm, k=10), ctx.normals(cs, k=10)

    def gpu():
        ctx.srand(1)
        rf_m = ctx.board_lrf(cm, nm, kpm, 0.02)
        rf_s = ctx.board_lrf(cs, ns, kps, 0.02)
        T, inst, n = ctx.hough3d_recognize(kpm, rf_m, kps, rf_s, corrs, 0.03, 3.0, max_inst=1024)
        return rf_m, rf_s, n
    t_gpu, (rf_m, rf_s, n_gpu) = _timeit(gpu, ctx.sync, 5)
    cm.close()
    cs.close()

    def cpu():
        o_m, used = orc.board_lrf(model, nm, kpm, 0.02)
        o_s, _ = orc.board_lrf(scene, ns, kps, 0.02, rand_skip=used)
        T, inst = orc.hough3d_recognize(kpm, o_m, kps, o_s, corrs, 0.03, 3.0, max_inst=1024)
        return o_m, o_s, len(T)
    t_cpu, (o_m, o_s, n_cpu) = _timeit(cpu, lambda: None, 1, warm=0)
    ok = ~np.isnan(o_s[:, 0]) & ~np.isnan(rf_s[:, 0])
    return {"workload": "BOARD frames (find_holes, r = 0.02) of %d model + %d scene keypoints on config 1's clouds, "
                        "Hough3DGrouping (bin 0.03, threshold 3) on its %d correspondences; normals given"
                        % (len(kpm), len(kps), len(corrs)),
            "api": "b200_board_lrf x 2 + b200_hough3d_recognize (host buffers)",
            "ms_e2e": t_gpu * 1e3, "cpu": {"ms": t_cpu * 1e3, "cores": orc.num_threads(), "kind": "port", "measured": True},
            "instances": int(n_gpu), "cpu_instances": int(n_cpu),
            "scene_frames_within_1e-5_of_cpu": float((np.abs(rf_s[ok] - o_s[ok]).max(axis=1) < 1e-5).mean())}


def run_hv_config(ctx, binding, synth, orc):
    joints = ("y", "diagonal", "horizontal")
    scene, poses = synth.make_kinect_scene(joints, 400000, scene_id=0, return_poses=True)
    rng = np.random.Generator(np.random.PCG64(77))
    hyps = []
    for j, T in zip(joints, poses):   # per joint: the true pose, a 2 mm near-duplicate, a displaced copy
        m = synth.make_model(j, 20000).astype(np.float64)
        for dt in (np.zeros(3), rng.normal(0, 0.002, 3), np.array([0.04, -0.03, 0.05])):
            hyps.append((m @ T[:3, :3].T + T[:3, 3] + dt).astype(np.float32))
    kw = dict(detect_clutter=0, regularizer=3.0, radius_normals=0.02)

    def gpu():
        hv = ctx.hypothesis_verification(None)
        hv.set_scene(scene)
        hv.add_models(hyps, occlusion_reasoning=True)
        hv.set_params(binding.hv_params(**kw))
        r = hv.verify()
        hv.close()
        return r
    t_gpu, rg = _timeit(gpu, ctx.sync, 5)
    t_cpu, rc = _timeit(lambda: orc.hv_verify(scene, hyps, orc.hv_params(occlusion_reasoning=1, **kw)), lambda: None, 1,
                        warm=0)
    return {"workload": "%d hypotheses of 20000 points against a %d-point Kinect-like scene, occlusion reasoning, "
                        "inlier 0.005, normals r=0.02, regulariser 3" % (len(hyps), len(scene)),
            "api": "b200_hv_set_scene + b200_hv_add_models + b200_hv_set_params + b200_hv_verify (host buffers)",
            "ms_e2e": t_gpu * 1e3, "hypotheses_per_s": len(hyps) / t_gpu,
            "cpu": {"ms": t_cpu * 1e3, "cores": orc.num_threads(), "kind": "port", "measured": True},
            "mask": rg["mask"].astype(int).tolist(), "same_mask_as_cpu": bool(rg["mask"].tolist() == rc["mask"].tolist()),
            "best_cost": rg["best_cost"], "cpu_best_cost": rc["best_cost"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="batch", choices=["batch", "sharded"],
                    help="batch: independent scenes per rank (weak scaling, the headline); sharded: one scene stream "
                         "split over the ranks (strong scaling)")
    ap.add_argument("--scene-points", type=int, default=1_000_000)
    ap.add_argument("--model-points", type=int, default=50_000)
    ap.add_argument("--cpu-sample", type=int, default=1500, help="scene keypoints in the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--blocking-sync", action="store_true", help="contexts sleep in host waits instead of spinning")
    ap.add_argument("--lanes", type=int, default=8, help="scenes in flight per GPU (context + stream + host thread each)")
    ap.add_argument("--scenes-per-lane", type=int, default=8, help="a step = lanes x this many scene registrations per GPU")
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic scenes per rank, registered round-robin")
    ap.add_argument("--total-scenes", type=int, default=0,
                    help="BASELINE config 5: a fixed batch of this many scenes sharded over the ranks in one step (strong "
                         "scaling), e.g. --total-scenes 256 --scene-points 500000 --pool 8")
    ap.add_argument("--other-configs", type=int, default=1,
                    help="also measure BASELINE configs 1, 2 and 4 (small) and report them under other_configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the registrations of the last step returned as "
                         "DIR/lane<l>_<name>.npy (float32/float64, at most 64 MB), to compare two builds on the same "
                         "inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.mode != "batch"):
        ap.error("--dump-outputs applies to --impl b200 --mode batch")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner)
    # goes to stderr instead
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.mode == "sharded":
        run_sharded(args, rank, world, local_rank)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
