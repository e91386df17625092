#!/usr/bin/env python
"""bench.py — LIMO-Velo localization hot path on B200: matched-points/sec per IESKF iteration.

One "step" = one Localizator::correct (all <= MAX_NUM_ITERS+1 h-evaluations of the iterated update:
world transform -> exact 5-NN -> plane fit -> residual/Jacobian -> HtH/Hth -> 23-DoF IESKF step)
on one synthetic 64k-point Velodyne sweep against a 1M-point map (BASELINE.json configs[1],
config/xaloc.yaml).  Prints ONE JSON line (see the task contract); `--impl reference` times the CPU
oracle (reference ikd-Tree compiled verbatim into oracle/_ref + restated plane/Jacobian/IESKF).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as G  # noqa: E402

METRIC = "matched-points/sec per IESKF iteration (64k-pt sweep, 1M-pt map)"
UNIT = "point-evaluations/s"
SEED = 20260924
MAP_POINTS = 1_000_000
RINGS, AZIMUTHS = 64, 1024           # Velodyne-64 pattern: 65 536 beams
N_SWEEPS = 8                          # distinct sweeps along the road, replayed round-robin
ALGO_BYTES_PER_POINT = 72             # 12 B query + 5 x 12 B neighbours (SURVEY.md 8d)

# BASELINE.json `configs` (SURVEY.md 8d "concrete synthetic inputs").  The driver's line is cfg1 (the config the
# metric is quoted on); the others are run with --config and land in profiles/bench_<cfg>.json.
#   sub_sweeps  a sweep is cut into this many consecutive pieces (firing order = time order), one update each
#               (kitti.yaml: delta 0.01 s -> 10 updates per 0.1 s rotation, README.md:14)
#   max_iters   MAX_NUM_ITERS override (cfg0: a single h-evaluation)
#   planar      ground-only map (BASELINE.json configs[0])
CONFIGS = {
    "cfg0": dict(yaml="xaloc.yaml", map_points=100_000, rings=64, azimuths=1024, elev=(-24.8, 2.0), sub_sweeps=1,
                 max_iters=0, planar=True, seed_off=0,
                 what="single 64k-pt Velodyne sweep vs 100k-pt planar map, 1 evaluation"),
    "cfg1": dict(yaml="xaloc.yaml", map_points=MAP_POINTS, rings=RINGS, azimuths=AZIMUTHS, elev=(-24.8, 2.0), sub_sweeps=1,
                 max_iters=None, planar=False, seed_off=1,
                 what="xaloc.yaml, 65536-pt Velodyne-64 sweep vs 1000000-pt map, MAX_NUM_ITERS=3 (<=4 evaluations)"),
    "cfg2": dict(yaml="kitti.yaml", map_points=5_000_000, rings=64, azimuths=2048, elev=(-24.8, 2.0), sub_sweeps=10,
                 max_iters=None, planar=False, seed_off=2,
                 what="kitti.yaml, 131072-pt sweeps cut into 10 sub-sweeps of 13107 pts (delta 0.01 s) vs 5M-pt map"),
    "cfg3": dict(yaml="ouster.yaml", map_points=10_000_000, rings=128, azimuths=2048, elev=(-22.5, 22.5), sub_sweeps=1,
                 max_iters=None, planar=False, seed_off=3,
                 what="ouster.yaml, 262144-pt Ouster-128 sweep vs 10M-pt map"),
    "cfg4": dict(yaml="xaloc.yaml", map_points=MAP_POINTS, rings=RINGS, azimuths=AZIMUTHS, elev=(-24.8, 2.0), sub_sweeps=1,
                 max_iters=None, planar=False, seed_off=10, sequences=8,
                 what="8 independent cfg1-like sequences (65536-pt sweeps, 1M-pt maps), a FIXED job spread over the GPUs"),
}


def metric_name(cfg):
    return METRIC if cfg == "cfg1" else "matched-points/sec per IESKF iteration (%s: %s)" % (cfg, CONFIGS[cfg]["what"])


def update_points(cfg):
    c = CONFIGS[cfg]
    return (c["rings"] * c["azimuths"]) // c["sub_sweeps"]


def workload_config(n_gpus, cfg="cfg1", sequences=None):
    c = CONFIGS[cfg]
    return {"workload": "%s: %s" % (cfg, c["what"]),
            "sweep_points": update_points(cfg), "map_points": c["map_points"], "yaml": c["yaml"],
            "sequences": sequences if sequences is not None else n_gpus,
            "parallelism": "one independent sequence per GPU (no data-path collective)",
            "l2": "flushed (256 MiB write) between timed steps; step time = CUDA events around each update"}


def config_params(lv, cfg, **over):
    """lv_params of a config: its YAML + the capacities of its sizes (+ overrides)"""
    c = CONFIGS[cfg]
    n = update_points(cfg)
    kw = dict(max_map_points=c["map_points"] + 4 * c["rings"] * c["azimuths"], max_points=n)
    kw.update(over)
    prm = lv.params_from_yaml(os.path.join(lv.CONFIG_DIR, c["yaml"]), **kw)
    if c["max_iters"] is not None:
        prm.MAX_NUM_ITERS = c["max_iters"]
    return prm


def make_scene(lv, rank, n_sweeps=N_SWEEPS, prm=None, cfg="cfg1"):
    """Seeded world + updates (sweeps or sub-sweeps) + predicted states for one sequence
    (seed base + seed_off + 10 * rank: SURVEY 8d cfg0..cfg4).  Returns world, map, updates, x_props, truths."""
    O = G.load_oracle()
    c = CONFIGS[cfg]
    rng = np.random.default_rng(SEED + 1000 + rank + 100 * (c["seed_off"] - 1))
    world = lv.SynthWorld(SEED + c["seed_off"] + 10 * rank, c["map_points"] if not c["planar"] else 6 * c["map_points"])
    mp = world.map()
    n_upd = update_points(cfg)
    sweeps, x_props, truths = [], [], []
    if c["planar"]:
        # ground-only map: the map_points ground samples closest to the road position of the sweeps; sweeps keep
        # only the returns from that disc (ray-cast at 4x the azimuth density so that enough of them remain)
        centre = world.pose(15.0, prm)[0:3]
        ground = mp[mp[:, 2] < -1.6]
        d2 = ((ground[:, :2] - centre[:2].astype(np.float32)) ** 2).sum(1)
        keep = np.argsort(d2, kind="stable")[:c["map_points"]]
        radius = float(np.sqrt(d2[keep[-1]]))
        mp = np.ascontiguousarray(ground[np.sort(keep)])
    for i in range(n_sweeps):
        truth = world.pose(15.0 + 1.5 * i, prm)            # 15 m/s at 10 Hz
        if c["planar"]:
            truth = world.pose(15.0 + 0.25 * i, prm)       # stay inside the disc
            raw = world.sweep(truth, rings=c["rings"], azimuths=4 * c["azimuths"], elev=c["elev"], min_dist=4.0,
                              range_sigma=0.02, seed=100 + i)
            gw = world_points(raw, truth)
            ok = (gw[:, 2] < -1.5) & (((gw[:, :2] - centre[:2].astype(np.float32)) ** 2).sum(1) < (radius - 1.0) ** 2)
            sw = np.ascontiguousarray(raw[ok][:c["rings"] * c["azimuths"]])
            assert len(sw) == c["rings"] * c["azimuths"], "planar scene: not enough ground returns (%d)" % len(sw)
        else:
            sw = world.sweep(truth, rings=c["rings"], azimuths=c["azimuths"], elev=c["elev"], min_dist=4.0,
                             range_sigma=0.02, seed=100 + i)
        for k in range(c["sub_sweeps"]):
            sweeps.append(np.ascontiguousarray(sw[k * n_upd:(k + 1) * n_upd]))
            d = np.zeros(23)
            d[0:3] = rng.uniform(-0.05, 0.05, 3)
            d[3:6] = rng.uniform(-0.5, 0.5, 3) * np.pi / 180.0
            x_props.append(O.boxplus(truth, d))
            truths.append(truth)
    return world, mp, sweeps, x_props, truths


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def wait_first(self, timeout=3.0):
        """block until nvidia-smi delivers its first row (its start-up takes ~0.1 s), then mark the window start"""
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.005)
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.rows = self.rows[getattr(self, "first", 0):]
        time.sleep(0.03)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [s.strip() for s in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_params(O, prm):
    return O.make_params(max_num_iters=prm.MAX_NUM_ITERS, estimate_extrinsics=prm.estimate_extrinsics,
                         max_dist_plane=prm.MAX_DIST_PLANE, planes_threshold=prm.PLANES_THRESHOLD,
                         lidar_noise=prm.LiDAR_noise, degeneracy_threshold=prm.degeneracy_threshold,
                         limits=list(prm.LIMITS))


_OUT_FD = None


def _emit(line):
    """The ONE JSON line, on the stdout this process was started with.  Everything else that writes to fd 1 while the bench runs
    (NCCL's version banner under torchrun, the reference ikd-Tree's thread messages) has been pointed at stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _OUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_OUT_FD, data)


class _StdoutToStderr:
    """The reference's ikd-Tree announces its rebuild thread on C stdout ("Multi thread started");
    keep this process' stdout clean for the ONE JSON line by pointing fd 1 at fd 2 meanwhile."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def cpu_leg(lv, prm, mp, sweeps, x_props, P0, budget_s, threads, max_updates=None):
    with _StdoutToStderr():
        out = _cpu_leg(lv, prm, mp, sweeps, x_props, P0, budget_s, threads, max_updates)
        import gc
        gc.collect()              # the oracle map (and the ikd-Tree's farewell message) goes here
    return out


def _cpu_leg(lv, prm, mp, sweeps, x_props, P0, budget_s, threads, max_updates=None):
    """Time the CPU oracle (Localizator::correct restated; kNN = the reference's own ikd-Tree when
    oracle/_ref is present) on whole updates of the same workload until `budget_s` is used."""
    O = G.load_oracle()
    # "reference-kNN+port": the 5-NN runs in the reference's own ikd_Tree.cpp (oracle/_ref, compiled verbatim); plane fit,
    # Jacobian rows and the IESKF are the oracle's restatement (Eigen / IKFoM cannot be built in this image)
    kind = "reference-kNN+port" if O.ref_available() else "port"
    om = O.Map(O.KNN_REF_IKDTREE if kind != "port" else O.KNN_KDTREE)
    om.build(mp)
    om.knn(mp[0])                       # forces the lazy tree build of the port backend
    O.set_threads(threads)
    oprm = oracle_params(O, prm)
    pts, secs, n_upd = 0, 0.0, 0
    t_start = time.perf_counter()
    i = 0
    while True:
        t0 = time.perf_counter()
        st, x, P, logs = om.update_iterated(x_props[i % len(sweeps)], P0, oprm, sweeps[i % len(sweeps)])
        dt = time.perf_counter() - t0
        pts += sweeps[i % len(sweeps)].shape[0] * len(logs)
        secs += dt
        n_upd += 1
        i += 1
        if (max_updates and n_upd >= max_updates) or (not max_updates and time.perf_counter() - t_start > budget_s):
            break
        if max_updates and budget_s and time.perf_counter() - t_start > budget_s:   # reference arm: never run away
            break
    what = ("%d full updates (%d-pt sweep, %d-pt map, %d point-evaluations) in %.1f s; kNN = %s" %
            (n_upd, sweeps[0].shape[0], mp.shape[0], pts, secs,
             "reference ikd_Tree.cpp compiled verbatim (oracle/_ref)" if kind != "port" else "oracle kd-tree port"))
    return {"value": pts / secs, "unit": UNIT, "cores": threads, "kind": kind, "sample": what}, pts, secs, n_upd


def run_reference(args, rank, world_size):
    if rank != 0:
        return
    lv = G.load_package()                    # the Python module only: this arm loads liblv_synth.so (inputs), never the CUDA library
    cfg = args.config
    prm = config_params(lv, cfg, _L=lv.synth_lib())
    O = G.load_oracle()
    _, mp, sweeps, x_props, _ = make_scene(lv, 0, n_sweeps=4, prm=prm, cfg=cfg)
    x0, P0 = O.init_state(initial_gravity=prm.initial_gravity[:], I_Rotation_L=prm.I_Rotation_L[:],
                          I_Translation_L=prm.I_Translation_L[:])
    ncores = os.cpu_count() or 1
    threads = 3 if ncores > 4 else (2 if ncores == 4 else 1)      # MP_PROC_NUM rule, CMakeLists.txt:19-36
    cpu_leg(lv, prm, mp, sweeps, x_props, P0, 0, threads, max_updates=max(1, args.warmup if args.warmup < 2 else 1))
    # one step = one full update (~0.16 s with the reference's 3-thread team); K steps, but never more than ~3 minutes
    base, pts, secs, n_upd = cpu_leg(lv, prm, mp, sweeps, x_props, P0, 170.0, threads, max_updates=args.steps)
    line = {"impl": "reference", "metric": metric_name(cfg), "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": n_upd, "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / n_upd,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 geometry / f64 Jacobian+filter", "data": "synthetic",
            "config": workload_config(args.gpus, cfg, sequences=1), "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "host_cpu_count": ncores,
            "product_library_loaded": any("liblimovelo_b200" in l for l in open("/proc/self/maps"))}
    _emit(line)


def run_native(args, rank, local_rank, world_size):
    import torch
    import torch.distributed as dist
    lv = G.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()            # a real (non-default) stream: the library launches on it
    torch.cuda.set_stream(stream)
    cfg = args.config
    prm = config_params(lv, cfg, device=local_rank, stream=stream.cuda_stream)
    if args.voxel:                                                  # tuning runs only; the default is the library's
        prm.voxel_size = args.voxel
    if args.sort_queries is not None:
        prm.sort_queries = args.sort_queries
    world, mp, sweeps, x_props, truths = make_scene(lv, rank, prm=prm, cfg=cfg)
    n = sweeps[0].shape[0]
    loc = lv.Localizer(prm)
    loc.map_build(mp)
    loc.init_state()
    _, P0 = loc.get_state()
    d_sweeps = [loc.upload(s) for s in sweeps]                      # inputs resident in HBM for `value`
    pinned = [lv.PinnedBuffer((n, 3)) for _ in sweeps]              # pinned host copies for `e2e`
    for pb, s in zip(pinned, sweeps):
        pb.array[:] = s

    def step_device(i):
        loc.set_state(x_props[i % len(sweeps)], P0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        loc.correct_device(d_sweeps[i % len(sweeps)], n)
        e1.record(stream)
        st, logs = loc.last_logs()                                  # syncs; outside the timed events
        loc.flush_l2()
        return e0, e1, logs

    clocks = ClockSampler(local_rank)
    clocks.start()
    for i in range(args.warmup):
        step_device(i)
    torch.cuda.synchronize()
    clocks.wait_first()                                             # rows from here on fall inside the timed regions
    if world_size > 1:
        dist.barrier()
    loc.profile(reset=True)
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    evs, evals, matched = [], 0, 0
    for i in range(args.steps):
        e0, e1, logs = step_device(args.warmup + i)
        evs.append((e0, e1))
        evals += len(logs)
        matched += sum(l["n_matches"] for l in logs)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    if world_size > 1:
        dist.barrier()
    launches = loc.profile(reset=True)["total_launches"]
    step_ms = sum(a.elapsed_time(b) for a, b in evs)
    pts = n * evals
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loc)

    # ---- per-kernel device time (roofline): the same steps again with CUDA events around each kernel group.
    # The timed region above replays an update as ONE CUDA graph; events between its kernels would add bubbles,
    # so the per-kernel numbers come from this separate pass of direct launches on the same stream. ----
    loc.profile_enable(True)
    loc.profile(reset=True)
    prof_steps = min(args.steps, 50)
    for i in range(prof_steps):
        step_device(args.warmup + i)
    torch.cuda.synchronize()
    prof = loc.profile(reset=True)
    loc.profile_enable(False)

    # ---- e2e: the public host-buffer call, pinned H2D + kernels + D2H of the result, wall clock ----
    for i in range(min(3, args.warmup)):
        loc.set_state(x_props[i % len(sweeps)], P0)
        loc.correct(None, raw_ptr=pinned[i % len(sweeps)].ptr, n=n)
    e2e_s, e2e_pts = 0.0, 0
    buf = loc.correct_buffers()
    for i in range(args.steps):
        j = (args.warmup + i) % len(sweeps)
        loc.flush_l2()
        loc.synchronize()
        loc.set_state(x_props[j], P0)
        t0 = time.perf_counter()
        st = loc.correct_raw(pinned[j].ptr, n, buf)                 # the C-ABI call a LIMO-Velo binding makes, nothing else
        e2e_s += time.perf_counter() - t0
        assert st == 0, st
        e2e_pts += n * buf["ne"].value
    x, P, logs = loc.correct_unpack(buf)
    pose_err = float(np.abs(G.load_oracle().boxminus(x, truths[j]))[:3].max())
    clock_info = clocks.stop()                                      # sampled over both timed regions

    # ---- per-sweep map update (Mapper::add + rebuild), reported beside the headline ----
    t_add = []
    for i in range(2):
        gpts = world_points(sweeps[i], truths[i])
        loc.synchronize()
        t0 = time.perf_counter()
        loc.map_add(gpts, downsample=True)
        loc.synchronize()
        t_add.append(time.perf_counter() - t0)

    # ---- per sweep on the device: update + Mapper::add (main.cpp:84-105), nothing visits the host in between.
    # It changes the map, so it runs after the headline's timed regions (which replay sweeps against a fixed map). ----
    per_sweep = None
    try:
        ps_steps = min(args.steps, 100)
        ps_ms, ps_upd_ms, ps_evals = 0.0, 0.0, 0
        for i in range(ps_steps):
            j = (args.warmup + i) % len(sweeps)
            loc.set_state(x_props[j], P0)
            ea, eb, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            ea.record(stream)
            loc.correct_device(d_sweeps[j], n)
            eb.record(stream)
            loc.map_add_last_sweep(True)                            # sweep -> world with the update's own result -> 0.2 m rule -> halo buckets
            ec.record(stream)
            st, lg = loc.last_logs()
            ps_ms += ea.elapsed_time(ec)
            ps_upd_ms += ea.elapsed_time(eb)
            ps_evals += len(lg)
            loc.flush_l2()
        loc.map_status()
        per_sweep = {"ms": ps_ms / ps_steps, "update_ms": ps_upd_ms / ps_steps, "map_add_ms": (ps_ms - ps_upd_ms) / ps_steps,
                     "point_evaluations_per_s": n * ps_evals / (ps_ms * 1e-3), "sweeps": ps_steps, "map_points_after": loc.map_size(),
                     "how": "lv_correct_device + lv_map_add_last_sweep per sweep, CUDA events on the library's stream, L2 flushed between sweeps; "
                            "the map grows by the sweep's new cells"}
    except Exception as e:
        per_sweep = {"error": str(e)}

    # ---- deskew (Compensator::compensate, SURVEY 8f row 2), reported beside the headline ----
    deskew = None
    try:
        dk = deskew_case(lv, world, prm, sweeps[0])
        d_in, d_t = loc.upload(dk["xyz"]), loc.upload(dk["t"])
        for _ in range(3):
            loc.compensate_device(dk["path"], dk["xt2"], d_in, d_t, n, d_in)
        reps = 50
        loc.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            loc.compensate_device(dk["path"], dk["xt2"], d_in, d_t, n, d_in)      # blocking: path upload + 2 kernels + flag
        dt_dev = (time.perf_counter() - t0) / reps
        t0 = time.perf_counter()
        for _ in range(reps):
            loc.compensate(dk["path"], dk["xt2"], dk["xyz"], dk["t"])                # host buffers: + H2D 20 B/pt, D2H 12 B/pt
        dt_host = (time.perf_counter() - t0) / reps
        loc.device_free(d_in); loc.device_free(d_t)
        cpu_ms = None
        if rank == 0 and not args.no_cpu:                           # the oracle's restatement, one host thread
            O = G.load_oracle()
            po = [O.State32.from_buffer_copy(s) for s in dk["path"]]
            xo = O.State32.from_buffer_copy(dk["xt2"])
            t0 = time.perf_counter()
            O.compensate(po, xo, dk["xyz"], dk["t"])
            cpu_ms = 1e3 * (time.perf_counter() - t0)
        deskew = {"points": n, "path_states": len(dk["path"]), "lv_compensate_device_ms": 1e3 * dt_dev, "cpu_oracle_ms": cpu_ms,
                  "lv_compensate_host_ms": 1e3 * dt_host, "points_per_s_device": n / dt_dev,
                  "bytes_per_point": 32, "note": "blocking calls, wall clock; launch-bound at this size"}
    except Exception as e:                                         # never let the side measurement break the headline
        deskew = {"error": str(e)}

    # ---- downsamplers (SURVEY 8f row 3), reported beside the headline ----
    downsample = None
    try:
        d_in, d_out = loc.upload(sweeps[0]), loc.device_alloc(n * 12)
        for _ in range(3):
            m = loc.voxelgrid_downsample_device(d_in, n, 0.5, d_out)
        reps = 30
        t0 = time.perf_counter()
        for _ in range(reps):
            m = loc.voxelgrid_downsample_device(d_in, n, 0.5, d_out)             # blocking: 10 launches + count read-back
        dt_vg = (time.perf_counter() - t0) / reps
        loc.device_free(d_in); loc.device_free(d_out)
        raw = np.ascontiguousarray(np.tile(sweeps[0], (4, 1)))                    # a raw message at downsample_rate 4
        loc.temporal_downsample(raw, 4, 4.0)
        t0 = time.perf_counter()
        for _ in range(10):
            kept, _ = loc.temporal_downsample(raw, 4, 4.0)
        dt_td = (time.perf_counter() - t0) / 10
        downsample = {"voxelgrid_points": n, "voxelgrid_leaves": int(m), "leaf_m": 0.5,
                      "lv_voxelgrid_downsample_device_ms": 1e3 * dt_vg,
                      "temporal_points": int(raw.shape[0]), "temporal_kept": int(kept.shape[0]),
                      "lv_temporal_downsample_host_ms": 1e3 * dt_td, "note": "blocking calls, wall clock"}
    except Exception as e:
        downsample = {"error": str(e)}

    # ---- several sequences per GPU (one update does not fill a B200): S handles on S streams, one step = S concurrent updates ----
    multi = None
    if args.sequences_per_gpu:
        try:
            multi = multi_sequence_leg(lv, torch, cfg, local_rank, rank, [int(v) for v in args.sequences_per_gpu.split(",")], min(args.steps, 200))
        except Exception as e:
            multi = {"error": str(e)}

    # ---- max over ranks / totals (limo-velo_b200/dist.py: MAX of the times, SUM of the work; covered by tests/test_dist_gloo.py) ----
    import importlib
    dist_mod = importlib.import_module("limovelo_b200.dist")
    red = dist_mod.reduce_counters(step_ms, pts, matched, e2e_s, e2e_pts, launches, device="cuda")
    step_ms_max, e2e_s_max = red["step_ms"], red["e2e_s"]
    pts_all, matched_all, e2e_pts_all, launches_all = red["points"], red["matched"], red["e2e_points"], red["launches"]

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        m_launches = max(1, prof["measure_launches"])
        m_ms = prof["measure_ms"] / m_launches
        k_ms = {"lv_search_kernel": prof["search_ms"] / m_launches, "lv_search_rings_kernel": prof["search_upper_ms"] / m_launches,
                "lv_fit_kernel": prof["fit_ms"] / m_launches, "lv_ieskf_step_kernel": prof["solve_ms"] / max(1, prof["solve_launches"])}
        # The roofline kernel is the search: the largest of the per-point kernels (SURVEY 8d's unit is the point).
        # lv_ieskf_step_kernel takes about as long per evaluation but moves no per-point bytes: it is ~12 us of
        # dependent fp64 23x23 algebra in one block (DESIGN.md 4); its time is listed in kernel_ms.
        dominant = "lv_search_kernel"
        # ... timed on the launches that search EVERY query (the first evaluation of each update): later evaluations only
        # search what the reuse test hands back, their launches are shorter for doing less, and 72 B x n is not their traffic
        first_ms = prof["search_first_ms"] / max(1, prof["search_first_launches"])
        k_ms["lv_search_kernel_first_evaluation"] = first_ms
        achieved = ALGO_BYTES_PER_POINT * n / (first_ms * 1e-3) / 1e9 if first_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:                                                        # dram bytes per launch from the committed ncu --set full capture
            if cfg != "cfg1" or args.sort_queries or args.voxel:
                raise LookupError("the capture is of the default cfg1 run")
            tr = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
            # the first evaluation's search (every query: the launch the algorithmic bytes are counted for)
            name = next(k for k in tr if k.startswith(dominant) and k.rstrip(">").endswith("0"))
            traffic = tr[name]["dram_bytes_per_launch"]
            traffic_src = "profiles/kernel_traffic.json [%s], from the committed ncu --set full capture of `bench.py --steps 2` (cfg1); not re-measured by this run" % name
        except Exception:
            pass
        cpu = None
        if not args.no_cpu:
            O = G.load_oracle()
            cpu, _, _, _ = cpu_leg(lv, prm, mp, sweeps, x_props, P0, args.cpu_seconds, 1)
        sz_ctrl = loc.result_bytes()
        line = {
            "metric": metric_name(cfg), "value": pts_all / (step_ms_max * 1e-3), "unit": UNIT, "n_gpus": world_size,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 geometry / f64 Jacobian+filter", "data": "synthetic", "config": workload_config(world_size, cfg),
            "evaluations_per_step": evals / args.steps, "accept_rate": matched_all / max(1.0, pts_all),
            "matched_points_per_s": matched_all / (step_ms_max * 1e-3),
            "wall_ms_total_incl_flush_and_readback": 1e3 * t_wall,
            "e2e": {"value": e2e_pts_all / e2e_s_max, "unit": UNIT, "h2d_bytes_per_step": n * 12 + 8 * (26 + 529),
                    "d2h_bytes_per_step": sz_ctrl, "ms_per_step": 1e3 * e2e_s_max / args.steps,
                    "how": "lv_correct() (C ABI, via ctypes) on a pinned host sweep, state upload + sweep H2D + update + result D2H, wall clock around the blocking call"},
            "gpu_launches": int(round(launches_all)) - args.steps * world_size,   # minus the L2-flush kernels
            "kernel_ms": {"how": "separate pass of %d steps, direct launches, CUDA events around each kernel group; "
                                 "the timed region replays each update as one CUDA graph" % prof_steps,
                          "per_evaluation": k_ms,
                          "measure_avg": m_ms, "measure_launches": prof["measure_launches"],
                          "idle_measure_launches": prof.get("idle_launches", 0),
                          "solve_avg": prof["solve_ms"] / max(1, prof["solve_launches"]),
                          "solve_launches": prof["solve_launches"]},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": achieved / peak_gbs, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": dominant, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_POINT * n,
                         "launches_timed": "first evaluation of every update (all %d queries searched): %d launches, %.2f us each (CUDA events, live pass)" % (n, prof["search_first_launches"], 1e3 * first_ms)},
            "cpu_baseline": cpu,
            "per_sweep": per_sweep,
            "map_update": {"lv_map_add_ms": 1e3 * min(t_add), "points_added": n, "map_points": loc.map_size(),
                           "how": "lv_map_add() from a pageable host buffer, wall clock incl. the H2D copy and a stream synchronisation"},
            "multi_sequence": multi,
            "deskew": deskew, "downsample": downsample,
            "final_position_error_m": pose_err,
            "clocks": clock_info,
        }
        _emit(line)
    for pb in pinned:
        pb.free()
    loc.close()
    if world_size > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, loc):
    """What the last timed step handed its caller (lv_last_logs, lv_get_state), as DIR/<name>.npy in float64: the
    status, the per-evaluation logs stacked along axis 0, and the updated state x (26) and covariance P (23 x 23).
    The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    st, logs = loc.last_logs()
    x, P = loc.get_state()
    out = {"status": [st], "x": x, "P": P}
    for k in ("n_matches", "converged", "degenerate", "HTH", "HTh", "dx", "x_after"):
        out[k] = [lg[k] for lg in logs]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.asarray(v, dtype=np.float64))


def multi_sequence_leg(lv, torch, cfg, local_rank, rank, s_list, steps):
    """point-evaluations/s of ONE GPU running S independent sequences at once (S handles, S streams, no shared state)"""
    out = []
    n = update_points(cfg)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for S in s_list:
        streams = [torch.cuda.Stream() for _ in range(S)]
        locs, data = [], []
        for s in range(S):
            prm = config_params(lv, cfg, device=local_rank, stream=streams[s].cuda_stream)
            world, mp, sweeps, x_props, truths = make_scene(lv, 50 + 8 * rank + s, n_sweeps=4, prm=prm, cfg=cfg)
            loc = lv.Localizer(prm)
            loc.map_build(mp)
            loc.init_state()
            _, P0 = loc.get_state()
            locs.append(loc)
            data.append(([loc.upload(sw) for sw in sweeps], x_props, P0))

        def step(i, timed):
            for s in range(S):
                locs[s].set_state(data[s][1][i % 4], data[s][2])
            fork, join = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(streams[0]):
                flush.fill_(i & 255)                                # L2 flush between steps
            fork.record(streams[0])
            ends = []
            for s in range(S):
                if s:
                    streams[s].wait_event(fork)
                locs[s].correct_device(data[s][0][i % 4], n)
                e = torch.cuda.Event()
                e.record(streams[s])
                ends.append(e)
            for e in ends[1:]:
                streams[0].wait_event(e)
            join.record(streams[0])
            evals = sum(len(locs[s].last_logs()[1]) for s in range(S))   # synchronises each stream
            return fork.elapsed_time(join), evals
        for i in range(3):
            step(i, False)
        ms, evals = 0.0, 0
        for i in range(steps):
            m, e = step(3 + i, True)
            ms += m
            evals += e
        out.append({"sequences": S, "ms_per_step": ms / steps, "point_evaluations_per_s": n * evals / (ms * 1e-3)})
        for loc in locs:
            loc.close()
        del locs, data
        torch.cuda.empty_cache()
    base = out[0]["point_evaluations_per_s"] if out and out[0]["sequences"] == 1 else None
    for o in out:
        o["vs_one_sequence"] = o["point_evaluations_per_s"] / base if base else None
    return {"how": "S independent handles on S CUDA streams of one GPU; one step = S concurrent updates, fork/join CUDA events, "
                   "L2 flushed between steps", "results": out}


def run_strong(args, rank, local_rank, world_size):
    """BASELINE.json configs[4]: a fixed job of 8 independent sequences over N GPUs (strong scaling).  Every rank runs its
    share concurrently (one handle + one stream per sequence); one step = every sequence does one update."""
    import importlib
    import torch
    import torch.distributed as dist
    lv = G.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dist_mod = importlib.import_module("limovelo_b200.dist")
    cfg = "cfg4"
    n_seq = CONFIGS[cfg]["sequences"]
    mine = dist_mod.sequence_for_rank(rank, world_size, n_seq)
    n = update_points(cfg)
    streams, locs, data = [], [], []
    for sq in mine:
        st = torch.cuda.Stream()
        prm = config_params(lv, cfg, device=local_rank, stream=st.cuda_stream)
        world, mp, sweeps, x_props, truths = make_scene(lv, sq, n_sweeps=4, prm=prm, cfg=cfg)
        loc = lv.Localizer(prm)
        loc.map_build(mp)
        loc.init_state()
        _, P0 = loc.get_state()
        pinned = [torch.from_numpy(sw.copy()).pin_memory() for sw in sweeps]
        dev = [torch.empty((n, 3), dtype=torch.float32, device="cuda") for _ in sweeps]
        for d, p in zip(dev, pinned):
            d.copy_(p)
        streams.append(st); locs.append(loc); data.append((dev, pinned, x_props, P0, truths))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    main = streams[0] if streams else torch.cuda.current_stream()

    def step(i, with_copies):
        for s, loc in enumerate(locs):
            loc.set_state(data[s][2][i % 4], data[s][3])
        fork, join = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(main):
            flush.fill_(i & 255)
        fork.record(main)
        ends = []
        for s, loc in enumerate(locs):
            if s:
                streams[s].wait_event(fork)
            d = data[s][0][i % 4]
            if with_copies:                                         # e2e: the sweep comes from pinned host memory inside the timed region
                with torch.cuda.stream(streams[s]):
                    d.copy_(data[s][1][i % 4], non_blocking=True)
            loc.correct_device(d.data_ptr(), n)
            e = torch.cuda.Event()
            e.record(streams[s])
            ends.append(e)
        for e in ends[1:]:
            main.wait_event(e)
        join.record(main)
        evals = 0
        for loc in locs:
            st_, lg = loc.last_logs()                               # D2H of the result (26.9 KB) + synchronisation
            evals += len(lg)
        return fork.elapsed_time(join), evals
    clocks = ClockSampler(local_rank)
    clocks.start()
    for i in range(max(3, args.warmup)):
        step(i, False)
    torch.cuda.synchronize()
    clocks.wait_first()
    if world_size > 1:
        dist.barrier()
    for loc in locs:
        loc.profile(reset=True)
    ms, evals = 0.0, 0
    for i in range(args.steps):
        m, e = step(args.warmup + i, False)
        ms += m
        evals += e
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()
    launches = sum(loc.profile(reset=True)["total_launches"] for loc in locs)
    e2e_ms, e2e_evals = 0.0, 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        m, e = step(args.warmup + i, True)
        e2e_ms += m
        e2e_evals += e
    e2e_wall = time.perf_counter() - t0
    clock_info = clocks.stop()
    err = max(float(np.abs(G.load_oracle().boxminus(loc.get_state()[0], data[s][4][(args.warmup + args.steps - 1) % 4]))[:3].max())
              for s, loc in enumerate(locs)) if locs else 0.0
    red = dist_mod.reduce_counters(ms, n * evals, 0, e2e_ms * 1e-3, n * e2e_evals, launches, device="cuda")
    if rank == 0:
        line = {"metric": metric_name(cfg), "value": red["points"] / (red["step_ms"] * 1e-3), "unit": UNIT, "n_gpus": world_size,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": red["step_ms"] / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32 geometry / f64 Jacobian+filter", "data": "synthetic",
                "config": dict(workload_config(world_size, cfg, sequences=n_seq),
                               parallelism="%d sequences per GPU, one handle + one CUDA stream each, no data-path collective" % len(mine)),
                "e2e": {"value": red["e2e_points"] / red["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": n_seq * n * 12,
                        "d2h_bytes_per_step": n_seq * locs[0].result_bytes(), "ms_per_step": 1e3 * red["e2e_s"] / args.steps,
                        "how": "per sequence: pinned-host sweep -> device (async copy on the sequence's stream), update, result D2H; "
                               "CUDA events fork/join over all streams of the rank, max over ranks"},
                "gpu_launches": int(round(red["launches"])), "sequences_total": n_seq, "sequences_per_gpu": len(mine),
                "e2e_wall_ms_per_step": 1e3 * e2e_wall / args.steps, "final_position_error_m": err, "clocks": clock_info}
        _emit(line)
    for loc in locs:
        loc.close()
    if world_size > 1:
        dist.destroy_process_group()


def deskew_case(lv, world, prm, sweep, t1=10.0, t2=10.1, n_states=4, imu_hz=400.0):
    """a 0.1 s sweep at 15 m/s: KF states every ~33 ms, IMU at 400 Hz, point stamps spread over the sweep"""
    rng = np.random.default_rng(SEED + 77)
    st_times = np.linspace(t1 - 0.012, t2 - 0.004, n_states)
    imu_t = np.arange(st_times[0] + 0.2 / imu_hz, t2 + 1.5 / imu_hz, 1.0 / imu_hz)   # Compensator::path: from the first state on
    imu_a = (np.array([0.3, -0.2, 9.8]) + rng.normal(0, 0.05, (len(imu_t), 3))).astype(np.float32)
    imu_w = (np.array([0.02, -0.01, 0.3]) + rng.normal(0, 0.01, (len(imu_t), 3))).astype(np.float32)
    states = []
    for ts in st_times:
        x = world.pose(15.0 + 15.0 * (ts - t1), prm).copy()
        x[14:17] = [15.0, 0.3, -0.1]
        j = int(np.searchsorted(imu_t, ts))
        states.append(lv.state_from_ikfom(prm, x, ts, imu_a[j], imu_w[j]))
    path = lv.compensator_upsample(states, imu_a, imu_w, imu_t)
    return dict(path=path, xt2=lv.compensator_get_t2(path, t2), xyz=np.ascontiguousarray(sweep, np.float32),
                t=np.linspace(t1, t2, len(sweep)))


def world_points(sweep, x):
    """LiDAR-frame sweep -> world frame with the true state (what main.cpp:101 hands to map.add)."""
    O = G.load_oracle()
    R = O.quat_to_rot(x[3:7])
    RL = O.quat_to_rot(x[7:11])
    p_imu = sweep.astype(np.float64) @ RL.T + x[11:14]
    return (p_imu @ R.T + x[0:3]).astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--config", default="cfg1", choices=sorted(CONFIGS), help="BASELINE.json config (default cfg1 = the metric's)")
    ap.add_argument("--sequences-per-gpu", default="", help="e.g. 1,2,4,8: also measure S concurrent sequences per GPU (multi_sequence)")
    ap.add_argument("--sort-queries", type=int, default=None, help="tuning: 1 = binned order + search from shared memory, 0 = per-query search")
    ap.add_argument("--voxel", type=float, default=0.0, help="tuning: finest voxel edge of the map (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the last step's results (state, covariance, per-evaluation logs) "
                         "as DIR/<name>.npy (float64, about 20 KB; rank 0's sequence)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.config == "cfg4"):
        ap.error("--dump-outputs writes the native single-sequence update (--impl native, --config cfg0..cfg3)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)             # keep the real stdout for the JSON line only
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world_size)
    elif args.config == "cfg4":
        run_strong(args, rank, local_rank, world_size)
    else:
        run_native(args, rank, local_rank, world_size)


if __name__ == "__main__":
    main()
