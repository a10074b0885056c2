#!/usr/bin/env python
"""bench.py -- grasp windows scored per second (all rolls) and ms per cloud, BASELINE.json's metric.

Default workload (N = 1): the per-GPU share of BASELINE.json configs[4] ("throughput mode"): 512 synthetic
100k-point clouds (seeds 1234 + i), G = 56, 12 rolls, area 32x44, approach (0,0,1), synthetic SVM model with
2048 support vectors (the trained model is missing from the reference checkout).  Weak scaling: every rank
processes its own 512 clouds (4096 at N = 8), clouds are sharded by rank with no data-path collective; only the
best-grasp records are exchanged (NCCL all_gather) inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload batch|grid512|table1]

`value`  : windows/s with the clouds already resident in HBM, K steps timed with CUDA events on the stream the
           kernels run on, max over ranks.  Inputs (614 MB / rank) are larger than L2, no flush needed.
`e2e`    : same metric through the C-ABI call with HOST (pinned) buffers: host->device copy of the clouds and
           device->host copy of the results inside the timed region.
`--impl reference` : the reference's own CPU path (its feature classes + svm-scale + svm-predict child processes
           on text files, compiled in place under oracle/_ref; the ROS-bound members restated by the oracle) on
           all host cores, one cloud per worker process, a bounded sample of the same workload per step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
FEATURES = os.path.join(ROOT, "tests", "golden", "refdata", "Features.txt")
RANGE = os.path.join(ROOT, "tests", "golden", "refdata", "range21062012_allfeatures")
METRIC = "grasp_windows_scored_per_sec_all_rolls"
UNIT = "windows/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="batch", choices=["batch", "grid512", "table1", "approach"])
    ap.add_argument("--clouds", type=int, default=512, help="clouds per GPU (batch workload)")
    ap.add_argument("--points", type=int, default=100000)
    ap.add_argument("--nsv", type=int, default=2048)
    ap.add_argument("--tc-passes", type=int, default=0, help="tensor-core products per k-slice: 0 = calibrated per model (default), 1 / 2 / 3 forced")
    ap.add_argument("--sv-table-global", type=int, default=0, help="experiment: 1 = tensor kernels read the SV table from global memory")
    ap.add_argument("--tc-variant", type=int, default=0, help="tensor kernel: 0 auto (X-resident CTA pair where eligible), 1 single CTA, 2 streaming CTA pair")
    ap.add_argument("--bin-variant", type=int, default=0, help="binning: 0 auto, 1 point-parallel kernel only, 2 whole-cloud kernel with scalar loads")
    ap.add_argument("--svm-mode", type=int, default=0, help="0 tcgen05 split-fp16 + FP64 guard (default), 1 FP64 exact, 2 FP32 SIMT + guard")
    ap.add_argument("--guard-kernel", type=int, default=0, help="guard band tier 2: 0 auto, 1 FP64 tensor cores (DMMA) always, 2 DFMA always")
    ap.add_argument("--graph", type=int, default=-1, help="1 = capture / replay one CUDA graph per request shape (single-pass calls without per-stage events); "
                                                            "-1 (default) = on for the single-goal workloads (table1, grid512, approach), off for batches (which never qualify)")
    ap.add_argument("--group", type=int, default=1, help="ONE process driving this many GPUs through the C ABI's multi-GPU context (haf_config.n_devices): "
                                                         "the path a C++ host takes; --clouds is per GPU; timed by wall clock (the member GPUs run on their own streams)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-clouds", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.graph < 0:
        args.graph = 1 if args.workload in ("table1", "grid512", "approach") else 0
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def model_path(nsv):
    from haf_grasping_b200 import synth
    d = os.path.join(tempfile.gettempdir(), "haf_bench_models")
    os.makedirs(d, exist_ok=True)
    p = os.path.join(d, "synth_%d_seed7.model" % nsv)
    if not os.path.exists(p):
        synth.write_synth_model(p, n_sv=nsv, seed=7)
    return p


def workload_config(args):
    if args.workload == "batch":
        return dict(grid=56, rmax=190, step=15, area=(32.0, 44.0), r=0.28, n_clouds=args.clouds, n_points=args.points)
    if args.workload == "approach":
        return dict(grid=56, rmax=190, step=15, area=(32.0, 44.0), r=0.28, n_clouds=1, n_points=0)
    if args.workload == "grid512":  # BASELINE.json configs[3]
        return dict(grid=512, rmax=190, step=15, area=(362.0, 362.0), r=2.56, n_clouds=1, n_points=1000000)
    return dict(grid=56, rmax=190, step=15, area=(32.0, 44.0), r=0.28, n_clouds=1, n_points=0)


def dump_outputs(out_dir, arrays):
    """one DIR/<name>.npy per array, float64 (exact for the int32 and float32 fields the library returns)"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


# the answer fields of haf_best (n_guard / reserved describe how the answer was computed, not the answer)
BEST_FIELDS = ("row", "col", "roll", "tilt", "approach_idx", "topval", "eval", "roll_rad", "M", "rolls_done", "n_windows_scored")


def best_arrays(best):
    """haf_best records of a batch -> {best_<field>: [n_clouds] or [n_clouds, 16] array}"""
    return {"best_" + f: [list(getattr(b, f)) if f == "M" else getattr(b, f) for b in best] for f in BEST_FIELDS}


def make_clouds(args, wc, rank):
    """list of float32 [n,3] arrays for this rank (seeds 1234 + global cloud index)"""
    import numpy as np
    from haf_grasping_b200 import synth
    if args.workload in ("table1", "approach"):
        z = np.load(os.path.join(ROOT, "tests", "golden", "clouds.npz"))
        return [np.ascontiguousarray(z["table1"])]
    base = 1234 + rank * wc["n_clouds"]
    return [synth.synth_cloud(base + i, wc["n_points"], r=wc["r"]) for i in range(wc["n_clouds"])]


class ClockSampler:
    # the sampler is started BEFORE the warm-up steps (nvidia-smi needs a few hundred ms to deliver its first row) and
    # only the rows stamped inside the timed region are kept
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            self.path = tempfile.mktemp(prefix="haf_clocks_", suffix=".csv")
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t_begin = time.time()

    def stop(self):
        t_end = time.time()
        t_begin = getattr(self, "t_begin", 0.0)
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        import datetime
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        with open(self.path) as fh:
            for ln in fh:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), [nm for k, nm in enumerate(names) if f[5 + k].lower().startswith("active")]))
                except ValueError:
                    continue
        os.remove(self.path)
        inside = [r for r in rows if t_begin - 0.005 <= r[0] <= t_end + 0.005]
        window = "timed region"
        if not inside and rows:   # a timed region shorter than the sampling period: the rows nearest to it (warm-up of the same steps)
            inside, window = rows[-3:], "last rows before the end of the timed region"
        if inside:
            out = {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": max(r[2] for r in inside),
                   "reasons": sorted({nm for r in inside for nm in r[3]}), "samples": len(inside), "window": window}
        return out


# ------------------------------------------------------------------------------------------------------
# reference CPU path (one cloud): reference feature class + svm-scale + svm-predict on files, per roll,
# exactly as server.cpp:616-656 and :754-800 do; the ROS-bound members come from the oracle restatement.
# ------------------------------------------------------------------------------------------------------
def _ref_cloud_worker(job):
    xyz, model, grid, step, rmax, area, kind, roll_limit = job
    from oracle import orc
    o = orc.Oracle(FEATURES, RANGE, model)
    t0 = time.perf_counter()
    R = rmax // step
    if roll_limit > 0:
        R = min(R, roll_limit)
    windows = 0
    if kind == "reference":
        r = orc.Ref(FEATURES, RANGE, model)
        av = o.normalize_approach((0, 0, 1))
        wd = tempfile.mkdtemp(prefix="hafref_")
        best = (-1000, -1, -1, -1)
        for roll in range(R):
            M = o.build_transform((0, 0, 0), av, 1, roll, step)
            integral = o.calc_intimage(o.generate_grid(xyz, M, grid))
            mask = o.pnt_in_box(integral, roll, (int(area[0]), int(area[1])), step)
            labels, _ = r.roll_file_exact(integral, mask, workdir=wd)
            _, top, _ = o.show_predicted_gps(labels, mask)
            windows += len(labels)
            if top[2] > best[0]:
                best = (top[2], top[0], top[1], roll)
        for f in os.listdir(wd):
            os.remove(os.path.join(wd, f))
        os.rmdir(wd)
    else:  # "port": the in-process oracle
        res = o.search(xyz, orc.make_request(area=area, roll_limit=roll_limit), G=grid, roll_step_deg=step, roll_max_deg=rmax, full=False)
        windows = int(res["best"].n_windows)
    return windows, time.perf_counter() - t0


def cpu_reference_rate(args, wc, clouds, n_workers, model, area=None, roll_limit=0):
    """windows/s of the reference CPU path over `clouds` with n_workers processes (one cloud each at a time).
    area / roll_limit bound the sample for the big-grid workload (windows/s is a per-window rate)."""
    import multiprocessing as mp
    from oracle import orc
    orc.build(ref=os.path.isdir("/root/reference"))
    kind = "reference" if orc.ref_available() else "port"
    jobs = [(c, model, wc["grid"], wc["step"], wc["rmax"], area or wc["area"], kind, roll_limit) for c in clouds]
    t0 = time.perf_counter()
    if n_workers <= 1:
        res = [_ref_cloud_worker(j) for j in jobs]
    else:
        with mp.get_context("fork").Pool(n_workers) as pool:
            res = pool.map(_ref_cloud_worker, jobs, chunksize=1)
    dt = time.perf_counter() - t0
    return sum(r[0] for r in res) / dt, sum(r[0] for r in res), dt, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wc = workload_config(args)
    model = model_path(args.nsv)
    cores = max(1, min(os.cpu_count() or 1, 64))
    per_step = cores
    if args.workload != "batch":
        per_step = 1
        cores = 1
    import numpy as np  # noqa: F401
    from haf_grasping_b200 import synth
    times, wins, kind = [], [], "port"
    sample_kw = {"area": (100.0, 100.0), "roll_limit": 1} if args.workload == "grid512" else {}
    for s in range(args.warmup + args.steps):
        if args.workload == "batch":
            clouds = [synth.synth_cloud(1234 + (s * per_step + i) % wc["n_clouds"], wc["n_points"], r=wc["r"]) for i in range(per_step)]
        else:
            clouds = make_clouds(args, wc, 0)
        rate, w, dt, kind = cpu_reference_rate(args, wc, clouds, cores, model, **sample_kw)
        if s >= args.warmup:
            times.append(dt)
            wins.append(w)
    value = sum(wins) / sum(times)
    sample = "%s%d cloud(s) per step (one per worker process), %d timed steps; %s" % (
        "roll 0 of a 100x100 cm sub-area of the 512-grid cloud; " if sample_kw else "", per_step, args.steps, "reference feature classes + svm-scale + svm-predict child processes on text files per roll"
        if kind == "reference" else "in-process oracle port")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": describe(args, wc), "n_sv": args.nsv},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def describe(args, wc):
    if args.workload == "batch":
        return ("configs[4] per-GPU share: %d synthetic clouds x %d points per GPU, G=56, 12 rolls, area 32x44, AV (0,0,1)"
                % (wc["n_clouds"], wc["n_points"]))
    if args.workload == "grid512":
        return "configs[3]: synthetic 1M-point cloud, G=512, area 362x362, 12 rolls"
    return "configs[1]: table1 scene (102876 points), G=56, 12 rolls, default request"


TILTED = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254)]


def run_approach(args):
    """BASELINE configs[2]: one goal on the objects_1 (= table1) scene with 5 approach vectors x 12 rolls = 60 units,
    sharded by (approach vector, roll) over the ranks; the per-unit tops are exchanged (NCCL all_reduce MAX) and the
    reference's sequential rules replayed on the merged array.  Strong scaling (total work fixed).  Every rank also
    checks the merged answer against its own unsharded search."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import haf_grasping_b200 as h
    from haf_grasping_b200 import distributed as hd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    model = model_path(args.nsv) if rank == 0 or world == 1 else None
    if world > 1:
        dist.barrier()
        model = model_path(args.nsv)
    wc = workload_config(args)
    big = args.workload == "grid512"    # configs[3] as ONE goal sharded by roll (strong scaling); else configs[2]
    if big:
        from haf_grasping_b200 import synth
        xyz = synth.synth_cloud(1234, wc["n_points"], r=wc["r"])
        approaches = [(0.0, 0.0, 1.0)]
    else:
        xyz = np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "clouds.npz"))["table1"])
        approaches = TILTED
    host = torch.empty((len(xyz), 3), dtype=torch.float32, pin_memory=True)
    host.numpy()[:] = xyz
    dev = host.cuda()
    gs = h.GraspSearch(FEATURES, RANGE, model, grid=wc["grid"], device=local, svm_mode=args.svm_mode, use_graph=bool(args.graph))
    stream = torch.cuda.current_stream()
    gs.set_stream(stream.cuda_stream)
    R, A = gs.R, len(approaches)
    windows = [0]

    def evaluate_on(buf):
        def evaluate(a, rb, re):
            res = gs.search(buf, [h.make_request(area=wc["area"], approach=approaches[a], roll_begin=rb, roll_limit=re)], outputs=False)
            windows[0] += gs.timing().n_windows
            return res["per_roll_top"][0][rb:re]
        return evaluate

    last = {}

    def step(buf):
        last["result"] = hd.sharded_goal_search(evaluate_on(buf), A, R, [0] * A, [119] * A, rank, world)
        return last["result"]

    ref = gs.search(dev, [h.make_request(area=wc["area"], approach=a) for a in approaches], outputs=False)
    per, overall, tops = step(dev)
    assert overall[0] == ref["best"].approach_idx and overall[1:] == ref["best"].astuple()[:3] + (ref["best"].topval,), (overall, ref["best"].astuple())
    assert np.array_equal(tops.reshape(A, R, 3), ref["per_roll_top"])

    def timed(buf, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        windows[0] = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step(buf)
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        w = float(windows[0])
        if world > 1:
            t = torch.tensor([ms, w], dtype=torch.float64, device="cuda")
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms, w = float(tm[0].item()), float(t[1].item())
        return ms, w

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(dev)
    sampler.mark_begin()
    l0 = gs.launch_count()
    ms_dev, w_dev = timed(dev, args.steps)
    launches = gs.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        per, overall, tops = last["result"]
        dump_outputs(args.dump_outputs, {"per_request_best": per, "overall_best": overall, "unit_tops": tops})
    for _ in range(3):          # the host-memory path has its own staging buffer (and, with graphs on, its own captures)
        step(host.numpy())
    ms_e2e, w_e2e = timed(host.numpy(), args.steps)
    if rank == 0:
        line = {"metric": METRIC, "value": w_dev / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": dtype_of(args.svm_mode, gs.timing().tc_passes),
                "data": "synthetic" if big else "tests/golden/clouds.npz:table1 (= data/objects_1.pcd of the reference)",
                "config": {"workload": ("configs[3] as ONE goal: synthetic 1M-point cloud, G=512, area 362x362, its 12 rolls sharded over the ranks (strong scaling); "
                                        if big else "configs[2]: objects_1 scene x 5 approach vectors x 12 rolls = 60 units sharded by (approach vector, roll) over the ranks; ") +
                                       "merged best grasp verified against the unsharded search on every rank",
                           "n_sv": gs.info.n_sv, "l2": "single goal: latency-bound, working set far below L2 (no flush: that is the operating point of one goal)",
                           "units_per_rank": [sum(re - rb for _, rb, re in hd.unit_blocks(A, R, r, world)) for r in range(world)]},
                "ms_per_goal": ms_dev / args.steps, "clocks": clocks,
                "e2e": {"value": w_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(len(xyz) * 12 * len(hd.unit_blocks(A, R, 0, world))),
                        "d2h_bytes_per_step": A * R * 12, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches),
                "cuda_graph": {"enabled": bool(args.graph), "replays_so_far": int(gs.timing().graph_replays)},
                "roofline": {"kernel": "svm_rbf_tc2_kernel", "bound": "tensor", "achieved": None, "peak": peaks()[2], "unit": "TFLOP/s", "frac": None,
                             "traffic": None, "note": "latency-bound single goal: see the default (batch) workload for the roofline of this kernel"}}
        emit(line)
    gs.close()
    if world > 1:
        dist.destroy_process_group()


def dtype_of(svm_mode, passes):
    """arithmetic type of the path's dominant stage (not a precision claim: labels equal the FP64 reference's)"""
    if svm_mode == 2:
        return "f32"
    if svm_mode == 1:
        return "f64"
    return "f32 (contraction: fp16 operands, %d tensor-core product%s per k-slice, f32 accumulate; f64 guard band)" % (passes, "" if passes == 1 else "s")


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import haf_grasping_b200 as h

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libhafgpu has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wc = workload_config(args)
    group = max(1, args.group)
    if group > 1:
        if world > 1:
            raise SystemExit("bench.py: --group is a single-process mode (no torchrun)")
        wc["n_clouds"] *= group if args.workload == "batch" else 1
    model = model_path(args.nsv) if rank == 0 or world == 1 else None
    if world > 1:
        dist.barrier()
        model = model_path(args.nsv)
    clouds = make_clouds(args, wc, rank)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    total_pts = int(offsets[-1])
    host = torch.empty((total_pts, 3), dtype=torch.float32, pin_memory=True)
    host.numpy()[:] = np.concatenate(clouds)
    dev = host.cuda(non_blocking=False)
    n_clouds = len(clouds)

    gs = h.GraspSearch(FEATURES, RANGE, model, grid=wc["grid"], roll_step_deg=wc["step"], roll_max_deg=wc["rmax"],
                       device=local, svm_mode=args.svm_mode, sv_table_global=args.sv_table_global, tc_passes=args.tc_passes,
                       tc_variant=args.tc_variant, bin_variant=args.bin_variant, devices=list(range(group)) if group > 1 else None,
                       guard_kernel=args.guard_kernel, use_graph=bool(args.graph))
    stream = torch.cuda.current_stream()
    gs.set_stream(stream.cuda_stream)
    # per-stage events in the timed region of the batch workloads (8 timing events per pass of ~10 ms: the kernel time of the
    # roofline is measured live); a single goal is a chain of ~18 kernels of 5-30 us and every timing event between them costs
    # about as much as one of those (it drains the pipeline): single goals are timed without, the stages come from a second pass
    prof_in_timed = n_clouds > 1
    gs.set_profiling(prof_in_timed)
    rq = h.make_request(area=wc["area"])
    # the one exchange of the path: the 32-byte best-grasp records (SURVEY 8e), packed by the library straight into a pinned
    # buffer, one async H2D copy, NCCL all_gather
    rec_host = torch.zeros((n_clouds, 8), dtype=torch.int32, pin_memory=True)
    rec_dev = torch.zeros((n_clouds, 8), dtype=torch.int32, device="cuda")
    gathered = torch.zeros((world * n_clouds, 8), dtype=torch.int32, device="cuda") if world > 1 else None

    last = {}

    def step(buf):
        best = gs.search_batch_packed(buf, offsets, rq)
        if world > 1:
            gs.pack_best_records(best, rec_host)
            rec_dev.copy_(rec_host, non_blocking=True)
            dist.all_gather_into_tensor(gathered, rec_dev)
        last["best"] = best
        return best

    def timed(buf, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        acc = dict(svm=0.0, bin=0.0, integral=0.0, mask=0.0, features=0.0, guard=0.0, score=0.0, windows=0, guardw=0, auditw=0, chunks=0, launches=0)
        for _ in range(steps):
            step(buf)
            t = gs.timing()
            for k in ("svm", "bin", "integral", "mask", "features", "guard", "score"):
                acc[k] += getattr(t, "ms_" + k)
            acc["windows"] += t.n_windows
            acc["guardw"] += t.n_guard
            acc["auditw"] += t.n_audit
            acc["chunks"] += t.n_chunks
            acc["launches"] += t.launches
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        if group > 1:
            ms = wall * 1e3   # the member GPUs run on their own streams: the host call's wall time is the honest clock here
        if world > 1:
            tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm.item())
            tw = torch.tensor([float(acc["windows"])], dtype=torch.float64, device="cuda")
            dist.all_reduce(tw, op=dist.ReduceOp.SUM)
            acc["windows_all"] = float(tw.item())
        else:
            acc["windows_all"] = float(acc["windows"])
        return ms, wall, acc

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(dev)
    sampler.mark_begin()
    ms_dev, wall_dev, acc = timed(dev, args.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, best_arrays(last["best"]))
    graph_replays = int(gs.timing().graph_replays)
    accs, ms_dev_prof = acc, ms_dev      # where the stage times come from
    if not prof_in_timed:
        gs.set_profiling(True)
        step(dev)
        ms_dev_prof, _, accs = timed(dev, args.steps)
    # end to end: host (pinned) buffers in, results out, through the same C-ABI call
    # (timed as a caller gets it: without the per-stage events; the stage breakdown comes from a short profiled pass afterwards)
    gs.set_profiling(False)
    for _ in range(2):
        step(host.numpy())
    ms_e2e, wall_e2e, acc2 = timed(host.numpy(), args.steps)
    gs.set_profiling(True)
    n_prof = max(2, min(args.steps, 3))
    step(host.numpy())
    ms_e2e_prof, _, acc2p = timed(host.numpy(), n_prof)
    # what bounds the end-to-end number from below: the same bytes copied host -> device and nothing else, all ranks at once
    def copies_only(steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            dev.copy_(host, non_blocking=True)
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm.item())
        return ms / steps
    ms_h2d = None
    if group == 1:   # (a group context spreads the batch over its GPUs from one host buffer: the per-rank floor does not apply)
        copies_only(1)
        ms_h2d = copies_only(max(3, min(args.steps, 5)))
    # the real caller hands pageable memory (a pcl::PointCloud): same call, ordinary numpy buffer
    pageable = np.array(host.numpy(), copy=True)
    step(pageable)
    ms_pageable, _, _ = timed(pageable, max(2, min(args.steps, 3)))
    ms_pageable /= max(2, min(args.steps, 3))

    if rank == 0:
        hbm, tf_burst, tf_sust, src = peaks()
        info = gs.info
        W_step = acc["windows"] / args.steps          # this rank
        value = acc["windows_all"] / (ms_dev * 1e-3)
        e2e = acc2["windows_all"] / (ms_e2e * 1e-3)
        svm_launches = accs["chunks"]
        svm_ms = accs["svm"] / max(svm_launches, 1)
        flops_per_window = info.n_sv * (2.0 * info.n_dims + 4.0)   # SURVEY 8d: W*S*(2D+4)
        svm_tflops = (acc["windows"] / max(svm_launches, 1)) * flops_per_window / (svm_ms * 1e-3) / 1e12 if svm_ms > 0 else 0.0
        # MEASURED_PEAKS.json: the burst figure is for a kernel timed alone / in a short region, the sustained one for a region
        # long enough to sit under the power cap (it was measured over 4 s): the timed region decides
        timed_s = ms_dev * 1e-3
        burst = timed_s < 1.0
        peak = tf_burst if burst else tf_sust
        t_last = gs.timing()
        tck = {0: "svm_rbf_tc3_kernel" if (t_last.tc_passes == 1 and args.tc_variant == 0) else "svm_rbf_tc2_kernel", 1: "svm_rbf_tc_kernel",
               2: "svm_rbf_tc2_kernel"}[args.tc_variant]
        kname = {2: "svm_rbf_simt_kernel", 1: "svm_exact_terms_kernel", 0: tck}[args.svm_mode]
        traffic = None
        try:  # DRAM bytes of the dominant kernel from the committed ncu --set full capture, if it is the same launch size
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                tr = json.load(fh).get(kname)
            w_launch = acc["windows"] / max(svm_launches, 1)
            if tr and tr["n_sv"] == info.n_sv and abs(tr["windows_per_launch"] - w_launch) <= 0.01 * w_launch and (args.svm_mode != 0 or tr.get("passes", 3) == t_last.tc_passes):
                traffic = tr["dram_bytes_per_launch"]
        except Exception:
            traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world * group, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype_of(args.svm_mode, t_last.tc_passes), "data": "synthetic",
            "config": {"workload": describe(args, wc), "tensor_passes": int(t_last.tc_passes), "guard_rel": info.reserved[1] * 1e-9, "n_sv": info.n_sv, "n_dims": info.n_dims, "grid": info.grid,
                       "rolls": info.n_rolls, "clouds_per_gpu": n_clouds, "windows_per_step_per_gpu": W_step,
                       "svm_mode": args.svm_mode, "l2": "inputs (%.0f MB per GPU per step) larger than L2, no flush" % (total_pts * 12 / 1e6),
                       "sharding": ("one process, one C-ABI context over %d GPUs (haf_config.n_devices): clouds in contiguous blocks per GPU, one host thread "
                                    "and stream each, records merged on the host; timed by wall clock" % group) if group > 1 else
                                   "clouds by rank, no data-path collective; NCCL all_gather of best-grasp records"},
            "ms_per_cloud": ms_dev / args.steps / n_clouds,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": total_pts * 12 + 0, "d2h_bytes_per_step": n_clouds * (32 + info.n_rolls * 12) + 64, "host_memory": "pinned",
                    "ms_per_step": ms_e2e / args.steps,
                    "stage_ms_per_step": {k: acc2p[k] / n_prof for k in ("bin", "integral", "mask", "features", "svm", "guard", "score")},
                    "stage_note": "stages from a separate pass of %d steps with per-stage events on (%.3f ms per step); the chunks of a host-staged batch alternate "
                                  "between several streams, so stage times overlap and sum to more than the step" % (n_prof, ms_e2e_prof / n_prof),
                    "chunks_per_step": acc2["chunks"] / args.steps,
                    "h2d_only_ms_per_step": ms_h2d, "h2d_only_GBps_per_gpu": (total_pts * 12 / (ms_h2d * 1e-3) / 1e9) if ms_h2d else None,
                    "frac_of_h2d_ceiling": (ms_h2d / (ms_e2e / args.steps)) if ms_h2d else None,
                    "note": "h2d_only = the step's input bytes copied host->device from the same pinned buffers by all ranks at once, nothing else "
                            "(the floor of any end-to-end number on this host); frac_of_h2d_ceiling = that floor / the measured end-to-end step",
                    "pageable_ms_per_step": ms_pageable, "pageable_value": acc2["windows_all"] / args.steps / (ms_pageable * 1e-3)},
            "gpu_launches": int(acc["launches"]),
            "roofline": {"kernel": kname, "bound": "tensor",
                         "achieved": svm_tflops, "peak": peak, "unit": "TFLOP/s", "frac": svm_tflops / peak if peak else None,
                         "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                         "algorithmic_bytes": 4.0 * info.n_dims * (acc["windows"] / max(svm_launches, 1) + info.n_sv) + 4.0 * acc["windows"] / max(svm_launches, 1),
                         "peak_source": src + (" bf16 burst (timed region %.2f s < 1 s)" % timed_s if burst else " bf16 sustained (timed region %.1f s)" % timed_s),
                         "frac_of_sustained": svm_tflops / tf_sust if tf_sust else None, "frac_of_burst": svm_tflops / tf_burst if tf_burst else None,
                         "algorithmic": "W*S*(2D+4) flop per launch, W=%.0f S=%d D=%d" % (acc["windows"] / max(svm_launches, 1), info.n_sv, info.n_dims),
                         "kernel_ms": svm_ms, "share_of_step": accs["svm"] / ms_dev_prof if ms_dev_prof else None,
                         "note": {2: "FP32 SIMT contraction (CUDA cores), measured against the bf16 tensor peak for comparability",
                                  1: "FP64 exact-order path", 0: "algorithmic flops; the split-fp16 scheme issues %d tensor-core MMA(s) per algorithmic MMA (calibrated per model: "
                                  "config.tensor_passes, audited per call), executed tensor flops = passes x (Krow/D) x algorithmic" % t_last.tc_passes}[args.svm_mode]},
            "audit": {"sample_windows_per_step": acc["auditw"] / args.steps, "max_rel_error_of_E": t_last.audit_max_rel, "escalations": int(t_last.escalations),
                      "note": "max |dec_tensor - dec_fp64| / (E + |rho|) over the guard band's and the 1-in-4096 sample's windows of the last step; the guard band is guard_rel wide"},
            "stage_ms_per_step": {k: accs[k] / args.steps for k in ("bin", "integral", "mask", "features", "svm", "guard", "score")},
            "stage_source": "per-stage CUDA events inside the timed region" if prof_in_timed else
                            "a second pass of %d steps with per-stage events on (%.4f ms per step; the timed region runs without them: %.4f ms)" % (args.steps, ms_dev_prof / args.steps, ms_dev / args.steps),
            "cuda_graph": {"enabled": bool(args.graph), "replays_in_timed_region_and_warmup": graph_replays},
            "stage_roofline": stage_roofline(accs, args.steps, total_pts, n_clouds * info.n_rolls, info.grid, info.n_dims, W_step, hbm),
            "guard_windows_per_step": acc["guardw"] / args.steps,
            "wall_ms_per_step": 1e3 * wall_dev / args.steps,
        }
        if world == 1 and not args.no_cpu_baseline:
            ns = min(args.cpu_sample_clouds, n_clouds)
            skw = {"area": (100.0, 100.0), "roll_limit": 1} if args.workload == "grid512" else {}
            rate, w, dt, kind = cpu_reference_rate(args, wc, clouds[:ns], 1, model, **skw)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": kind,
                                    "sample": "%sfirst %d cloud(s) of the same workload, %s, %d windows in %.1f s; %s" % (
                                        "roll 0 of a 100x100 cm sub-area; " if skw else "", ns, "1 roll" if skw else "all 12 rolls", w, dt, "reference feature classes + svm-scale/svm-predict child processes on text files"
                                        if kind == "reference" else "in-process oracle port")}
        emit(line)
    gs.close()
    if world > 1:
        dist.destroy_process_group()


def stage_roofline(acc, steps, n_points, n_units, G, D, W, hbm_gbs):
    """HBM-bound stages against the measured copy bandwidth: ALGORITHMIC bytes per step (SURVEY 8d) / stage time.
    bin: 12 N + 4 U G^2; integral: 4 U G^2 + 4 U (G+1)^2; mask + Haar + scale: 4 U (G+1)^2 + U G^2 + 4 D W (the operand
    matrix counted once, FP32, as 8d defines it); stencil + argmax: U G^2 + 4 U G^2 + 32 U."""
    GG, LL = G * G, (G + 1) * (G + 1)
    rows = {"bin": (12.0 * n_points + 4.0 * n_units * GG, acc["bin"]),
            "integral": (4.0 * n_units * GG + 4.0 * n_units * LL, acc["integral"]),
            "mask+features": (4.0 * n_units * LL + n_units * GG + 4.0 * D * W, acc["mask"] + acc["features"]),
            "score": (5.0 * n_units * GG + 32.0 * n_units, acc["score"])}
    out = {}
    for k, (b, ms_total) in rows.items():
        ms = ms_total / steps
        gbs = b / (ms * 1e-3) / 1e9 if ms > 0 else None
        out[k] = {"algorithmic_bytes": b, "ms": ms, "GBps": gbs, "frac_of_hbm_peak": (gbs / hbm_gbs) if gbs and hbm_gbs else None}
    return out


_JSON_OUT = None


def protect_stdout():
    """Everything that is not the ONE JSON line (NCCL's version banner, library chatter) goes to stderr: fd 1 is
    pointed at stderr and the JSON line is written to a private duplicate of the original stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    protect_stdout()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "approach" or (args.workload == "grid512" and int(os.environ.get("WORLD_SIZE", "1")) > 1):
        run_approach(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
