"""What the device-side grasp poses cost: each workload is timed with the plain entry point and with its _grasps
counterpart, the two alternating call by call after a warm-up, on one GPU.

  python tools/grasp_output_overhead.py [--goal-iters 2000] [--batch-iters 20] [--out FILE.json]

Workloads (the same inputs as bench.py's table1 and batch workloads, 2048-SV synthetic model):
  goal   the table1 scene, default request, CUDA graphs on: haf_search vs haf_search_grasps
  batch  512 synthetic clouds x 100 k points, device-resident and from pinned host memory:
         haf_search_batch_packed vs haf_search_batch_packed_grasps
Per call: wall time (host clock around the call, which ends in a stream synchronise) and device time (haf_timing.ms_total,
CUDA events on the call's stream); medians over the alternating calls.  Prints one JSON document with the card's name and
power limit next to the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FEATURES = os.path.join(ROOT, "tests", "golden", "refdata", "Features.txt")
RANGE = os.path.join(ROOT, "tests", "golden", "refdata", "range21062012_allfeatures")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, plimit, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": plimit, "clocks_max_sm": clk}
    except Exception as exc:   # the numbers are still the card's; say that its description could not be read
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % exc}


def alternate(gs, calls, iters, warmup):
    """calls: {label: fn}; runs them in turn iters times after warmup rounds; per-call wall and device ms"""
    for _ in range(warmup):
        for fn in calls.values():
            fn()
    wall = {k: [] for k in calls}
    dev = {k: [] for k in calls}
    for _ in range(iters):
        for k, fn in calls.items():
            t0 = time.perf_counter()
            fn()
            wall[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(gs.timing().ms_total)
    res = {}
    for k in calls:
        res[k] = {"wall_ms_median": statistics.median(wall[k]), "device_ms_median": statistics.median(dev[k]),
                  "wall_ms_min": min(wall[k]), "device_ms_min": min(dev[k]), "calls": iters}
    return res


def added(res, plain, grasp):
    return {"wall_ms_median": res[grasp]["wall_ms_median"] - res[plain]["wall_ms_median"],
            "device_ms_median": res[grasp]["device_ms_median"] - res[plain]["device_ms_median"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--goal-iters", type=int, default=2000)
    ap.add_argument("--batch-iters", type=int, default=20)
    ap.add_argument("--clouds", type=int, default=512)
    ap.add_argument("--points", type=int, default=100000)
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import haf_grasping_b200 as h
    from haf_grasping_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("grasp_output_overhead.py: no CUDA device (libhafgpu has no CPU fallback)")
    model = os.path.join(tempfile.mkdtemp(prefix="haf_grasp_cost_"), "synth_2048_seed7.model")
    synth.write_synth_model(model, n_sv=2048, seed=7)
    doc = {"card": card(), "model": "synthetic, 2048 SVs (seed 7)", "svm_mode": "tensor (default)"}

    # ---- one goal: table1, default request, CUDA graphs on
    xyz = np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "clouds.npz"))["table1"])
    gs = h.GraspSearch(FEATURES, RANGE, model, use_graph=True)
    rq = [h.make_request()]
    res = alternate(gs, {"haf_search": lambda: gs.search(xyz, rq, outputs=False),
                         "haf_search_grasps": lambda: gs.search_grasps(xyz, rq)}, args.goal_iters, 50)
    res["graph_replays"] = gs.timing().graph_replays
    res["added"] = added(res, "haf_search", "haf_search_grasps")
    doc["goal_table1_graph"] = res
    gs.close()

    # ---- the batch: 512 clouds x 100 k points, resident and from pinned host memory
    clouds = [synth.synth_cloud(1234 + i, args.points, r=0.28) for i in range(args.clouds)]
    off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    host = torch.empty((int(off[-1]), 3), dtype=torch.float32, pin_memory=True)
    host.numpy()[:] = np.concatenate(clouds)
    dev = host.cuda()
    gs = h.GraspSearch(FEATURES, RANGE, model)
    brq = h.make_request()
    for label, buf in (("resident", dev), ("pinned", host)):
        res = alternate(gs, {"haf_search_batch_packed": lambda: gs.search_batch_packed(buf, off, brq),
                             "haf_search_batch_packed_grasps": lambda: gs.search_batch_packed_grasps(buf, off, brq)},
                        args.batch_iters, 3)
        res["n_chunks"] = gs.timing().n_chunks
        res["added"] = added(res, "haf_search_batch_packed", "haf_search_batch_packed_grasps")
        doc["batch_%dx%dk_%s" % (args.clouds, args.points // 1000, label)] = res
    gs.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
