"""What the ranked candidates cost (haf_search_batch_candidates against haf_search_batch_requests with grasp poses), on one GPU.

  python tools/candidates_bench.py [--iters 20] [--clouds 512] [--points 100000] [--out profiles/candidates.json]

Candidates: k = 16, per_unit = 64, min_distance = 0.03.  Workloads:
  batch_resident / batch_pinned  bench.py's batch (512 synthetic clouds x 100 k points, 2048-SV synthetic model), default request
  table1_graph                   the table1 scene (tests/golden/clouds.npz) as one goal, device-resident, CUDA graphs on
  grid512                        configs[3]: synthetic 1 M-point cloud, G = 512, area 362 x 362, 12 rolls, one goal
The two calls alternate in one run; per call the wall time (host clock around the call, which ends in a stream synchronise) and
the device time (haf_timing.ms_total), medians after a warm-up.  The new kernels' times come from a separate torch.profiler run
of the candidates call (CUDA activity; summed over the profiled calls, divided by their number).  The card's name and power limit are
read in the same run and printed next to the numbers.
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from grasp_output_overhead import FEATURES, RANGE, alternate, card  # noqa: E402

RANK = dict(k=16, per_unit=64, min_distance=0.03)
RANK_KERNELS = ("rank_unit_kernel", "rank_tile_kernel", "rank_cloud_kernel")


def kernel_times(fn, calls):
    """per-call device time of each rank kernel (us), from a torch.profiler trace of `calls` calls"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for kname in RANK_KERNELS:
        durs = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                for e in prof.events() if kname in e.name and e.device_type.name == "CUDA"]
        if durs:
            out[kname + "_us_per_call"] = sum(durs) / calls
            out[kname + "_launches_per_call"] = len(durs) / calls
    return out or "not measured (no rank kernel in the profiler trace)"


def compare(gs, buf, off, reqs, iters, warmup):
    calls = {"haf_search_batch_requests": lambda: gs.search_batch_requests(buf, off, reqs),
             "haf_search_batch_candidates": lambda: gs.search_batch_candidates(buf, off, reqs, **RANK)}
    r = alternate(gs, calls, iters, warmup)
    r["added"] = {k: r["haf_search_batch_candidates"][k] - r["haf_search_batch_requests"][k] for k in ("wall_ms_median", "device_ms_median")}
    r["kernels"] = kernel_times(calls["haf_search_batch_candidates"], min(iters, 10))
    calls["haf_search_batch_candidates"]()
    r["n_chunks"] = gs.timing().n_chunks
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--clouds", type=int, default=512)
    ap.add_argument("--points", type=int, default=100000)
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import haf_grasping_b200 as h
    from haf_grasping_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("candidates_bench.py: no CUDA device (libhafgpu has no CPU fallback)")
    tmp = tempfile.mkdtemp(prefix="haf_candidates_")
    model = os.path.join(tmp, "synth_2048_seed7.model")
    synth.write_synth_model(model, n_sv=2048, seed=7)
    doc = {"card": card(), "model": "synthetic, 2048 SVs (seed 7)", "svm_mode": "tensor (default)", "rank": RANK}

    n = args.clouds
    clouds = [synth.synth_cloud(1234 + i, args.points, r=0.28) for i in range(n)]
    off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    host = torch.empty((int(off[-1]), 3), dtype=torch.float32, pin_memory=True)
    host.numpy()[:] = np.concatenate(clouds)
    dev = host.cuda()
    gs = h.GraspSearch(FEATURES, RANGE, model)
    reqs = h.make_requests(n)
    doc["batch"] = "%d synthetic clouds x %d points, default request" % (n, args.points)
    doc["batch_resident"] = compare(gs, dev, off, reqs, args.iters, 3)
    doc["batch_pinned"] = compare(gs, host, off, reqs, args.iters, 3)
    gs.close()
    del dev, host

    g1 = h.GraspSearch(FEATURES, RANGE, model, use_graph=True)
    t1 = torch.from_numpy(np.ascontiguousarray(np.load(os.path.join(ROOT, "tests", "golden", "clouds.npz"))["table1"])).cuda()
    doc["table1_graph"] = compare(g1, t1, [0, len(t1)], h.make_requests(1), max(args.iters, 200), 10)
    doc["table1_graph"]["graph_replays"] = g1.timing().graph_replays
    g1.close()

    g5 = h.GraspSearch(FEATURES, RANGE, model, grid=512)
    x5 = torch.from_numpy(synth.synth_cloud(1234, 1000000, r=2.56)).cuda()
    doc["grid512"] = compare(g5, x5, [0, len(x5)], h.make_requests(1, areas=(362.0, 362.0)), max(3, args.iters // 4), 1)
    g5.close()

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
