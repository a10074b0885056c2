"""What per-cloud requests cost in a batch (haf_search_batch_requests), on one GPU.

  python tools/batch_requests_bench.py [--iters 20] [--clouds 512] [--points 100000] [--out profiles/batch_requests.json]

Inputs: 512 synthetic clouds x 100 k points (bench.py's batch), 2048-SV synthetic model, grasp poses on; each workload
device-resident and from pinned host memory:
  a  identical   the default request for every cloud: haf_search_batch_requests vs haf_search_batch_packed_grasps, alternating
  b  centres     one request per cloud with its own grasp-area centre (changes the windows, so they are reported)
  c  approaches  one request per cloud with its own random approach vector: a table entry per job
  d  five        configs[2]'s five approach vectors per cloud (2560 requests)
Per call: wall time (host clock around the call, which ends in a stream synchronise) and device time (haf_timing.ms_total);
medians after a warm-up.  Host time from entry to the first kernel launch (device-resident): the C entry point called
directly with prepared arguments (no Python marshalling), the span from its entry to the CPU-side launch record of its first
kernel (copy_params_kernel) in a torch.profiler trace, median over 10 calls, for the new call and for
haf_search_batch_packed_grasps.  Prints one JSON document with the card's name and power limit next to the numbers.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from grasp_output_overhead import FEATURES, RANGE, alternate, card  # noqa: E402

TILTED = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254)]


def host_to_first_launch_ms(fn, calls=10):
    """entry of fn -> CPU start of its first kernel launch, from a torch.profiler trace"""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile, record_function
    fn()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            with record_function("haf_call"):
                fn()
    ev = prof.events()
    spans = sorted((e.time_range.start, e.time_range.end) for e in ev if e.name == "haf_call" and e.device_type == DeviceType.CPU)
    launches = sorted(e.time_range.start for e in ev if e.name in ("cudaLaunchKernel", "cudaLaunchKernelExC", "cuLaunchKernel", "cuLaunchKernelEx"))
    out = []
    for s, t in spans:
        first = [x for x in launches if s <= x <= t]
        if first:
            out.append((first[0] - s) / 1e3)
    torch.cuda.synchronize()
    return {"median_ms": statistics.median(out), "calls": len(out)} if out else "not measured (no launch record in the profiler trace)"


def _cargs(gs, buf, off):
    import ctypes as C
    n = len(off) - 1
    return C.c_void_p(buf.data_ptr()), (C.c_size_t * len(off))(*[int(o) for o in off]), n


def direct_requests(gs, buf, off, reqs, ro):
    import ctypes as C

    import haf_grasping_b200 as h
    ptr, coff, n = _cargs(gs, buf, off)
    roff = None if ro is None else (C.c_int * len(ro))(*[int(o) for o in ro])
    best, bpr, grasp = (h.haf_best * n)(), (h.haf_best * len(reqs))(), (h.haf_grasp * n)()
    return lambda: gs._check(gs.L.haf_search_batch_requests(gs.h, ptr, coff, n, reqs, roff, best, bpr, None, grasp, None, None))


def direct_packed(gs, buf, off, rq):
    import ctypes as C

    import haf_grasping_b200 as h
    ptr, coff, n = _cargs(gs, buf, off)
    best, grasp = (h.haf_best * n)(), (h.haf_grasp * n)()
    return lambda: gs._check(gs.L.haf_search_batch_packed_grasps(gs.h, ptr, coff, n, C.byref(rq), best, grasp, None))


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
        raise SystemExit("batch_requests_bench.py: no CUDA device (libhafgpu has no CPU fallback)")
    model = os.path.join(tempfile.mkdtemp(prefix="haf_batch_requests_"), "synth_2048_seed7.model")
    synth.write_synth_model(model, n_sv=2048, seed=7)
    doc = {"card": card(), "model": "synthetic, 2048 SVs (seed 7)", "svm_mode": "tensor (default)",
           "batch": "%d synthetic clouds x %d points" % (args.clouds, args.points)}

    n = args.clouds
    clouds = [synth.synth_cloud(1234 + i, args.points, r=0.28) for i in range(n)]
    off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
    host = torch.empty((int(off[-1]), 3), dtype=torch.float32, pin_memory=True)
    host.numpy()[:] = np.concatenate(clouds)
    dev = host.cuda()
    rng = np.random.default_rng(5)
    av = rng.normal(size=(n, 3))
    av[:, 2] = np.abs(av[:, 2]) + 1.0
    workloads = {
        "a_identical": (h.make_requests(n), None),
        "b_centres": (h.make_requests(centers=rng.uniform(-0.05, 0.05, (n, 3))), None),
        "c_approaches": (h.make_requests(approaches=av), None),
        "d_five": (h.make_requests(approaches=np.tile(np.array(TILTED), (n, 1))), np.arange(0, 5 * n + 1, 5)),
    }
    gs = h.GraspSearch(FEATURES, RANGE, model)
    rq = h.make_request()
    for label, buf in (("resident", dev), ("pinned", host)):
        res = {}
        for name, (reqs, ro) in workloads.items():
            calls = {"haf_search_batch_requests": (lambda reqs=reqs, ro=ro: gs.search_batch_requests(buf, off, reqs, ro))}
            if name == "a_identical":
                calls["haf_search_batch_packed_grasps"] = lambda: gs.search_batch_packed_grasps(buf, off, rq)
            r = alternate(gs, calls, args.iters, 3)
            calls["haf_search_batch_requests"]()
            t = gs.timing()
            r["requests"], r["windows"], r["n_chunks"] = len(reqs), t.n_windows, t.n_chunks
            if name == "a_identical":
                r["added"] = {k: r["haf_search_batch_requests"][k] - r["haf_search_batch_packed_grasps"][k]
                              for k in ("wall_ms_median", "device_ms_median")}
            r["windows_per_cloud"] = t.n_windows / n
            if label == "resident":
                r["host_entry_to_first_launch"] = host_to_first_launch_ms(direct_requests(gs, buf, off, reqs, ro))
                if name == "a_identical":
                    r["host_entry_to_first_launch_batch_packed_grasps"] = host_to_first_launch_ms(direct_packed(gs, buf, off, rq))
            res[name] = r
        doc["batch_%s" % label] = res
    gs.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
