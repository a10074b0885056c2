"""What decoding a batch of PCD files on the device in one call buys, on one GPU.

  python tools/batch_pcd_bench.py [--iters 5] [--out profiles/batch_pcd.json]

Workloads (each > 126 MB of L2 as a whole; every file is its own copy in the batch buffer):
  compressed  512 binary_compressed files cycling the bundled table1 / table2 / table3 bytes (74-103 k points, ~10 B per point)
  binary      the same 512 clouds as DATA binary files (12 B per point)
  ascii       64 ASCII files of the same clouds ("%.9g", exact round trip)
Routes, alternated within the run (default request for every cloud, grasp poses on):
  a_pageable / a_pinned  search_batch_pcd on the batch buffer (numpy array / pinned torch tensor)
  b_loop                 pcd_decode per file + a device-to-device copy into one buffer, then search_batch_requests on it
  c_decoded              search_batch_requests on the already decoded clouds in pinned memory (no decode: the floor)
Per call: wall time (host clock around the call, which ends in a stream synchronise), median after a warm-up.  Decode only:
device time (CUDA events on the default stream, which the library's stream follows) of pcd_decode_batch from pinned memory vs
the pcd_decode + copy loop.  The outputs of a, b and c are compared record for record.  Prints one JSON document with the
card's name and power limit next to the numbers.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from grasp_output_overhead import FEATURES, RANGE, card  # noqa: E402


def pcd_text(xyz, kind):
    n = len(xyz)
    hdr = ("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\n"
           "WIDTH %d\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %d\nDATA %s\n" % (n, n, kind)).encode()
    if kind == "binary":
        return hdr + xyz.astype("<f4").tobytes()
    return hdr + "".join("%.9g %.9g %.9g\n" % tuple(p) for p in xyz.tolist()).encode()


class DeviceView:
    """a device pointer as a torch tensor (float32 [n, 3]) through __cuda_array_interface__"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n, 3), "typestr": "<f4", "data": (ptr, False), "version": 2, "strides": None}


def records(res):
    return [bytes(b) for b in res["best"]] + [bytes(g) for g in res["grasp"]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--files", type=int, default=512)
    ap.add_argument("--ascii-files", type=int, default=64)
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import haf_grasping_b200 as h
    from haf_grasping_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("batch_pcd_bench.py: no CUDA device (libhafgpu has no CPU fallback)")
    golden = os.path.join(ROOT, "tests", "golden")
    z = np.load(os.path.join(golden, "pcd_files.npz"))
    cl = np.load(os.path.join(golden, "clouds.npz"))
    tables = ("table1", "table2", "table3")
    model = os.path.join(tempfile.mkdtemp(prefix="haf_batch_pcd_"), "synth_2048_seed7.model")
    synth.write_synth_model(model, n_sv=2048, seed=7)
    doc = {"card": card(), "model": "synthetic, 2048 SVs (seed 7)", "svm_mode": "tensor (default)", "iters": args.iters,
           "timing": "wall ms per call (host clock, the call ends in a stream synchronise), median after one warm-up round"}
    gs = h.GraspSearch(FEATURES, RANGE, model)
    per_kind = {"compressed": {t: z[t].tobytes() for t in tables},
                "binary": {t: pcd_text(cl[t], "binary") for t in tables},
                "ascii": {t: pcd_text(cl[t], "ascii") for t in tables}}
    ok_all = True
    for kind, n_files in (("compressed", args.files), ("binary", args.files), ("ascii", args.ascii_files)):
        seq = [tables[i % 3] for i in range(n_files)]
        files = [per_kind[kind][t] for t in seq]
        blob = np.frombuffer(b"".join(files), np.uint8).copy()
        offs = np.cumsum([0] + [len(f) for f in files]).astype(np.int64)
        pinned = torch.empty(len(blob), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = blob
        po = np.cumsum([0] + [len(cl[t]) for t in seq]).astype(np.int64)
        xyz = torch.empty((int(po[-1]), 3), dtype=torch.float32, pin_memory=True)
        xyz.numpy()[:] = np.concatenate([cl[t] for t in seq])
        dst = torch.empty((int(po[-1]), 3), dtype=torch.float32, device="cuda")
        reqs = h.make_requests(n_files)

        def loop_decode():
            for f in range(n_files):
                d, n = gs.pcd_decode(files[f])
                dst[po[f]:po[f + 1]].copy_(torch.as_tensor(DeviceView(d, n), device="cuda"))

        def route_b():
            loop_decode()
            return gs.search_batch_requests(dst, po, reqs)

        calls = {"a_pageable": lambda: gs.search_batch_pcd((blob, offs), reqs),
                 "a_pinned": lambda: gs.search_batch_pcd((pinned, offs), reqs),
                 "b_loop": route_b,
                 "c_decoded": lambda: gs.search_batch_requests(xyz, po, reqs)}
        outs = {k: fn() for k, fn in calls.items()}     # warm-up round, outputs kept for the comparison
        ref = records(outs["c_decoded"])
        equal = {k: records(v) == ref for k, v in outs.items()}
        ok_all &= all(equal.values())
        wall = {k: [] for k in calls}
        for _ in range(args.iters):
            for k, fn in calls.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                wall[k].append((time.perf_counter() - t0) * 1e3)
        # decode only: device time of the batch decode (pinned source) vs the per-file loop, alternating
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        dec = {"batch_pinned": [], "loop": []}
        for _ in range(args.iters):
            torch.cuda.synchronize()
            ev[0].record()
            gs.pcd_decode_batch((pinned, offs))
            ev[1].record()
            ev[2].record()
            loop_decode()
            ev[3].record()
            torch.cuda.synchronize()
            dec["batch_pinned"].append(ev[0].elapsed_time(ev[1]))
            dec["loop"].append(ev[2].elapsed_time(ev[3]))
        med = {k: statistics.median(v) for k, v in wall.items()}
        doc[kind] = {
            "files": n_files, "bytes": int(len(blob)), "points": int(po[-1]),
            "wall_ms_median": med, "wall_ms_all": wall,
            "a_pinned_over_b": med["a_pinned"] / med["b_loop"], "a_pageable_over_b": med["a_pageable"] / med["b_loop"],
            "a_pinned_over_c": med["a_pinned"] / med["c_decoded"], "a_pageable_over_c": med["a_pageable"] / med["c_decoded"],
            "decode_device_ms_median": {k: statistics.median(v) for k, v in dec.items()},
            "outputs_equal_to_c": equal,
        }
        print(kind, json.dumps(doc[kind]["wall_ms_median"]), json.dumps(doc[kind]["decode_device_ms_median"]), equal, flush=True)
        del pinned, xyz, dst
    doc["outputs_equal"] = ok_all
    gs.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    if not ok_all:
        raise SystemExit("batch_pcd_bench.py: the routes' outputs differ")


if __name__ == "__main__":
    main()
