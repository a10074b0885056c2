"""What searching depth images directly buys, on one GPU: the images cross PCIe at 2 bytes per pixel instead of 12 per point.

  python tools/depth_bench.py [--iters 7] [--images 512] [--out profiles/depth.json]

Workload: `--images` synthetic heightfield scenes (haf_grasping_b200.synth surface, 150 k points each) rendered as 320 x 320
U16 depth images (millimetres) by a camera 0.7 m above the scene looking straight down (fx = fy = 380, cx = cy = 159.5); the
default request for every image, grasp poses on.  Routes, alternated within the run:
  a_pinned / a_pageable  search_batch_depth on the image stack (pinned torch tensor / numpy array)
  b_numpy                numpy back-projection (the contract of include/hafgpu.h) into pinned xyz, then search_batch_requests:
                         what a caller does without this entry point
  c_resident             search_batch_requests on the clouds already in device memory (no ingest at all: the floor)
Per call: wall time (host clock around the call, which ends in a stream synchronise), median after a warm-up round.  Kernel:
depth_project_kernel's device time on device-resident images (torch.profiler, its own pass), bytes = 2 read + 12 written
per pixel, against the 7.7 TB/s HBM3e data-sheet figure; and the whole call with its tables prebuilt (CUDA events on the
library's stream, which is the default stream).  The outputs of a, b and c are compared record for record.  Prints one JSON document with
the card's name and power limit next to the numbers.
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

H = W = 320
CAM = (380.0, 380.0, 159.5, 159.5)
HEIGHT = 0.7


def camera_pose():
    import numpy as np
    M = np.eye(4, dtype=np.float32)
    M[:3, :3] = [[1, 0, 0], [0, -1, 0], [0, 0, -1]]
    M[2, 3] = HEIGHT
    return M


def render(xyz, pose):
    import numpy as np
    M = pose.astype(np.float64)
    c = (xyz.astype(np.float64) - M[:3, 3]) @ M[:3, :3]
    u = np.round(CAM[0] * c[:, 0] / c[:, 2] + CAM[2])
    v = np.round(CAM[1] * c[:, 1] / c[:, 2] + CAM[3])
    ok = (c[:, 2] > 0.05) & (u >= 0) & (u < W) & (v >= 0) & (v < H)
    depth = np.full(H * W, np.inf)
    np.minimum.at(depth, (v[ok] * W + u[ok]).astype(np.int64), c[ok, 2])
    return np.where(np.isfinite(depth), np.round(depth * 1000.0), 0).astype(np.uint16).reshape(H, W)


def back_project(stack, pose, out):
    """numpy float32 restatement of haf_depth_to_xyz_batch (U16, default scale, has_pose) into out [N * H * W, 3]"""
    import numpy as np
    s = np.float32(0.001)
    kx, ky = np.float32(float(s) / CAM[0]), np.float32(float(s) / CAM[1])
    cxf, cyf = np.float32(CAM[2]), np.float32(CAM[3])
    v, u = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
    m = pose.astype(np.float32)
    o = out.reshape(len(stack), H, W, 3)
    with np.errstate(all="ignore"):
        for i, img in enumerate(stack):
            D = img.astype(np.float32)
            x = ((u - cxf) * D) * kx
            y = ((v - cyf) * D) * ky
            z = D * s
            for r in range(3):
                o[i, :, :, r] = ((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3]
            o[i][img == 0] = np.float32("nan")
    return out


def records(res):
    return [bytes(b) for b in res["best"]] + [bytes(g) for g in res["grasp"]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=7)
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--kernel-iters", type=int, default=50)
    ap.add_argument("--out", help="also write the JSON document to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    import haf_grasping_b200 as h
    from haf_grasping_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("depth_bench.py: no CUDA device (libhafgpu has no CPU fallback)")
    n = args.images
    pose = camera_pose()
    t0 = time.perf_counter()
    stack = np.stack([render(synth.synth_cloud(1000 + i, 150000), pose) for i in range(n)])
    render_s = time.perf_counter() - t0
    model = os.path.join(tempfile.mkdtemp(prefix="haf_depth_"), "synth_2048_seed7.model")
    synth.write_synth_model(model, n_sv=2048, seed=7)
    gs = h.GraspSearch(FEATURES, RANGE, model)
    reqs = h.make_requests(n)
    pinned = torch.empty(stack.shape, dtype=torch.int16, pin_memory=True)
    pinned.numpy()[:] = stack.view(np.int16)
    dev_img = torch.from_numpy(stack.view(np.int16)).cuda()
    npix = n * H * W
    xyz_pinned = torch.empty((npix, 3), dtype=torch.float32, pin_memory=True)
    back_project(stack, pose, xyz_pinned.numpy())
    xyz_dev = xyz_pinned.cuda()
    po = np.arange(n + 1, dtype=np.int64) * H * W

    def route_b():
        back_project(stack, pose, xyz_pinned.numpy())
        return gs.search_batch_requests(xyz_pinned, po, reqs)

    calls = {"a_pinned": lambda: gs.search_batch_depth(pinned, CAM, pose),
             "a_pageable": lambda: gs.search_batch_depth(stack, CAM, pose),
             "b_numpy": route_b,
             "c_resident": lambda: gs.search_batch_requests(xyz_dev, po, reqs)}
    outs = {k: fn() for k, fn in calls.items()}          # warm-up round, outputs kept for the comparison
    ref = records(outs["c_resident"])
    equal = {k: records(v) == ref for k, v in outs.items()}
    got = gs.depth_to_xyz_batch_to_host(dev_img, CAM, pose)
    want = xyz_pinned.numpy()
    nan_w = np.isnan(want)
    xyz_equal = bool(np.array_equal(np.isnan(np.concatenate(got)), nan_w) and
                     np.array_equal(np.concatenate(got).view(np.uint32)[~nan_w], want.view(np.uint32)[~nan_w]))
    wall = {k: [] for k in calls}
    for _ in range(args.iters):
        for k, fn in calls.items():
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            fn()
            wall[k].append((time.perf_counter() - t1) * 1e3)
    # the kernel alone: device-resident images, the batch tables built once (the Python loop over 512 records would otherwise
    # set the pace); events around many calls, and the kernel's own device time from torch.profiler in a separate pass
    tables = gs._depth_batch(dev_img, CAM, pose, 0.0)[:3]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gs.depth_to_xyz_batch(tables)
    torch.cuda.synchronize()
    per_call = []
    for _ in range(5):
        ev0.record()
        for _ in range(args.kernel_iters):
            gs.depth_to_xyz_batch(tables)
        ev1.record()
        torch.cuda.synchronize()
        per_call.append(ev0.elapsed_time(ev1) / args.kernel_iters)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.kernel_iters):
            gs.depth_to_xyz_batch(tables)
        torch.cuda.synchronize()
    kern = [e.device_time_total / e.count / 1e3 for e in prof.key_averages() if "depth_project_kernel" in e.key]
    if not kern:
        raise SystemExit("depth_bench.py: the profiler saw no depth_project_kernel")
    k_ms = kern[0]
    k_bytes = npix * (2 + 12)
    med = {k: statistics.median(v) for k, v in wall.items()}
    doc = {"card": card(), "model": "synthetic, 2048 SVs (seed 7)", "svm_mode": "tensor (default)", "iters": args.iters,
           "images": n, "height": H, "width": W, "camera": CAM, "camera_height_m": HEIGHT, "render_s": render_s,
           "image_bytes": int(stack.nbytes), "xyz_bytes": int(npix * 12),
           "timing": "wall ms per call (host clock, the call ends in a stream synchronise), median after one warm-up round",
           "wall_ms_median": med, "wall_ms_all": wall,
           "a_pinned_minus_c_ms": med["a_pinned"] - med["c_resident"], "b_numpy_minus_c_ms": med["b_numpy"] - med["c_resident"],
           "kernel": {"what": "depth_project_kernel on device-resident images: mean device time over %d launches (torch.profiler)"
                              % args.kernel_iters,
                      "ms": k_ms, "bytes": k_bytes, "GB_per_s": k_bytes / k_ms / 1e6, "share_of_7700_GB_per_s": k_bytes / k_ms / 1e6 / 7700.0,
                      "call_ms": statistics.median(per_call), "call_ms_all": per_call,
                      "call_what": "depth_to_xyz_batch with prebuilt tables on device-resident images (parameter copy + launch), "
                                   "CUDA events, median of 5 windows of %d calls" % args.kernel_iters},
           "outputs_equal_to_c": equal, "xyz_equal_to_numpy": xyz_equal}
    ok = all(equal.values()) and xyz_equal
    doc["outputs_equal"] = ok
    gs.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    if not ok:
        raise SystemExit("depth_bench.py: the routes' outputs differ")


if __name__ == "__main__":
    main()
