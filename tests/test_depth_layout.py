"""ctypes layout of haf_depth_image (haf_grasping_b200/api.py) against the C header: size and field offsets (include/hafgpu.h),
checked against an offsetof probe compiled with the host compiler."""
import ctypes as C
import os
import subprocess

from conftest import ROOT

FIELDS = ["width", "height", "encoding", "has_pose", "step", "fx", "fy", "cx", "cy", "depth_scale", "camera_to_base", "reserved"]


def test_layout_matches_the_header(tmp_path):
    from haf_grasping_b200 import api
    src = tmp_path / "probe.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"hafgpu.h\"\nint main(void) {\n"
                   "    printf(\"size %zu\\n\", sizeof(haf_depth_image));\n"
                   "    printf(\"U16 %d\\n\", HAF_DEPTH_U16);\n    printf(\"F32 %d\\n\", HAF_DEPTH_F32);\n" +
                   "".join("    printf(\"%s %%zu\\n\", offsetof(haf_depth_image, %s));\n" % (f, f) for f in FIELDS) +
                   "    return 0;\n}\n")
    exe = str(tmp_path / "probe")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(api.haf_depth_image) == 136
    assert int(got["U16"]) == api.HAF_DEPTH_U16 and int(got["F32"]) == api.HAF_DEPTH_F32
    for f in FIELDS:
        assert int(got[f]) == getattr(api.haf_depth_image, f).offset, f
    assert [f[0] for f in api.haf_depth_image._fields_] == FIELDS
    assert api.haf_depth_image.camera_to_base.size == 64 and api.haf_depth_image.reserved.size == 12


def test_batch_tables_from_arrays():
    """the byte offsets, steps and records the Python binding builds for a list of images (no device involved)"""
    import numpy as np
    from haf_grasping_b200.api import GraspSearch, HAF_DEPTH_F32, HAF_DEPTH_U16
    a = np.arange(12, dtype=np.uint16).reshape(3, 4)
    padded = np.zeros((3, 7), np.uint16)
    padded[:, :4] = a
    f = np.full((2, 5), 1.5, np.float32)
    pose = np.arange(16, dtype=np.float32).reshape(4, 4)
    data, off, recs, n = GraspSearch._depth_batch([a, padded[:, :4], np.zeros((0, 5), np.float32), f], (500.0, 510.0, 2.5, -1.0),
                                                  [None, pose, None, pose], [0.0, 0.0002, 0.0, 1.0])
    assert n == 4 and list(off) == [0, 24, 66, 66, 106]
    assert [(r.width, r.height, r.step, r.encoding, r.has_pose) for r in recs] == [
        (4, 3, 8, HAF_DEPTH_U16, 0), (4, 3, 14, HAF_DEPTH_U16, 1), (5, 0, 20, HAF_DEPTH_F32, 0), (5, 2, 20, HAF_DEPTH_F32, 1)]
    assert data[:24].view(np.uint16).tolist() == a.reshape(-1).tolist()
    assert data[24:66].view(np.uint16).reshape(3, 7)[:, :4].tolist() == a.tolist()
    assert data[66:].view(np.float32).tolist() == [1.5] * 10
    assert list(recs[1].camera_to_base) == list(range(16)) and (recs[1].fx, recs[1].fy, recs[1].cx, recs[1].cy) == (500.0, 510.0, 2.5, -1.0)
    assert recs[1].depth_scale == np.float32(0.0002) and recs[0].depth_scale == 0.0
