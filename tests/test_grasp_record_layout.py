"""CPU: the ctypes haf_grasp of the Python binding has the C struct's size and field offsets (include/hafgpu.h), checked
against an offsetof probe compiled with the host compiler."""
import ctypes as C
import os
import subprocess

from conftest import ROOT

FIELDS = ["eval", "roll", "graspPoint1", "graspPoint2", "averagedGraspPoint", "approachVector", "row", "col", "roll_index", "reserved"]


def test_haf_grasp_layout_matches_the_header(tmp_path):
    from haf_grasping_b200.api import haf_grasp
    src = tmp_path / "probe.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"hafgpu.h\"\nint main(void) {\n"
                   "    printf(\"size %zu\\n\", sizeof(haf_grasp));\n" +
                   "".join("    printf(\"%s %%zu\\n\", offsetof(haf_grasp, %s));\n" % (f, f) for f in FIELDS) +
                   "    return 0;\n}\n")
    exe = str(tmp_path / "probe")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(haf_grasp)
    for f in FIELDS:
        assert int(got[f]) == getattr(haf_grasp, f).offset, f
    assert [f[0] for f in haf_grasp._fields_] == FIELDS
