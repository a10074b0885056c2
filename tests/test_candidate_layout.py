"""CPU: the ctypes haf_rank_params and haf_candidate of the Python binding have the C structs' sizes and field offsets
(include/hafgpu.h), checked against an offsetof probe compiled with the host compiler."""
import ctypes as C
import os
import subprocess

import pytest

from conftest import ROOT

STRUCTS = {
    "haf_rank_params": ["k", "per_unit", "min_distance", "reserved"],
    "haf_candidate": ["grasp", "score", "request"],
}


@pytest.mark.parametrize("name", sorted(STRUCTS))
def test_layout_matches_the_header(tmp_path, name):
    from haf_grasping_b200 import api
    fields = STRUCTS[name]
    src = tmp_path / "probe.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"hafgpu.h\"\nint main(void) {\n"
                   "    printf(\"size %%zu\\n\", sizeof(%s));\n" % name +
                   "".join("    printf(\"%s %%zu\\n\", offsetof(%s, %s));\n" % (f, name, f) for f in fields) +
                   "    return 0;\n}\n")
    exe = str(tmp_path / "probe")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines())
    cls = getattr(api, name)
    assert int(got["size"]) == C.sizeof(cls)
    for f in fields:
        assert int(got[f]) == getattr(cls, f).offset, f
    assert [f[0] for f in cls._fields_] == fields


def test_candidate_is_128_bytes():
    from haf_grasping_b200.api import haf_candidate
    assert C.sizeof(haf_candidate) == 128
