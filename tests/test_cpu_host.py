"""CPU-side tests (no GPU): decimal text emulation vs glibc, C-ABI exports, loaders' host logic, PCD reader,
oracle golden pins."""
import ctypes as C
import gzip
import json
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE, ROOT


def test_decimal_round_emulation_matches_glibc(tmp_path):
    exe = str(tmp_path / "drc")
    subprocess.run(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-ffp-contract=off", "-o", exe,
                    os.path.join(ROOT, "tests", "decimal_round_check.cpp"), "-lm"], check=True)
    out = subprocess.run([exe, "400000", "11"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "mismatches=0" in out.stdout and "unsupported_text4=0" in out.stdout


def test_library_builds_and_exports_every_declared_symbol():
    from haf_grasping_b200 import api, build
    lib = build.build_lib()
    L = C.CDLL(lib)
    header = open(os.path.join(ROOT, "include", "hafgpu.h")).read()
    declared = set(re.findall(r"\b(haf_[a-z0-9_]+)\s*\(", header))
    assert declared == set(api.EXPORTS), declared ^ set(api.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name


def test_library_is_sm100a_native_tcgen05_tma_tmem_dmma():
    """The built library carries sm_100a SASS only, and the tensor kernels are tcgen05 / TMEM / TMA code (not mma.sync):
    UTCHMMA.2CTA (tcgen05.mma cta_group::2), UTMALDG (TMA loads), LDTM (tcgen05.ld), UTCBAR multicast commits in the SVM
    kernels; DMMA in the FP64 guard tier; RED.MAX in the binning kernels.  (cuobjdump runs without a GPU.)"""
    import shutil
    from haf_grasping_b200 import build
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    lib = build.build_lib()
    elf = subprocess.run([cuobjdump, "-lelf", lib], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"sm_\d+a?", elf))
    assert archs == {"sm_100a"}, archs
    out = subprocess.run([os.sys.executable, os.path.join(ROOT, "tools", "sass_excerpt.py")], capture_output=True, text=True, check=True).stdout
    blocks = {}
    for blk in out.split("## ")[1:]:
        name, _, body = blk.partition("\n")
        blocks[name.strip()] = body
    def ops(sub):
        found = [b for n, b in blocks.items() if sub in n]
        assert found, (sub, list(blocks))
        return found
    for body in ops("svm_rbf_tc3_kernelILi2") + ops("svm_rbf_tc2_kernel"):
        for op in ("UTCHMMA.2CTA", "UTMALDG.2D", "LDTM", "UTCBAR.2CTA.MULTICAST", "MUFU.EX2"):
            assert op in body, op
        assert "HMMA." not in body.replace("UTCHMMA", "")      # no mma.sync in the product kernels
    assert any("DMMA.8x8x4" in b for b in ops("guard_dmma_kernel"))
    assert all("REDG.E.MAX" in b for b in ops("bin_maxz_cloud_kernel"))


def test_docs_reference_existing_profile_files():
    """every `profiles/...` file the docs, the sources and the tests point at exists (evidence must be committed, not scratch)"""
    pat = re.compile(r"profiles/([A-Za-z0-9_][A-Za-z0-9_.\-]*\.(?:md|txt|json|csv))")
    files = [os.path.join(ROOT, f) for f in ("DESIGN.md", "README.md", "INTEGRATION.md", "bench.py", os.path.join("profiles", "README.md"))]
    for sub in (os.path.join("haf_grasping_b200", "csrc"), "tests", "include", "tools"):
        for dp, _, fn in os.walk(os.path.join(ROOT, sub)):
            files += [os.path.join(dp, f) for f in fn if f.endswith((".cu", ".cuh", ".hpp", ".h", ".py", ".sh", ".cpp"))]
    missing = set()
    for path in files:
        for name in pat.findall(open(path, errors="ignore").read()):
            if "NN" in name or "*" in name:
                continue
            if not os.path.exists(os.path.join(ROOT, "profiles", name)):
                missing.add((os.path.relpath(path, ROOT), name))
    assert not missing, sorted(missing)


def test_no_gpu_means_loud_failure_not_fallback(tmp_models):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import haf_grasping_b200 as h
    with pytest.raises(h.HafError) as e:
        h.GraspSearch(FEATURES, RANGE, tmp_models(256))
    assert e.value.code == -4


def test_host_transform_matches_oracle(oracle_lib):
    import haf_grasping_b200 as h
    o = oracle_lib.Oracle(FEATURES, RANGE)
    rng = np.random.default_rng(5)
    cases = [((0, 0, 0), (0, 0, 1), 1), ((0.1, -0.2, 0.05), (0.5, 0, 0.8660254), 1), ((0, 0, 0), (0, 0, -1), 2),
             ((0.3, 0.1, 0), (0.2, -0.7, 0.4), 3)]
    cases += [(tuple(rng.uniform(-1, 1, 3)), tuple(rng.uniform(-1, 1, 3)), int(rng.integers(1, 4))) for _ in range(20)]
    for center, av, width in cases:
        for roll in range(12):
            M = h.build_transform(h.make_request(center=center, approach=av, width=width), roll)
            M2 = o.build_transform(center, o.normalize_approach(av), width, roll)
            assert M.tobytes() == M2.tobytes()


def test_best_key_orders_like_the_reference_rule():
    import haf_grasping_b200 as h
    L = h.load_library()
    # strictly greater topval wins; equal topval -> the EARLIER unit wins (server.cpp:953 strict >)
    assert L.haf_best_key(90, 5) > L.haf_best_key(89, 0)
    assert L.haf_best_key(90, 3) > L.haf_best_key(90, 4)
    assert L.haf_best_key(-1000, 0) < L.haf_best_key(0, 100)


def _reference_pcd_file(tmp_path, name):
    """one of the reference's bundled PCD files, written back from its committed bytes (tests/golden/pcd_files.npz)"""
    path = tmp_path / (name + ".pcd")
    path.write_bytes(np.load(os.path.join(GOLDEN, "pcd_files.npz"))[name].tobytes())
    return str(path)


def test_pcd_reader_on_reference_files(tmp_path):
    from haf_grasping_b200.pcd import read_pcd
    clouds = np.load(os.path.join(GOLDEN, "clouds.npz"))
    a = read_pcd(_reference_pcd_file(tmp_path, "pcd4"))
    assert a.shape == (200, 3)  # POINTS 200 although the file carries 208 lines
    assert a.tobytes() == clouds["pcd4"].tobytes()
    t = read_pcd(_reference_pcd_file(tmp_path, "table1"))
    assert t.tobytes() == clouds["table1"].tobytes()


def test_pcd_roundtrip_formats(tmp_path):
    from haf_grasping_b200.pcd import read_pcd
    rng = np.random.default_rng(0)
    pts = rng.normal(size=(37, 3)).astype(np.float32)
    hdr = "# .PCD v0.7\nVERSION 0.7\nFIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 37\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 37\n"
    p = tmp_path / "b.pcd"
    p.write_bytes((hdr + "DATA binary\n").encode() + pts.tobytes())
    assert read_pcd(str(p)).tobytes() == pts.tobytes()
    p2 = tmp_path / "a.pcd"
    p2.write_text(hdr + "DATA ascii\n" + "\n".join(" ".join(repr(float(v)) for v in row) for row in pts) + "\nextra 1 2\n")
    assert read_pcd(str(p2)).tobytes() == pts.tobytes()


def test_oracle_reproduces_committed_pins(oracle_lib, tmp_path):
    """expected.json was written by the oracle; this guards the oracle (and the fixtures) against drift."""
    with open(os.path.join(GOLDEN, "expected.json")) as fh:
        exp = json.load(fh)
    model = str(tmp_path / "trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(model, "wb") as dst:
        dst.write(src.read())
    clouds = np.load(os.path.join(GOLDEN, "clouds.npz"))
    o = oracle_lib.Oracle(FEATURES, RANGE, model)
    for name in ("pcd2", "pcd7", "pcd4", "table1"):
        res = o.search(clouds[name], oracle_lib.make_request())
        e = exp["trained/" + name]
        assert list(res["best"].astuple()) == e["best"]
        assert res["per_roll_top"].tolist() == e["per_roll_top"]
        assert res["mask"].reshape(12, -1).sum(1).tolist() == e["mask_popcount"]


def test_oracle_quirks(oracle_lib):
    o = oracle_lib.Oracle(FEATURES, RANGE)
    assert o.F == 324                              # trailing blank line -> phantom feature (II2FV.cpp:60-82)
    reg, w = o.feature_table()
    assert (w[:, 3] == 0).all()                    # 4th region weight never set (Haar.cpp:55-60)
    patch = np.random.default_rng(1).uniform(0, 3, (15, 15)).astype(np.float32)
    f = o.featurevalues(patch)
    assert f[323] == -1.0                          # SHAF with every region skipped
    assert o.text4(0.123449) == 0.1234 and o.text4(1234567.0) == 1235000.0 and o.text4(1e5) == 1e5
    sc = o.scale(f[None, :])
    assert sc.shape == (1, 324) and sc[0, 323] == 0.0  # dropped by svm-scale (single-valued attribute)


def test_synth_cloud_is_deterministic():
    from haf_grasping_b200 import synth
    a, b = synth.synth_cloud(1234, 5000), synth.synth_cloud(1234, 5000)
    assert a.tobytes() == b.tobytes()
    assert a.dtype == np.float32 and a.shape == (5000, 3)
    assert np.abs(a[:, :2]).max() < 0.28
    import zlib
    assert zlib.crc32(synth.synth_cloud(1234, 1000).tobytes()) == zlib.crc32(a[:1000].tobytes())  # counter-based


def _fnv1a(b):
    h = 1469598103934665603
    for x in b:
        h = ((h ^ x) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def _lzf_literal_stream(data: bytes) -> bytes:
    """a valid LZF stream made of literal runs only (enough to exercise the container + SoA layout)"""
    out = bytearray()
    for i in range(0, len(data), 32):
        chunk = data[i:i + 32]
        out.append(len(chunk) - 1)
        out += chunk
    return bytes(out)


def test_cpp_pcd_reader_all_formats(tmp_path):
    """haf_cli --dump-pcd (C++ reader of csrc/host/pcd_io.hpp) == the Python reader, on ASCII / binary / binary_compressed."""
    import struct
    from haf_grasping_b200 import build
    from haf_grasping_b200.pcd import read_pcd
    cli = build.build_cli()
    rng = np.random.default_rng(2)
    pts = rng.normal(size=(53, 3)).astype(np.float32)
    hdr = "# .PCD v0.7\nVERSION 0.7\nFIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH 53\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 53\n"
    files = {}
    files["a.pcd"] = (hdr + "DATA ascii\n" + "\n".join(" ".join("%.9g" % v for v in row) for row in pts) + "\n0 0 0\n").encode()
    files["b.pcd"] = (hdr + "DATA binary\n").encode() + pts.tobytes()
    soa = np.ascontiguousarray(pts.T).tobytes()
    comp = _lzf_literal_stream(soa)
    files["c.pcd"] = (hdr + "DATA binary_compressed\n").encode() + struct.pack("<II", len(comp), len(soa)) + comp
    for name, blob in files.items():
        f = tmp_path / name
        f.write_bytes(blob)
        py = read_pcd(str(f))
        assert py.tobytes() == pts.tobytes(), name
        out = subprocess.run([cli, "--pcd", str(f), "--dump-pcd"], capture_output=True, text=True, check=True).stdout.split()
        assert int(out[0]) == 53 and int(out[1]) == _fnv1a(pts.tobytes()), name
    for name in ("pcd5", "table2"):
        path = _reference_pcd_file(tmp_path, name)
        out = subprocess.run([cli, "--pcd", path, "--dump-pcd"], capture_output=True, text=True, check=True).stdout.split()
        py = read_pcd(path)
        assert int(out[0]) == len(py) and int(out[1]) == _fnv1a(py.tobytes())


def test_bench_stage_roofline_and_clock_sampler_parsing(tmp_path):
    """bench.py helpers that run on the GPU box only: the algorithmic-byte rows of SURVEY 8d and the nvidia-smi row filter."""
    import importlib.util
    import time
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    acc = dict(bin=2.0, integral=0.2, mask=0.2, features=9.8, score=0.5)
    sr = b.stage_roofline(acc, 2, n_points=1000, n_units=12, G=56, D=323, W=100.0, hbm_gbs=6447.5)
    assert sr["bin"]["algorithmic_bytes"] == 12.0 * 1000 + 4.0 * 12 * 56 * 56
    assert sr["integral"]["algorithmic_bytes"] == 4.0 * 12 * 56 * 56 + 4.0 * 12 * 57 * 57
    assert sr["mask+features"]["algorithmic_bytes"] == 4.0 * 12 * 57 * 57 + 12 * 56 * 56 + 4.0 * 323 * 100.0
    assert sr["mask+features"]["ms"] == 5.0 and abs(sr["bin"]["GBps"] - sr["bin"]["algorithmic_bytes"] / 1e-3 / 1e9) < 1e-9
    assert abs(sr["bin"]["frac_of_hbm_peak"] - sr["bin"]["GBps"] / 6447.5) < 1e-12
    # clock sampler: only rows stamped inside the timed region count; a throttle reason is reported
    s = b.ClockSampler(0)
    s.path = str(tmp_path / "clocks.csv")
    now = time.time()

    def stamp(t):
        return time.strftime("%Y/%m/%d %H:%M:%S", time.localtime(t)) + ".%03d" % int((t % 1) * 1000)
    with open(s.path, "w") as fh:
        fh.write("%s, 1200, 1965, 700.0, Active, Not Active, Not Active, Not Active, Not Active\n" % stamp(now - 30))
        fh.write("%s, 1900, 1965, 900.0, Active, Not Active, Not Active, Not Active, Active\n" % stamp(now - 0.5))
        fh.write("%s, 1800, 1965, 900.0, Active, Not Active, Not Active, Not Active, Active\n" % stamp(now - 0.2))

    class Done:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
    s.proc, s.fh = Done(), open(os.devnull, "w")
    s.t_begin = now - 1.0
    out = s.stop()
    assert out["samples"] == 2 and out["sm_mhz"] == 1850.0 and out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"


def test_bench_dump_outputs_writes_every_answer_field_of_the_batch_records(tmp_path):
    """bench.py --dump-outputs: one float64 .npy per answer field of the haf_best records, values exact."""
    import importlib.util
    from haf_grasping_b200 import api
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    best = (api.haf_best * 3)()
    best[1].row, best[2].topval, best[0].roll_rad, best[2].M[3] = 7, -1000, np.float32(0.1), 0.5
    b.dump_outputs(str(tmp_path / "out"), b.best_arrays(best))
    assert sorted(os.listdir(tmp_path / "out")) == sorted("best_%s.npy" % f for f in b.BEST_FIELDS)
    load = lambda f: np.load(tmp_path / "out" / ("best_%s.npy" % f))  # noqa: E731
    assert all(load(f).dtype == np.float64 for f in b.BEST_FIELDS)
    assert load("row").tolist() == [0, 7, 0] and load("topval").tolist() == [0, 0, -1000]
    assert load("roll_rad")[0] == np.float32(0.1) and load("M").shape == (3, 16) and load("M")[2, 3] == 0.5
