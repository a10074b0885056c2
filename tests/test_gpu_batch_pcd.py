"""Batches of PCD files and PointCloud2 buffers decoded on the device in one pass (haf_pcd_decode_batch, haf_search_batch_pcd,
haf_pointcloud2_batch_to_xyz).

Every cloud of a batch must be byte-equal to what the single-file decode and the host readers (haf_grasping_b200/pcd.py,
csrc/host/pcd_io.hpp) give for that file alone; the number of kernel launches must not grow with the number of files; a
search on the decoded batch must equal haf_search_batch_requests on the host-decoded clouds field for field.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE
from test_pcd_device import make_pcd

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pcd_files():
    return np.load(os.path.join(GOLDEN, "pcd_files.npz"))


@pytest.fixture(scope="module")
def clouds():
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="module")
def gpu(hg, tmp_models):
    g = hg.GraspSearch(FEATURES, RANGE, tmp_models(256))
    yield g
    g.close()


def _generated_xyz(n=70000):
    rng = np.random.default_rng(5)
    xyz = (rng.normal(size=(n, 3)) * np.array([0.3, 0.3, 0.05])).astype(np.float32)
    xyz[:, 2] = np.round(xyz[:, 2], 2)
    xyz[1000:9000, 0] = -0.125
    xyz[5] = [np.nan, 1e-42, -3.4e38]        # nan token, subnormal, near FLT_MAX
    rgb = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    lab = rng.integers(0, 250, n).astype(np.uint8)
    nrm = rng.normal(size=(n, 3)).astype(np.float32)
    return xyz, rgb, lab, nrm


def _generated_cases(xyz, rgb, lab, nrm):
    """the generated files of test_pcd_device.test_generated_pcd_files_decode_byte_equal"""
    return [
        ("ascii", dict()),
        ("ascii", dict(sep="\t", eol="\r\n", fmt="%.7e")),
        ("ascii", dict(sep="  ", surplus=37, fmt="%.8f")),
        ("ascii", dict(fields=("normal", "y", "rgb", "x", "z"), extra={"normal": ("F", 4, 3, nrm), "rgb": ("U", 4, 1, rgb)})),
        ("binary", dict()),
        ("binary", dict(fields=("label", "x", "rgb", "z", "y"), extra={"label": ("U", 1, 1, lab), "rgb": ("U", 4, 1, rgb)})),
        ("binary", dict(fields=("normal", "z", "x", "y"), extra={"normal": ("F", 4, 3, nrm)})),
        ("binary_compressed", dict()),
        ("binary_compressed", dict(fields=("x", "label", "y", "normal", "z"), extra={"label": ("U", 1, 1, lab), "normal": ("F", 4, 3, nrm)})),
    ]


def _check_batch(gpu, files, want):
    got = gpu.pcd_decode_batch_to_host(files)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and g.tobytes() == w.tobytes(), i
    return got


def test_all_bundled_files_in_one_batch(gpu, pcd_files, clouds):
    names = sorted(pcd_files.keys())
    asc = [n for n in names if b"DATA ascii" in pcd_files[n].tobytes()[:2000]]
    comp = [n for n in names if n not in asc]
    assert len(asc) == 13 and len(comp) == 3
    order = []          # kinds interleaved
    for k in range(len(asc)):
        order.append(asc[k])
        if k < len(comp):
            order.append(comp[k])
    for seq in (order, order[::-1]):
        files = [pcd_files[n].tobytes() for n in seq]
        d, po = gpu.pcd_decode_batch(files)
        assert list(po) == list(np.cumsum([0] + [len(clouds[n]) for n in seq]))
        got = _check_batch(gpu, files, [clouds[n] for n in seq])
        for n, g in zip(seq[:4], got[:4]):
            assert gpu.pcd_decode_to_host(pcd_files[n].tobytes()).tobytes() == g.tobytes(), n


def test_generated_mixed_batch(gpu):
    from haf_grasping_b200 import pcd
    xyz, rgb, lab, nrm = _generated_xyz()
    files = [make_pcd("ascii", xyz[:0]), make_pcd("binary", xyz[:0])]                          # POINTS 0 at the start
    for kind, kw in _generated_cases(xyz, rgb, lab, nrm):
        files.append(make_pcd(kind, xyz, **kw))
    files.append(make_pcd("binary_compressed", xyz[:0]))                                        # POINTS 0 in the middle
    for kind in ("ascii", "binary", "binary_compressed"):                                       # 1-point files
        files.append(make_pcd(kind, xyz[7:8]))
    # no final newline, followed directly by another file
    files.append(make_pcd("ascii", xyz[:100])[:-1])
    files.append(make_pcd("ascii", xyz[200:300]))
    files.append(make_pcd("ascii", xyz[300:350]) + b"   \t \n")                                # ends in a line of blanks
    files.append(make_pcd("ascii", xyz[300:351])[:-1] + b"\n \t")                               # ... with no newline
    files.append(make_pcd("binary", xyz[:333]) + b"x")                                         # bytes after the records
    for pad in (b"", b"#"):                      # data sections at an even and an odd offset of the batch (17-byte records)
        files.append(pad + make_pcd("binary", xyz[1:3000], fields=("label", "x", "rgb", "z", "y"),
                                    extra={"label": ("U", 1, 1, lab[1:3000]), "rgb": ("U", 4, 1, rgb[1:3000])}))
        files.append(pad + make_pcd("binary_compressed", xyz[1:2000]))
    files.append(make_pcd("ascii", xyz[:0]))                                                    # POINTS 0 at the end
    offs = np.cumsum([0] + [len(f) for f in files])
    data_at = [int(o) + f.index(b"\n", f.index(b"\nDATA ") + 1) + 1 for o, f in zip(offs, files)]
    assert any(d % 2 for d, f in zip(data_at, files) if b"DATA binary\n" in f) and any(d % 2 == 0 for d in data_at)
    want = [pcd.read_pcd_bytes(f) if f.count(b"POINTS 0\n") == 0 else np.zeros((0, 3), np.float32) for f in files]
    _check_batch(gpu, files, want)

    # one ASCII file of more than 4 MB (more than one 1024-tile scan round) beside 300 tiny files
    rng = np.random.default_rng(11)
    big = make_pcd("ascii", rng.normal(size=(150000, 3)).astype(np.float32))
    assert len(big) > 4 << 20
    tiny = [make_pcd(("ascii", "binary", "binary_compressed")[i % 3], rng.normal(size=(1 + i % 7, 3)).astype(np.float32)) for i in range(300)]
    files = tiny[:150] + [big] + tiny[150:]
    _check_batch(gpu, files, [pcd.read_pcd_bytes(f) for f in files])


def test_launches_do_not_grow_with_the_number_of_files(gpu):
    rng = np.random.default_rng(2)

    def batch(n):
        return [make_pcd(("ascii", "binary", "binary_compressed")[i % 3], rng.normal(size=(50 + i, 3)).astype(np.float32)) for i in range(n)]

    deltas = []
    for n in (3, 300):
        files = batch(n)
        gpu.pcd_decode_batch(files)
        l0 = gpu.launch_count()
        gpu.pcd_decode_batch(files)
        deltas.append(gpu.launch_count() - l0)
    assert deltas[0] == deltas[1] == 5, deltas        # ASCII count / scan / parse, LZF, gather


def _assert_same(a, b, keys):
    for k in keys:
        x, y = a[k], b[k]
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y), k
        else:
            assert len(x) == len(y), k
            for i in range(len(x)):
                assert bytes(x[i]) == bytes(y[i]), (k, i)


def test_search_parity_with_host_decoded_clouds(gpu, hg, pcd_files, clouds):
    names = sorted(pcd_files.keys())
    seq = [names[i % len(names)] for i in range(24)]
    files = [pcd_files[n].tobytes() for n in seq]
    xyz = np.concatenate([clouds[n] for n in seq])
    po = np.cumsum([0] + [len(clouds[n]) for n in seq])
    rng = np.random.default_rng(4)
    reqs, ro = [], [0]
    for c in range(24):
        k = 2 if c % 3 == 0 else 1
        for j in range(k):
            reqs.append(hg.make_request(center=tuple(rng.uniform(-0.03, 0.03, 3)),
                                        approach=(0.0, 0.0, 1.0) if j == 0 else (0.5, 0.0, 0.8660254)))
        ro.append(len(reqs))
    kw = dict(grasps=True, per_roll=True, per_roll_top=True)
    a = gpu.search_batch_pcd(files, reqs, ro, **kw)
    b = gpu.search_batch_requests(xyz, po, reqs, ro, **kw)
    assert list(a["point_offsets"]) == list(po)
    _assert_same(a, b, ("best", "best_per_request", "grasp", "grasp_per_request", "grasp_per_roll", "per_roll_top"))
    # a one-file batch == search_pcd / search_grasps (n_guard aside, as in every batch call)
    for n in ("table1", "pcd2"):
        one = gpu.search_batch_pcd([pcd_files[n].tobytes()], per_roll_top=True)
        single = gpu.search_pcd(pcd_files[n].tobytes())
        g = gpu.search_grasps(clouds[n])
        sb = single["best"]
        sb.n_guard = 0
        assert bytes(one["best"][0]) == bytes(sb), n
        assert np.array_equal(one["per_roll_top"][0], single["per_roll_top"][0]), n
        assert bytes(one["grasp"][0]) == bytes(g["grasp"]), n


def test_pageable_and_pinned_sources_agree(gpu, pcd_files):
    import torch
    names = sorted(pcd_files.keys())
    files = [pcd_files[names[i % len(names)]].tobytes() for i in range(40)]
    blob = np.frombuffer(b"".join(files), np.uint8)
    assert len(blob) > 4 << 20
    offs = np.cumsum([0] + [len(f) for f in files])
    pinned = torch.empty(len(blob), dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = blob
    a = gpu.search_batch_pcd((blob.copy(), offs), per_roll_top=True)
    xa = gpu.pcd_decode_batch_to_host((blob.copy(), offs))
    b = gpu.search_batch_pcd((pinned, offs), per_roll_top=True)
    xb = gpu.pcd_decode_batch_to_host((pinned, offs))
    _assert_same(a, b, ("best", "best_per_request", "grasp", "grasp_per_request", "per_roll_top", "point_offsets"))
    assert all(x.tobytes() == y.tobytes() for x, y in zip(xa, xb))


def _bad_cases():
    from test_pcd_device import make_pcd as mk
    xyz = np.random.default_rng(1).normal(size=(50, 3)).astype(np.float32)
    bad = [(mk("ascii", xyz, points=60), -2, "fewer records"),
           (mk("binary", xyz)[:-7], -2, "truncated"),
           (mk("binary_compressed", xyz)[:-3], -2, "truncated"),
           (mk("ascii", xyz).replace(b"FIELDS x y z", b"FIELDS x y w"), -2, "x/y/z"),
           (mk("ascii", xyz).replace(b"TYPE F F F", b"TYPE F F I"), -5, "float32"),
           (mk("ascii", xyz).replace(b"DATA ascii", b"DATA zipped"), -5, "DATA kind")]
    raw = mk("binary_compressed", xyz)
    k = raw.index(b"DATA binary_compressed\n") + len(b"DATA binary_compressed\n") + 8
    bad.append((raw[:k] + bytes([0xE0 | 0x1F, 0xFF, 0xFF]) + raw[k + 3:], -2, "corrupt LZF"))
    lines = mk("ascii", xyz).split(b"\n")
    lines[20] = lines[20].split(b" ")[0]
    bad.append((b"\n".join(lines), -2, "short ASCII record"))
    return bad


def test_errors_name_the_file(gpu, hg, pcd_files, clouds):
    names = sorted(pcd_files.keys())
    good = [pcd_files[names[i]].tobytes() for i in range(5)]
    want = [clouds[names[i]] for i in range(5)]
    for j, (raw, code, text) in enumerate(_bad_cases()):
        k = j % 5
        files = good[:k] + [raw] + good[k:]
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode_batch(files)
        with pytest.raises(hg.HafError) as single:
            gpu.pcd_decode(raw)
        msg = str(e.value)
        assert e.value.code == code and ("PCD file %d: " % k) in msg and text in msg, (k, code, text, msg)
        single_text = str(single.value).split(": ", 1)[1]        # "libhafgpu error <code>: <text>"
        assert msg.endswith("PCD file %d: %s" % (k, single_text)), (msg, single_text)
    bad = _bad_cases()
    for lo, hi in ((bad[0], bad[7]), (bad[6], bad[1]), (bad[3], bad[5])):   # device / device, device / host, host / host
        files = good[:1] + [lo[0]] + good[1:3] + [hi[0]] + good[3:]
        with pytest.raises(hg.HafError) as e:
            gpu.pcd_decode_batch(files)
        if lo[2] in ("corrupt LZF", "fewer records") and hi[2] == "truncated":
            assert "PCD file 4: " in str(e.value)          # size checks run on the host, before any device work
        else:
            assert "PCD file 1: " in str(e.value) and lo[2] in str(e.value), str(e.value)
    _check_batch(gpu, good, want)                          # the context decodes the next good batch


def test_pointcloud2_batch(gpu, hg, clouds):
    import torch
    rng = np.random.default_rng(8)
    layouts = [(16, 0, 4, 8), (32, 4, 12, 20), (13, 1, 5, 9), (16, 0, 4, 8), (32, 4, 12, 20)]
    sizes = [len(clouds["table1"]), 5000, 0, 1, 777]
    bufs, want = [], []
    for (step, ox, oy, oz), n in zip(layouts, sizes):
        xyz = clouds["table1"][:n] if n > 5000 else rng.normal(size=(n, 3)).astype(np.float32)
        b = rng.integers(0, 256, (n, step), dtype=np.uint8)
        for k, o in enumerate((ox, oy, oz)):
            b[:, o:o + 4] = xyz[:, k].copy().view(np.uint8).reshape(n, 4)
        bufs.append(b.reshape(-1))
        # numpy gather of the records
        want.append(np.stack([b[:, o:o + 4].copy().view(np.float32).reshape(n) for o in (ox, oy, oz)], 1) if n else np.zeros((0, 3), np.float32))
    data = np.concatenate(bufs)
    offs = np.cumsum([0] + [len(b) for b in bufs])
    po_want = np.cumsum([0] + sizes)
    for src in (data, torch.from_numpy(data).cuda()):
        d, po = gpu.pointcloud2_batch_to_xyz(src, offs, layouts)
        assert list(po) == list(po_want)
        got = gpu.debug_pcd_xyz(int(po[-1]))
        for c in range(len(sizes)):
            assert got[po[c]:po[c + 1]].tobytes() == want[c].tobytes(), c
    bad_layout = list(layouts)
    bad_layout[3] = (16, 0, 4, 13)
    with pytest.raises(hg.HafError) as e:
        gpu.pointcloud2_batch_to_xyz(data, offs, bad_layout)
    assert e.value.code == -1 and "cloud 3" in str(e.value)
    bad_offs = offs.copy()
    bad_offs[2] += 1                       # cloud 1 gets a byte too many, cloud 2 ... a negative span is not allowed either
    bad_offs[3] += 1
    with pytest.raises(hg.HafError) as e:
        gpu.pointcloud2_batch_to_xyz(data, bad_offs, layouts)
    assert e.value.code == -1 and "cloud 1" in str(e.value)


def test_group_context_equals_one_gpu(hg, tmp_models, pcd_files):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    names = sorted(pcd_files.keys())
    files = [pcd_files[names[i % len(names)]].tobytes() for i in range(12)]
    one = hg.GraspSearch(FEATURES, RANGE, tmp_models(256))
    two = hg.GraspSearch(FEATURES, RANGE, tmp_models(256), devices=[0, 1])
    try:
        a = one.search_batch_pcd(files, per_roll=True, per_roll_top=True)
        b = two.search_batch_pcd(files, per_roll=True, per_roll_top=True)
        _assert_same(a, b, ("best", "best_per_request", "grasp", "grasp_per_request", "grasp_per_roll", "per_roll_top", "point_offsets"))
    finally:
        one.close()
        two.close()


def test_cli_batch_prints_what_single_runs_print(pcd_files, trained_model_path, tmp_path):
    from haf_grasping_b200 import build
    cli = build.build_cli()
    paths = []
    for name in ("pcd2", "table1", "pcd4"):
        f = tmp_path / (name + ".pcd")
        f.write_bytes(pcd_files[name].tobytes())
        paths.append(str(f))
    base = [cli, "--features", FEATURES, "--range", RANGE, "--model", trained_model_path]
    for extra in ([], ["--json"], ["--host-pcd"], ["--json", "--host-pcd"]):
        singles = "".join(subprocess.run(base + ["--pcd", p] + extra, capture_output=True, text=True, check=True).stdout for p in paths)
        args = list(base)
        for p in paths:
            args += ["--pcd", p]
        batch = subprocess.run(args + extra, capture_output=True, text=True, check=True).stdout
        assert batch == singles, extra
        assert len(batch.splitlines()) == 3
