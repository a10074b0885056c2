"""Ranked grasp candidates on the device (haf_search_batch_candidates): the k best distinct grasps of every cloud against a
numpy restatement of the semantics in include/hafgpu.h, built from the CPU oracle's grids (Oracle.search(..., full=True)) or,
where the oracle has no counterpart (roll_begin, probability heights, G = 512), from the library's own per-roll grids.  Poses
come from the oracle's transform_gp_in_wcs; records are compared byte for byte."""
import ctypes as C
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE

pytestmark = pytest.mark.gpu

TILTED = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254)]
VARIANTS = [dict(approach=(0.5, 0.0, 0.8660254), center=(0.05, 0.2, 0.0)), dict(width=2, area=(30.0, 40.0)), dict(return_only_best=1)]
# kernels haf_search_batch_candidates launches on top of haf_search_batch_requests with grasps for a call in one chunk at G <= 90:
# rank_unit_kernel (once per chunk) + rank_cloud_kernel (once per call)
RANK_KERNELS_ONE_CHUNK = 2


@pytest.fixture(scope="module")
def clouds():
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="module")
def trained_model(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("trained_c") / "substitute_trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(p, "wb") as dst:
        dst.write(src.read())
    return p


@pytest.fixture(scope="module")
def prob_model(tmp_path_factory):
    """the substitute model + the probA / probB lines svm-train -b 1 produced for it (as tests/test_probability.py builds it)"""
    with open(os.path.join(GOLDEN, "substitute_trained.prob.json")) as fh:
        pj = json.load(fh)
    text = gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb").read().decode()
    head, tail = text.split("nr_sv", 1)
    p = str(tmp_path_factory.mktemp("prob_model_c") / "substitute_trained.prob.model")
    with open(p, "w") as fh:
        fh.write(head + "probA %s\nprobB %s\nnr_sv" % (pj["probA"], pj["probB"]) + tail)
    return p


@pytest.fixture(scope="module")
def gpu(hg, trained_model):
    g = hg.GraspSearch(FEATURES, RANGE, trained_model)
    yield g
    g.close()


@pytest.fixture(scope="module")
def orc(oracle_lib, trained_model):
    return oracle_lib.Oracle(FEATURES, RANGE, trained_model)


# ---- the reference restatement ------------------------------------------------------------------------------------------
class Grids:
    """per request: graspseval / mask / heights [R][G][G] and the evaluated rolls [rb, rb + rd)"""

    def __init__(self, ev, mask, heights, rb, rd):
        self.ev, self.mask, self.heights, self.rb, self.rd = ev, mask, heights, rb, rd


def _unit_lists(grids, P):
    """every unit's first P eligible cells, merged: (-score, q, r, cell) ascending = the order of the semantics"""
    ents = []
    for q, g in enumerate(grids):
        for r in range(g.rb, g.rb + g.rd):
            cells = np.flatnonzero(g.mask[r].ravel() == 1)
            sc = g.ev[r].ravel()[cells].astype(np.float64)
            for i in np.lexsort((cells, -sc))[:P]:
                ents.append((-float(sc[i]), q, r, int(cells[i])))
    ents.sort()
    return ents


def _record(hg, pose, ev, row, col, roll, score, q):
    c = hg.haf_candidate()
    g = c.grasp
    g.eval, g.roll = int(ev), float(pose[12])
    g.graspPoint1[:], g.graspPoint2[:] = pose[0:3], pose[3:6]
    g.averagedGraspPoint[:], g.approachVector[:] = pose[6:9], pose[9:12]
    g.row, g.col, g.roll_index = int(row), int(col), int(roll)
    c.score, c.request = float(score), int(q)
    return c


def _d2(a, b):
    dx, dy, dz = a[0] - b[0], a[1] - b[1], a[2] - b[2]
    return (dx * dx + dy * dy) + dz * dz


def expected(hg, o, orqs, grids, win, k, P, md):
    """win: (request, roll, row, col, topval) of the cloud's best grasp, or None when no roll was evaluated"""
    if win is None:
        return []
    q0, r0, row0, col0, top0 = win
    G = grids[0].ev.shape[-1]
    pose = o.transform_gp_in_wcs(orqs[q0], grids[q0].heights[r0], row0, col0, r0)
    out = [_record(hg, pose, top0 - 20, row0, col0, r0, grids[q0].ev[r0][row0, col0], q0)]
    avgs = [pose[6:9]]
    for negs, q, r, cell in _unit_lists(grids, P):
        if len(out) == k:
            break
        row, col = divmod(cell, G)
        if (q, r, row, col) == (q0, r0, row0, col0):
            continue
        pose = o.transform_gp_in_wcs(orqs[q], grids[q].heights[r], row, col, r)
        if md > 0 and any(_d2(pose[6:9], a) < md * md for a in avgs):
            continue
        score = np.float32(-negs)
        out.append(_record(hg, pose, int(score) - 20, row, col, r, score, q))
        avgs.append(pose[6:9])
    return out


def oracle_case(o, oracle_lib, xyz, kws):
    """grids and winner from the oracle, one search per request; winner: strict >, earliest request"""
    orqs, grids, win = [], [], None
    for kw in kws:
        orq = oracle_lib.make_request(**kw)
        r = o.search(xyz, orq, full=True)
        orqs.append(orq)
        grids.append(Grids(r["graspseval"], r["mask"], r["heights"], 0, r["best"].rolls_done))
        b = r["best"]
        if b.roll >= 0 and (win is None or b.topval > win[4]):
            win = (len(orqs) - 1, b.roll, b.row, b.col, b.topval)
    return orqs, grids, win


def gpu_grid_case(gpu, hg, oracle_lib, xyz, kws):
    """grids and winner from the library's own search(..., outputs=True) (roll_begin, probability mode, large grids)"""
    R = gpu.R
    res = gpu.search(xyz, [hg.make_request(**kw) for kw in kws], outputs=True)
    orqs, grids = [], []
    for q, kw in enumerate(kws):
        okw = {a: v for a, v in kw.items() if a in ("center", "area", "approach", "width")}
        orqs.append(oracle_lib.make_request(**okw))
        rl = kw.get("roll_limit", 0)
        end = min(R, rl) if rl > 0 else R
        rb = max(0, min(kw.get("roll_begin", 0), end))
        grids.append(Grids(res["graspseval"][q], res["mask"][q], res["heights"][q], rb, res["best_per_request"][q].rolls_done))
    b = res["best"]
    win = None if b.roll < 0 else (b.approach_idx, b.roll, b.row, b.col, b.topval)
    return orqs, grids, win


def check(res, exp, c=0, k=None):
    k = k if k is not None else len(res["candidates"]) // len(res["n_candidates"])
    n = int(res["n_candidates"][c])
    assert n == len(exp), (n, len(exp))
    for i in range(n):
        assert bytes(res["candidates"][c * k + i]) == bytes(exp[i]), (c, i, res["candidates"][c * k + i].grasp.row, exp[i].grasp.row)
    empty = bytes(C.sizeof(exp[0]) if exp else 128)
    for i in range(n, k):
        assert bytes(res["candidates"][c * k + i]) == empty


def same(a, b):
    assert list(a["n_candidates"]) == list(b["n_candidates"])
    for key in ("best", "grasp", "candidates"):
        assert bytes(a[key]) == bytes(b[key]), key


# ---- tests --------------------------------------------------------------------------------------------------------------
def test_bundled_clouds_default_request(gpu, orc, oracle_lib, hg, clouds):
    for name in sorted(clouds.files):
        xyz = clouds[name]
        orqs, grids, win = oracle_case(orc, oracle_lib, xyz, [{}])
        ref = gpu.search_batch_requests(xyz, [0, len(xyz)], [hg.make_request()])
        for k in (1, 16, 64):
            for P in (k, 1024):
                for md in (0.0, 0.02, 0.05):
                    res = gpu.search_candidates(xyz, k=k, per_unit=P, min_distance=md)
                    check(res, expected(hg, orc, orqs, grids, win, k, P, md))
                    # rank 0 is the cloud's best grasp, exactly grasp_per_cloud
                    assert bytes(res["candidates"][0].grasp) == bytes(res["grasp"][0]), name
                    assert bytes(res["grasp"]) == bytes(ref["grasp"]) and bytes(res["best"]) == bytes(ref["best"])
                    if md <= 0:   # no suppression, per_unit >= k: the global top k of the eligible cells after rank 0
                        _check_global_topk(res, grids, win, k)


def _check_global_topk(res, grids, win, k):
    G = grids[0].ev.shape[-1]
    allc = []
    for q, g in enumerate(grids):
        for r in range(g.rb, g.rb + g.rd):
            cells = np.flatnonzero(g.mask[r].ravel() == 1)
            allc += [(-float(g.ev[r].ravel()[c]), q, r, int(c)) for c in cells]
    allc.sort()
    q0, r0, row0, col0, _ = win
    top = [e for e in allc if (e[1], e[2], e[3]) != (q0, r0, row0 * G + col0)][:k - 1]
    got = [(-float(c.score), c.request, c.grasp.roll_index, c.grasp.row * G + c.grasp.col) for c in res["candidates"][1:int(res["n_candidates"][0])]]
    assert got == top


@pytest.mark.parametrize("kw", VARIANTS, ids=["tilted", "width2_area30x40", "only_best"])
def test_request_variants(gpu, orc, oracle_lib, hg, clouds, kw):
    for name in ("pcd2", "plastic_mug2", "table1"):
        xyz = clouds[name]
        orqs, grids, win = oracle_case(orc, oracle_lib, xyz, [kw])
        for k, P, md in ((16, 0, 0.03), (64, 64, 0.0), (8, 1024, 0.05)):
            res = gpu.search_candidates(xyz, [hg.make_request(**kw)], k=k, per_unit=P, min_distance=md)
            check(res, expected(hg, orc, orqs, grids, win, k, P if P else max(k, 64), md))
            if kw.get("return_only_best"):   # candidates only from the rolls the early exit left
                rd = grids[0].rd
                assert all(c.grasp.roll_index < rd for c in res["candidates"][:int(res["n_candidates"][0])])


def test_roll_range(gpu, oracle_lib, hg, clouds):
    xyz = clouds["table1"]
    cases = [[dict(roll_begin=3, roll_limit=9)], [dict(roll_begin=2, return_only_best=1, graspval_top=60)],
             [dict(roll_limit=4), dict(roll_begin=7, approach=TILTED[1])]]
    for kws in cases:
        orqs, grids, win = gpu_grid_case(gpu, hg, oracle_lib, xyz, kws)
        for k, md in ((16, 0.03), (32, 0.0)):
            res = gpu.search_candidates(xyz, [hg.make_request(**kw) for kw in kws], k=k, min_distance=md)
            check(res, expected(hg, gpu_oracle(oracle_lib), orqs, grids, win, k, max(k, 64), md))


_ORC_POSE = {}


def gpu_oracle(oracle_lib):
    """an oracle for poses only (transform_gp_in_wcs needs no model)"""
    if "o" not in _ORC_POSE:
        _ORC_POSE["o"] = oracle_lib.Oracle(FEATURES, RANGE)
    return _ORC_POSE["o"]


def test_five_approach_vectors(gpu, orc, oracle_lib, hg, clouds):
    xyz = clouds["table1"]
    kws = [dict(approach=a) for a in TILTED]
    orqs, grids, win = oracle_case(orc, oracle_lib, xyz, kws)
    for k, P, md in ((64, 0, 0.02), (64, 64, 0.0), (256, 1024, 0.01)):
        res = gpu.search_candidates(xyz, [hg.make_request(**kw) for kw in kws], k=k, per_unit=P, min_distance=md)
        exp = expected(hg, orc, orqs, grids, win, k, P if P else max(k, 64), md)
        check(res, exp)
        assert len({c.request for c in exp}) > 1   # the list crosses requests
        assert res["candidates"][0].request == res["best"][0].approach_idx


def _mixed_batch(clouds, hg):
    from haf_grasping_b200 import synth
    names = sorted(clouds.files)
    xs, kws_all = [], []
    rng = np.random.default_rng(5)
    for i in range(40):
        xs.append(clouds[names[i % len(names)]] if i % 3 else synth.synth_cloud(100 + i, 30000))
        n = 1 + i % 4
        kws_all.append([dict(approach=TILTED[int(a)], center=tuple(rng.uniform(-0.02, 0.02, 3))) for a in rng.integers(0, 5, n)])
    off = np.concatenate([[0], np.cumsum([len(x) for x in xs])])
    ro = np.concatenate([[0], np.cumsum([len(k) for k in kws_all])])
    reqs = [hg.make_request(**kw) for kws in kws_all for kw in kws]
    return np.concatenate(xs).astype(np.float32), off, ro, reqs, xs, kws_all


def test_batch_mixed_clouds_all_inputs(gpu, hg, clouds):
    import torch
    xyz, off, ro, reqs, xs, kws_all = _mixed_batch(clouds, hg)
    k, md = 16, 0.03
    singles = [gpu.search_candidates(x, [hg.make_request(**kw) for kw in kws], k=k, min_distance=md) for x, kws in zip(xs, kws_all)]
    for src in (torch.from_numpy(xyz).cuda(), torch.from_numpy(xyz).pin_memory(), xyz):
        res = gpu.search_batch_candidates(src, off, reqs, ro, k=k, min_distance=md)
        if not hasattr(src, "is_cuda") or not src.is_cuda:
            assert gpu.timing().n_chunks > 1
        for c, s in enumerate(singles):
            assert int(res["n_candidates"][c]) == int(s["n_candidates"][0])
            assert bytes(res["best"][c]) == bytes(s["best"][0]) and bytes(res["grasp"][c]) == bytes(s["grasp"][0])
            assert bytes(res["candidates"])[c * k * 128:(c + 1) * k * 128] == bytes(s["candidates"])


def test_probability_mode(hg, oracle_lib, prob_model, clouds):
    g = hg.GraspSearch(FEATURES, RANGE, prob_model)
    try:
        o = gpu_oracle(oracle_lib)
        for name in ("pcd2", "table1"):
            xyz = clouds[name]
            kws = [dict(svm_with_probability=1)]
            orqs, grids, win = gpu_grid_case(g, hg, oracle_lib, xyz, kws)
            for k, md in ((16, 0.0), (16, 0.03)):
                res = g.search_candidates(xyz, [hg.make_request(**kws[0])], k=k, min_distance=md)
                check(res, expected(hg, o, orqs, grids, win, k, 64, md))
    finally:
        g.close()


def test_svm_modes_agree(hg, trained_model, clouds):
    xyz = clouds["table1"]
    outs = []
    for mode in (0, 1, 2):
        g = hg.GraspSearch(FEATURES, RANGE, trained_model, svm_mode=mode)
        try:
            outs.append(g.search_candidates(xyz, [hg.make_request(approach=a) for a in TILTED[:2]], k=32, min_distance=0.02))
        finally:
            g.close()
    same(outs[0], outs[1])
    same(outs[0], outs[2])


def test_graph_replay(hg, trained_model, gpu, clouds):
    import torch
    names = ("pcd2", "table1", "plastic_mug2")
    xs = [clouds[n] for n in names]
    off = np.concatenate([[0], np.cumsum([len(x) for x in xs])])
    d = torch.from_numpy(np.concatenate(xs)).cuda()
    reqs = [hg.make_request(approach=TILTED[i]) for i in range(3)]
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, use_graph=True)
    try:
        for k, md in ((16, 0.03), (16, 0.03), (16, 0.03), (4, 0.0), (4, 0.0), (4, 0.0), (16, 0.05), (16, 0.05)):
            want = gpu.search_batch_candidates(d, off, reqs, k=k, min_distance=md)
            got = g.search_batch_candidates(d, off, reqs, k=k, min_distance=md)
            same(got, want)
        assert g.timing().graph_replays >= 2
    finally:
        g.close()


def test_grid512_multi_cta_selection(hg, oracle_lib, tmp_models):
    from haf_grasping_b200 import synth
    model = tmp_models(64, seed=11)
    xyz = synth.synth_cloud(1234, 1000000, r=2.56)
    g = hg.GraspSearch(FEATURES, RANGE, model, grid=512)
    try:
        kws = [dict(area=(362.0, 362.0), roll_limit=1)]
        orqs, grids, win = gpu_grid_case(g, hg, oracle_lib, xyz, kws)
        o = gpu_oracle(oracle_lib)
        for k, P, md in ((16, 64, 0.03), (64, 1024, 0.0), (32, 1024, 0.01)):
            res = g.search_candidates(xyz, [hg.make_request(**kws[0])], k=k, per_unit=P, min_distance=md)
            check(res, expected(hg, o, orqs, grids, win, k, P, md))
        assert int(res["n_candidates"][0]) == 32
    finally:
        g.close()


def test_edge_cases(gpu, oracle_lib, hg, clouds):
    o = gpu_oracle(oracle_lib)
    empty = np.zeros((0, 3), np.float32)
    orqs, grids, win = gpu_grid_case(gpu, hg, oracle_lib, empty, [{}])
    res = gpu.search_candidates(empty, k=8)
    check(res, expected(hg, o, orqs, grids, win, 8, 64, 0.0))
    # roll_limit leaving no roll: no candidate, grasp_per_cloud is the roll -1 record
    xyz = clouds["pcd4"]
    rq = hg.make_request(roll_begin=5, roll_limit=3)
    res = gpu.search_candidates(xyz, [rq], k=8)
    assert int(res["n_candidates"][0]) == 0 and res["grasp"][0].roll_index == -1
    assert bytes(res["grasp"]) == bytes(gpu.search_batch_requests(xyz, [0, len(xyz)], [rq])["grasp"])
    # fewer eligible cells than k: one roll of a 20 x 20 area
    small = dict(area=(20.0, 20.0), roll_limit=1)
    orqs, grids, win = gpu_grid_case(gpu, hg, oracle_lib, xyz, [small])
    res = gpu.search_candidates(xyz, [hg.make_request(**small)], k=256, per_unit=1024)
    exp = expected(hg, o, orqs, grids, win, 256, 1024, 0.0)
    assert 1 < len(exp) < 256
    check(res, exp)
    # a huge min_distance: exactly the best
    res = gpu.search_candidates(clouds["table1"], k=64, min_distance=1e6)
    assert int(res["n_candidates"][0]) == 1
    assert bytes(res["candidates"][0].grasp) == bytes(res["grasp"][0])


def test_bad_parameters(gpu, hg, clouds):
    xyz = clouds["pcd4"]
    off = [0, len(xyz)]
    bad = [dict(k=0), dict(k=257), dict(k=16, per_unit=15), dict(k=16, per_unit=1025), dict(k=4, min_distance=float("nan"))]
    bad += [dict(k=4, reserved=i) for i in range(4)]
    for b in bad:
        rp = hg.haf_rank_params()
        rp.k, rp.per_unit, rp.min_distance = b.get("k", 16), b.get("per_unit", 0), b.get("min_distance", 0.0)
        if "reserved" in b:
            rp.reserved[b["reserved"]] = 1
        with pytest.raises(hg.HafError) as e:
            gpu.search_batch_candidates(xyz, off, [hg.make_request()], rank_params=rp)
        assert e.value.code == -1, b
    gpu.search_candidates(xyz, k=16, per_unit=16)   # the context is still usable


def test_two_gpus_equal_one(hg, trained_model, gpu, clouds):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    xyz, off, ro, reqs, _, _ = _mixed_batch(clouds, hg)
    grp = hg.GraspSearch(FEATURES, RANGE, trained_model, devices=[0, 1])
    try:
        same(grp.search_batch_candidates(xyz, off, reqs, ro, k=16, min_distance=0.03),
             gpu.search_batch_candidates(xyz, off, reqs, ro, k=16, min_distance=0.03))
    finally:
        grp.close()


def test_launch_count(gpu, hg, clouds):
    """the candidates add the same launches whatever k and the number of clouds in the chunk"""
    import torch
    names = sorted(clouds.files)
    for n_clouds in (4, 16):
        xs = [clouds[names[i % len(names)]] for i in range(n_clouds)]
        off = np.concatenate([[0], np.cumsum([len(x) for x in xs])])
        d = torch.from_numpy(np.concatenate(xs)).cuda()
        reqs = [hg.make_request() for _ in range(n_clouds)]
        gpu.search_batch_requests(d, off, reqs)
        base = gpu.timing().launches
        assert gpu.timing().n_chunks == 1
        for k in (1, 16, 256):
            gpu.search_batch_candidates(d, off, reqs, k=k, min_distance=0.02)
            assert gpu.timing().launches == base + RANK_KERNELS_ONE_CHUNK, (n_clouds, k)


def test_cli_top(hg, gpu, trained_model, tmp_path):
    from haf_grasping_b200 import build
    pcd_files = np.load(os.path.join(GOLDEN, "pcd_files.npz"))
    cli = build.build_cli()
    names = ("pcd2", "table1", "pcd4")
    paths = []
    for name in names:
        f = tmp_path / (name + ".pcd")
        f.write_bytes(pcd_files[name].tobytes())
        paths.append(str(f))
    base = [cli, "--features", FEATURES, "--range", RANGE, "--model", trained_model]
    xyzs = gpu.pcd_decode_batch_to_host([pcd_files[n].tobytes() for n in names])
    for p, xyz in zip(paths, xyzs):
        plain = subprocess.run(base + ["--pcd", p, "--json"], capture_output=True, text=True, check=True).stdout
        out = subprocess.run(base + ["--pcd", p, "--json", "--top", "12", "--min-distance", "0.03", "--per-unit", "32"],
                             capture_output=True, text=True, check=True).stdout
        lines = out.splitlines()
        assert len(lines) == 2 and lines[0] + "\n" == plain
        got = json.loads(lines[1])["candidates"]
        res = gpu.search_candidates(xyz, k=12, per_unit=32, min_distance=0.03)
        assert len(got) == int(res["n_candidates"][0])
        for i, c in enumerate(got):
            r = res["candidates"][i]
            g = r.grasp
            assert (c["rank"], c["eval"], c["request"], c["row"], c["col"], c["roll_index"]) == (i, g.eval, r.request, g.row, g.col, g.roll_index)
            assert np.float32(c["score"]) == np.float32(r.score)
            assert c["averagedGraspPoint"] == list(g.averagedGraspPoint) and c["graspPoint1"] == list(g.graspPoint1)
            assert c["graspPoint2"] == list(g.graspPoint2) and c["approachVector"] == list(g.approachVector)
    # several files: one batch, each file's line and list as a run on that file alone prints them
    extra = ["--top", "5", "--min-distance", "0.02"]
    singles = "".join(subprocess.run(base + ["--pcd", p] + extra, capture_output=True, text=True, check=True).stdout for p in paths)
    args = list(base)
    for p in paths:
        args += ["--pcd", p]
    assert subprocess.run(args + extra, capture_output=True, text=True, check=True).stdout == singles
