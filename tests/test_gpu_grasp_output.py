"""Grasp poses on the device (haf_search_grasps / haf_search_batch_packed_grasps): the GraspOutput records of
transform_gp_in_wcs_and_publish (server.cpp:1274-1401) against the oracle's restatement (oracle/haf_oracle.cpp,
orc_transform_gp_in_wcs).  Every comparison is exact: the 13 float64 values with np.array_equal, eval / row / col / roll
index with ==, and records of two library calls byte for byte."""
import ctypes as C
import gzip
import json
import os

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE

pytestmark = pytest.mark.gpu

# kernels haf_search_grasps launches on top of haf_search for a goal that runs in one chunk: grasp_unit_kernel (once per
# chunk) + grasp_gather_kernel (once per call)
GRASP_KERNELS_ONE_CHUNK = 2

TILTED = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254)]
VARIANTS = [dict(approach=(0.5, 0.0, 0.8660254), center=(0.05, 0.2, 0.0)), dict(width=2, area=(30.0, 40.0)), dict(return_only_best=1)]


@pytest.fixture(scope="module")
def clouds():
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="module")
def trained_model(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("trained_g") / "substitute_trained.model")
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
    p = str(tmp_path_factory.mktemp("prob_model_g") / "substitute_trained.prob.model")
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


def _same(a, b):
    return bytes(a) == bytes(b)


def _check_record(rec, pose, row, col, roll, ev):
    assert np.array_equal(rec.as_array(), pose), (rec.as_array(), pose)
    assert (rec.eval, rec.row, rec.col, rec.roll_index) == (ev, row, col, roll)


def _check_best_vs_oracle(o, orq, ores, rec):
    b = ores["best"]
    pose = o.transform_gp_in_wcs(orq, ores["heights"][max(b.roll, 0)], b.row, b.col, b.roll)
    _check_record(rec, pose, b.row, b.col, b.roll, b.eval)


def _goal(gpu, o, oracle_lib, hg, xyz, **kw):
    grq, orq = hg.make_request(**kw), oracle_lib.make_request(**kw)
    res = gpu.search_grasps(xyz, [grq])
    plain = gpu.search(xyz, [grq], outputs=False)
    assert _same(res["best"], plain["best"])
    assert _same(res["best_per_request"][0], plain["best_per_request"][0])
    ores = o.search(xyz, orq, full=True)
    assert res["best"].astuple() == ores["best"].astuple()
    _check_best_vs_oracle(o, orq, ores, res["grasp"])
    assert _same(res["grasp"], res["grasp_per_request"][0])
    return res


def test_bundled_clouds_default_request(gpu, orc, oracle_lib, hg, clouds):
    for name in sorted(clouds.files):
        _goal(gpu, orc, oracle_lib, hg, clouds[name])


@pytest.mark.parametrize("kw", VARIANTS, ids=["tilted", "width2_area30x40", "only_best"])
def test_bundled_clouds_request_variants(gpu, orc, oracle_lib, hg, clouds, kw):
    for name in ("pcd2", "plastic_mug2", "table1"):
        _goal(gpu, orc, oracle_lib, hg, clouds[name], **kw)


def test_five_approach_vectors_per_request_and_per_roll(gpu, orc, oracle_lib, hg, clouds):
    xyz = clouds["table1"]
    R = gpu.R
    res = gpu.search_grasps(xyz, [hg.make_request(approach=a) for a in TILTED], per_roll=True)
    for a, av in enumerate(TILTED):
        orq = oracle_lib.make_request(approach=av)
        ores = orc.search(xyz, orq)
        _check_best_vs_oracle(orc, orq, ores, res["grasp_per_request"][a])
        assert np.array_equal(res["per_roll_top"][a], ores["per_roll_top"])
        for roll in range(R):
            top = ores["per_roll_top"][roll]
            pose = orc.transform_gp_in_wcs(orq, ores["heights"][roll], top[0], top[1], roll)
            _check_record(res["grasp_per_roll"][a][roll], pose, top[0], top[1], roll, max(int(top[2]) - 20, 10))
    win = res["best"].approach_idx
    assert _same(res["grasp"], res["grasp_per_request"][win])


def test_roll_range_leaves_other_rolls_untouched(gpu, orc, oracle_lib, hg, clouds, hg_grasp_array):
    xyz = clouds["table1"]
    R = gpu.R
    sentinel = hg_grasp_array(R, 0xA5)
    res = gpu.search_grasps(xyz, [hg.make_request(roll_begin=5, roll_limit=9)], per_roll=sentinel)
    fill = bytes(hg_grasp_array(1, 0xA5)[0])
    orq = oracle_lib.make_request()
    ores = orc.search(xyz, orq)
    for roll in range(R):
        rec = sentinel[roll]
        if 5 <= roll < 9:
            top = ores["per_roll_top"][roll]
            pose = orc.transform_gp_in_wcs(orq, ores["heights"][roll], top[0], top[1], roll)
            _check_record(rec, pose, top[0], top[1], roll, max(int(top[2]) - 20, 10))
        else:
            assert bytes(rec) == fill, roll
    b = res["best"]
    assert 5 <= b.roll < 9
    pose = orc.transform_gp_in_wcs(orq, ores["heights"][b.roll], b.row, b.col, b.roll)
    _check_record(res["grasp"], pose, b.row, b.col, b.roll, b.topval - 20)


@pytest.fixture(scope="module")
def hg_grasp_array(hg):
    def make(n, byte):
        arr = (hg.haf_grasp * n)()
        C.memset(arr, byte, C.sizeof(arr))
        return arr
    return make


def test_edge_cases(gpu, orc, oracle_lib, hg, clouds):
    G, R = gpu.G, gpu.R
    # no roll evaluated: roll -1, roll 0's matrices, h_locmax = -10 - 0.01, eval = -1000 - 20
    res = gpu.search_grasps(clouds["pcd2"], [hg.make_request(roll_begin=R)])
    assert res["best"].roll == -1 and res["best"].topval == -1000
    pose = orc.transform_gp_in_wcs(oracle_lib.make_request(), np.zeros((G, G), np.float32), -1, -1, -1)
    _check_record(res["grasp"], pose, -1, -1, -1, -1020)
    # an empty cloud, and a cloud with every point outside the box
    _goal(gpu, orc, oracle_lib, hg, np.zeros((0, 3), np.float32))
    far = clouds["pcd2"].copy()
    far[:, 0] += 10.0
    _goal(gpu, orc, oracle_lib, hg, far)


def test_large_grid_two_kernel_integral_path(hg, oracle_lib, trained_model):
    """G = 192 > 158: integral_rows_kernel + integral_cols_kernel"""
    from haf_grasping_b200 import synth
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, grid=192, roll_step_deg=45, roll_max_deg=190)
    try:
        o = oracle_lib.Oracle(FEATURES, RANGE, trained_model)
        xyz = synth.synth_cloud(77, 150000, r=0.96)
        kw = dict(area=(60.0, 52.0))
        res = g.search_grasps(xyz, [hg.make_request(**kw)])
        orq = oracle_lib.make_request(**kw)
        ores = o.search(xyz, orq, G=192, roll_step_deg=45, roll_max_deg=190)
        assert res["best"].astuple() == ores["best"].astuple()
        b = ores["best"]
        pose = o.transform_gp_in_wcs(orq, ores["heights"][max(b.roll, 0)], b.row, b.col, b.roll, roll_step_deg=45)
        _check_record(res["grasp"], pose, b.row, b.col, b.roll, b.eval)
    finally:
        g.close()


def _batch_clouds(clouds):
    from haf_grasping_b200 import synth
    cl = [clouds[k] for k in sorted(clouds.files)]
    cl.append(np.zeros((0, 3), np.float32))
    for i in range(50):
        cl.append(synth.synth_cloud(900 + i, 1000 + (i * 7919) % 20000))
    off = np.zeros(len(cl) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in cl])
    return cl, np.ascontiguousarray(np.concatenate(cl), np.float32), off


def test_batches_equal_single_goals(gpu, hg, clouds, monkeypatch):
    import torch
    cl, xyz, off = _batch_clouds(clouds)
    n, R = len(cl), gpu.R
    assert n >= 64 and xyz.nbytes >= (4 << 20)
    single = [gpu.search_grasps(c, per_roll=True) for c in cl]
    plain = gpu.search_batch_packed(xyz, off)

    def check(res):
        for c in range(n):
            assert _same(res["grasp"][c], single[c]["grasp"]), c
            assert _same(res["best"][c], plain[c]), c
            for roll in range(R):
                assert _same(res["grasp_per_roll"][c * R + roll], single[c]["grasp_per_roll"][0][roll]), (c, roll)

    check(gpu.search_batch_packed_grasps(torch.from_numpy(xyz).cuda(), off, per_roll=True))
    pinned = torch.from_numpy(xyz).pin_memory()
    for src in (pinned, xyz):   # pinned host memory (copy engine), pageable >= 4 MB (the library's own staging)
        for dual in (None, "0"):
            if dual is not None:
                monkeypatch.setenv("HAF_DUAL_STREAM", dual)
            check(gpu.search_batch_packed_grasps(src, off, per_roll=True))
            assert gpu.timing().n_chunks > 1
            monkeypatch.delenv("HAF_DUAL_STREAM", raising=False)
        # and without per-roll records
        res = gpu.search_batch_packed_grasps(src, off)
        for c in range(n):
            assert _same(res["grasp"][c], single[c]["grasp"]), c


def test_launch_count(gpu, hg, clouds):
    xyz = clouds["table1"]
    gpu.search(xyz, outputs=False)
    n_plain = gpu.timing().launches
    gpu.search_grasps(xyz)
    n_grasp = gpu.timing().launches
    assert gpu.timing().n_chunks == 1
    assert n_grasp - n_plain == GRASP_KERNELS_ONE_CHUNK
    gpu.search(xyz, outputs=False)
    assert gpu.timing().launches == n_plain


def test_graphs_alternating_entry_points(hg, trained_model, clouds):
    xyz = clouds["table1"]
    ref = hg.GraspSearch(FEATURES, RANGE, trained_model)
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, use_graph=True)
    try:
        want_plain = ref.search(xyz, outputs=False)
        want_grasp = ref.search_grasps(xyz, per_roll=True)
        replays = []
        for _ in range(4):
            p = g.search(xyz, outputs=False)
            assert _same(p["best"], want_plain["best"]) and np.array_equal(p["per_roll_top"], want_plain["per_roll_top"])
            q = g.search_grasps(xyz, per_roll=True)
            assert _same(q["best"], want_grasp["best"]) and _same(q["grasp"], want_grasp["grasp"])
            assert all(_same(a, b) for a, b in zip(q["grasp_per_roll"][0], want_grasp["grasp_per_roll"][0]))
            replays.append(g.timing().graph_replays)
        assert replays[-1] > replays[0]
    finally:
        g.close()
        ref.close()


def test_probability_mode(hg, oracle_lib, prob_model, clouds):
    g = hg.GraspSearch(FEATURES, RANGE, prob_model)
    try:
        o = oracle_lib.Oracle(FEATURES, RANGE, prob_model)
        for name in ("pcd2", "plastic_mug2"):
            xyz = clouds[name]
            res = g.search_grasps(xyz, [hg.make_request(svm_with_probability=1)])
            orq = oracle_lib.make_request()
            row, col, roll, _, top = o.search_prob(xyz, orq)["best"]
            assert (res["best"].row, res["best"].col, res["best"].roll, res["best"].topval) == (row, col, roll, top)
            M = o.build_transform((0.0, 0.0, 0.0), o.normalize_approach((0.0, 0.0, 1.0)), 1, max(roll, 0))
            heights = o.generate_grid(xyz, M, g.G)
            pose = o.transform_gp_in_wcs(orq, heights, row, col, roll)
            _check_record(res["grasp"], pose, row, col, roll, top - 20)
    finally:
        g.close()


@pytest.mark.parametrize("mode", ["FP32_GUARD", "FP64_EXACT"])
def test_svm_modes_give_tensor_mode_records(hg, gpu, trained_model, clouds, mode):
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, svm_mode=getattr(hg, "HAF_SVM_" + mode))
    try:
        for name in ("pcd2", "table1"):
            reqs = [hg.make_request(approach=a) for a in TILTED[:2]]
            a, b = gpu.search_grasps(clouds[name], reqs, per_roll=True), g.search_grasps(clouds[name], reqs, per_roll=True)
            assert _same(a["grasp"], b["grasp"])
            assert all(_same(x, y) for x, y in zip(a["grasp_per_request"], b["grasp_per_request"]))
            for r in range(len(reqs)):
                assert all(_same(x, y) for x, y in zip(a["grasp_per_roll"][r], b["grasp_per_roll"][r]))
    finally:
        g.close()


def test_two_gpus_equal_one(hg, gpu, trained_model, clouds):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    grp = hg.GraspSearch(FEATURES, RANGE, trained_model, devices=[0, 1])
    try:
        R = gpu.R
        xyz = clouds["table1"]
        reqs = [hg.make_request(approach=a) for a in TILTED]
        a, b = gpu.search_grasps(xyz, reqs, per_roll=True), grp.search_grasps(xyz, reqs, per_roll=True)
        assert _same(a["best"], b["best"]) and _same(a["grasp"], b["grasp"])
        assert all(_same(x, y) for x, y in zip(a["grasp_per_request"], b["grasp_per_request"]))
        for r in range(len(reqs)):
            assert all(_same(x, y) for x, y in zip(a["grasp_per_roll"][r], b["grasp_per_roll"][r]))
        none = [hg.make_request(roll_begin=R)]
        assert _same(gpu.search_grasps(xyz, none)["grasp"], grp.search_grasps(xyz, none)["grasp"])
        cl, xyz_all, off = _batch_clouds(clouds)
        cl, off = cl[:64], off[:65]
        xyz_all = xyz_all[:off[-1]]
        a, b = gpu.search_batch_packed_grasps(xyz_all, off, per_roll=True), grp.search_batch_packed_grasps(xyz_all, off, per_roll=True)
        assert bytes(a["grasp"]) == bytes(b["grasp"]) and bytes(a["grasp_per_roll"]) == bytes(b["grasp_per_roll"])
    finally:
        grp.close()
