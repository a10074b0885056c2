"""Batched goals with their own requests (haf_search_batch_requests): every output of a cloud equals what haf_search_grasps
returns for that cloud with that request list, and the unit parameters the call builds on the device are bit-equal to the
host build of haf_search_grasps.  Every comparison is exact (bytes of the records, n_guard aside: batch calls report 0)."""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE

pytestmark = pytest.mark.gpu

TILTED = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254)]
# Guard band of this module's contexts.  Its calls score far more windows per context than the other suites, and the tensor
# path's audit (an FP64 re-evaluation of the guard band and of a 1-in-4096 sample, whose members depend on the order of the
# window list) meets windows of this model whose contraction is off by up to ~1.04e-6 E.  That is inside the default band of
# 4e-6 E, but under the 4x margin the audit demands, so such a call is refused whichever entry point makes it (single goals
# included).  1e-5 E keeps the audit on, with the margin.
GUARD_REL = 1e-5


@pytest.fixture(scope="module")
def clouds():
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="module")
def trained_model(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("trained_br") / "substitute_trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(p, "wb") as dst:
        dst.write(src.read())
    return p


@pytest.fixture(scope="module")
def gpu(hg, trained_model):
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, guard_rel=GUARD_REL)
    yield g
    g.close()


@pytest.fixture(scope="module")
def batch(clouds):
    """every bundled cloud, replicated to 64 clouds (14 MB: the pageable path stages it with the library's own threads)"""
    names = sorted(clouds.files)
    cl = [clouds[names[i % len(names)]] for i in range(64)]
    off = np.zeros(len(cl) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in cl])
    return cl, np.ascontiguousarray(np.concatenate(cl), np.float32), off


def _no_guard(b):
    c = type(b).from_buffer_copy(b)
    c.n_guard = 0
    return bytes(c)


def _requests(hg, per_cloud, seed):
    """per-cloud centres, areas, widths, tilted approach vectors, roll ranges and return_only_best; per_cloud[c] requests for cloud c"""
    rng = np.random.default_rng(seed)
    n = int(sum(per_cloud))
    areas = np.array([(32.0, 44.0), (30.0, 40.0), (27.5, 35.9), (40.0, 30.0)])[rng.integers(0, 4, n)]
    reqs = hg.make_requests(centers=rng.uniform(-0.04, 0.04, (n, 3)), approaches=np.array(TILTED)[rng.integers(0, len(TILTED), n)],
                            areas=areas, widths=rng.integers(1, 4, n), return_only_best=rng.integers(0, 2, n),
                            roll_begin=rng.integers(0, 3, n), roll_limit=rng.choice([0, 0, 7, 10], n))
    ro = np.zeros(len(per_cloud) + 1, np.int32)
    ro[1:] = np.cumsum(per_cloud)
    return reqs, ro


def _check_against_singles(gpu, res, single, ro):
    R = gpu.R
    for c, s in enumerate(single):
        assert _no_guard(res["best"][c]) == _no_guard(s["best"]), c
        assert bytes(res["grasp"][c]) == bytes(s["grasp"]), c
        for k, r in enumerate(range(ro[c], ro[c + 1])):
            assert _no_guard(res["best_per_request"][r]) == _no_guard(s["best_per_request"][k]), (c, k)
            assert bytes(res["grasp_per_request"][r]) == bytes(s["grasp_per_request"][k]), (c, k)
            assert np.array_equal(res["per_roll_top"][r], s["per_roll_top"][k]), (c, k)
            got = b"".join(bytes(g) for g in res["grasp_per_roll"][r * R:(r + 1) * R])
            assert got == b"".join(bytes(g) for g in s["grasp_per_roll"][k]), (c, k)


def test_unit_params_bit_equal_to_host_build(gpu, hg, clouds):
    """512 distinct requests: haf_search_grasps builds their unit parameters on the host, haf_search_batch_requests (one request
    per cloud) on the device"""
    R = gpu.R
    rng = np.random.default_rng(11)
    n = 512
    ap = rng.normal(size=(n, 3)) * rng.uniform(0.2, 5.0, (n, 1))   # unnormalised lengths, negative z
    special = [(0.0, 0.0, 1.0), (0.0, 0.0, -1.0), (-0.0, 0.0, 1.0), (0.0, -0.0, 1.0), (-0.0, -0.0, -2.5), (0.0, 0.0, 7.0),
               (1e-30, 0.0, 1.0), (0.0, -1e-30, -1.0), (1e-8, 1e-8, 1.0), (-1e-7, 2e-7, -0.3), (1.0, 0.0, 0.0), (0.0, -1.0, 0.0)]
    ap[:len(special)] = special
    centers = rng.uniform(-0.2, 0.2, (n, 3))
    centers[::7] = rng.uniform(-1e3, 1e3, (len(centers[::7]), 3))
    areas = np.stack([rng.choice([3.0, 13.5, 15.0, 17.9, 21.0, 31.0, 32.0, 44.0, 57.3], n),
                      rng.choice([2.0, 14.0, 16.5, 29.0, 44.0, 51.7], n)], 1)
    reqs = hg.make_requests(centers=centers, approaches=ap, areas=areas, widths=rng.integers(1, 5, n),
                            roll_begin=rng.choice([0, 0, 2, 5], n), roll_limit=rng.choice([0, 0, 6, 12], n))
    xyz = clouds["pcd4"]
    host = [[], [], []]
    for k in range(0, n, 64):   # one chunk per goal: 64 requests at a time
        gpu.search_grasps(xyz, list(reqs[k:k + 64]))
        for i, a in enumerate(gpu.debug_unit_params(64 * R)):
            host[i].append(a)
    host = [np.concatenate(h) for h in host]
    cl = np.ascontiguousarray(np.concatenate([xyz] * n), np.float32)
    off = np.arange(n + 1, dtype=np.int64) * len(xyz)
    gpu.search_batch_requests(cl, off, reqs)
    dev = gpu.debug_unit_params(n * R)
    for h, d in zip(host, dev):
        assert h.shape == d.shape == (n * R, h.shape[1])
        assert h.tobytes() == d.tobytes()
    assert np.all(host[0][:, 12:].view(np.uint32) == np.array([0.0, 0.0, 0.0, 1.0], np.float32).view(np.uint32))


@pytest.mark.parametrize("shape", ["one", "five", "varying"])
def test_equal_to_single_goals(gpu, hg, batch, monkeypatch, shape):
    import torch
    cl, xyz, off = batch
    n = len(cl)
    per_cloud = {"one": [1] * n, "five": [5] * n, "varying": list(np.random.default_rng(3).integers(1, 7, n))}[shape]
    reqs, ro = _requests(hg, per_cloud, seed=len(shape))
    single = [gpu.search_grasps(cl[c], list(reqs[ro[c]:ro[c + 1]]), per_roll=True) for c in range(n)]

    def run(src):
        res = gpu.search_batch_requests(src, off, reqs, ro, per_roll=True, per_roll_top=True)
        _check_against_singles(gpu, res, single, ro)

    run(torch.from_numpy(xyz).cuda())
    pinned = torch.from_numpy(xyz).pin_memory()
    for src in (pinned, xyz):   # pinned host memory (copy engine), pageable >= 4 MB (the library's own staging)
        for dual in (None, "0"):
            if dual is not None:
                monkeypatch.setenv("HAF_DUAL_STREAM", dual)
            run(src)
            assert gpu.timing().n_chunks > 1
            monkeypatch.delenv("HAF_DUAL_STREAM", raising=False)
    if shape != "one":   # chunks of 7 requests: clouds whose requests straddle a chunk boundary, on three streams
        monkeypatch.setenv("HAF_STAGE_SCHED", "7")
        assert any(ro[c] < k < ro[c + 1] for k in range(7, int(ro[-1]), 7) for c in range(n))
        run(pinned)
        assert gpu.timing().n_chunks >= int(ro[-1]) // 7
        monkeypatch.delenv("HAF_STAGE_SCHED")


def test_staged_chunks_wait_for_their_copies(gpu, hg, batch, monkeypatch):
    """Every chunk of a host-staged batch waits, on its own stream, for the copy piece that holds its last cloud (pieces are
    copied in order, so that piece's event covers every earlier one).  Five requests per cloud put chunk ends inside pieces,
    and chunks on different streams end in the same piece: each of them must wait for it, not only the first."""
    import torch
    cl, xyz, off = batch
    n = len(cl)
    reqs, ro = _requests(hg, [5] * n, seed=21)
    pinned = torch.from_numpy(xyz).pin_memory()
    shared = 0
    for sched in (None, "7"):
        if sched:
            monkeypatch.setenv("HAF_STAGE_SCHED", sched)
        for src in (pinned, xyz):   # copy engine; the library's own staging of pageable memory
            gpu.search_batch_requests(src, off, reqs, ro)
            w = gpu.debug_chunk_copy_waits()
            assert len(w) == gpu.timing().n_chunks > 1
            assert np.array_equal(w[1:, 0], w[:-1, 1] - (w[1:, 0] < w[:-1, 1]))   # chunks follow each other (sharing a cloud at most)
            assert w[-1, 1] == n
            assert np.all(w[:, 3] >= 0) and np.all(w[:, 4] >= w[:, 1]), w
            shared += sum(1 for k in range(1, len(w)) if any(w[i, 3] == w[k, 3] and w[i, 2] != w[k, 2] for i in range(k)))
    assert shared > 0
    gpu.search_batch_requests(torch.from_numpy(xyz).cuda(), off, reqs, ro)
    assert np.all(gpu.debug_chunk_copy_waits()[:, 3] == -1)


def test_against_oracle(gpu, hg, oracle_lib, trained_model, clouds):
    o = oracle_lib.Oracle(FEATURES, RANGE, trained_model)
    names = ["pcd2", "plastic_mug2", "pcd12", "table1"]
    kws = [[dict(center=(0.03, -0.02, 0.0), approach=TILTED[1]), dict(width=2, area=(30.0, 40.0))],
           [dict(approach=TILTED[3], center=(-0.01, 0.0, 0.01))],
           [dict(area=(27.0, 35.0), approach=TILTED[4]), dict(return_only_best=1), dict(width=3, approach=TILTED[2])],
           [dict(center=(0.02, 0.02, -0.01), approach=TILTED[1], width=2)]]
    flat = [kw for ks in kws for kw in ks]
    ro = np.cumsum([0] + [len(ks) for ks in kws])
    cl = [clouds[k] for k in names]
    off = np.cumsum([0] + [len(c) for c in cl])
    res = gpu.search_batch_requests(np.concatenate(cl), off, [hg.make_request(**kw) for kw in flat], ro)
    for c, xyz in enumerate(cl):
        for r in range(ro[c], ro[c + 1]):
            orq = oracle_lib.make_request(**flat[r])
            ores = o.search(xyz, orq, full=True)
            b = ores["best"]
            assert res["best_per_request"][r].astuple() == b.astuple()
            pose = o.transform_gp_in_wcs(orq, ores["heights"][max(b.roll, 0)], b.row, b.col, b.roll)
            rec = res["grasp_per_request"][r]
            assert np.array_equal(rec.as_array(), pose)
            assert (rec.eval, rec.row, rec.col, rec.roll_index) == (b.eval, b.row, b.col, b.roll)


def test_identical_requests_equal_batch_packed_grasps(gpu, hg, batch):
    import torch
    cl, xyz, off = batch
    rq = hg.make_request(approach=TILTED[1], center=(0.01, 0.0, 0.0), width=2)
    d = torch.from_numpy(xyz).cuda()
    want = gpu.search_batch_packed_grasps(d, off, rq, per_roll=True)
    got = gpu.search_batch_requests(d, off, [rq] * len(cl), per_roll=True)
    assert bytes(got["best"]) == bytes(want["best"])
    assert bytes(got["grasp"]) == bytes(want["grasp"])
    assert bytes(got["grasp_per_roll"]) == bytes(want["grasp_per_roll"])


def test_launch_count(gpu, hg, batch):
    import torch
    cl, xyz, off = batch
    d = torch.from_numpy(xyz).cuda()
    rq = hg.make_request()
    gpu.search_batch_packed_grasps(d, off, rq)
    n_grasp = gpu.timing().launches
    gpu.search_batch_requests(d, off, [rq] * len(cl))
    assert gpu.timing().launches == n_grasp + 1   # + expand_units_kernel
    gpu.search_batch_packed(d, off, rq)
    n_plain = gpu.timing().launches
    gpu.search_batch_requests(d, off, [rq] * len(cl), grasps=False)
    assert gpu.timing().launches == n_plain + 1   # no pose kernel


def test_graphs_replay_new_requests(hg, trained_model, clouds):
    import torch
    names = sorted(clouds.files)[:12]
    cl = [clouds[k] for k in names]
    off = np.cumsum([0] + [len(c) for c in cl])
    d = torch.from_numpy(np.ascontiguousarray(np.concatenate(cl), np.float32)).cuda()
    ro = np.arange(0, 2 * len(cl) + 1, 2)
    ref = hg.GraspSearch(FEATURES, RANGE, trained_model, guard_rel=GUARD_REL)
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, use_graph=True, guard_rel=GUARD_REL)
    try:
        sets = []
        for seed in (1, 2):   # same shape (areas, roll ranges), different centres and approach vectors
            rng = np.random.default_rng(seed)
            reqs = hg.make_requests(centers=rng.uniform(-0.03, 0.03, (len(ro) - 1, 3)).repeat(2, 0),
                                    approaches=np.array(TILTED)[rng.integers(0, 5, 2 * len(cl))])
            sets.append((reqs, ref.search_batch_requests(d, off, reqs, ro, per_roll=True)))
        replays = []
        for _ in range(3):
            for reqs, want in sets:
                got = g.search_batch_requests(d, off, reqs, ro, per_roll=True)
                for k in want:
                    assert bytes(got[k]) == bytes(want[k]), k
                replays.append(g.timing().graph_replays)
        assert replays[-1] > replays[0]
        assert bytes(sets[0][1]["grasp_per_request"]) != bytes(sets[1][1]["grasp_per_request"])
    finally:
        g.close()
        ref.close()


def test_two_gpus_equal_one(hg, gpu, trained_model, batch):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    grp = hg.GraspSearch(FEATURES, RANGE, trained_model, devices=[0, 1], guard_rel=GUARD_REL)
    try:
        cl, xyz, off = batch
        reqs, ro = _requests(hg, list(np.random.default_rng(5).integers(1, 7, len(cl))), seed=9)
        a = gpu.search_batch_requests(xyz, off, reqs, ro, per_roll=True, per_roll_top=True)
        b = grp.search_batch_requests(xyz, off, reqs, ro, per_roll=True, per_roll_top=True)
        for k in a:
            assert bytes(a[k]) == bytes(b[k]), k
    finally:
        grp.close()


def test_argument_errors(gpu, hg, clouds):
    xyz = np.concatenate([clouds["pcd4"], clouds["pcd5"]])
    off = [0, 200, 400]
    reqs = [hg.make_request(), hg.make_request(), hg.make_request()]
    for ro in ([0, 2, 1], [0, 0, 3], [0, 3, 3], [1, 2, 3], [-1, 1, 3]):   # decreasing, empty cloud, out of range
        with pytest.raises(hg.HafError) as e:
            gpu.search_batch_requests(xyz, off, reqs, ro)
        assert e.value.code == -1, ro
    mixed = [hg.make_request(), hg.make_request(svm_with_probability=1)]
    with pytest.raises(hg.HafError) as e:
        gpu.search_batch_requests(xyz, off, mixed)
    assert e.value.code == -1
    gpu.search_batch_requests(xyz, off, reqs, [0, 1, 3])   # and a valid call afterwards
