"""Batches of depth images back-projected into the base frame on the device (haf_depth_to_xyz_batch, haf_search_batch_depth).

The back-projection must equal a numpy float32 restatement of the contract in include/hafgpu.h bit for bit (any NaN matches
any NaN); a search on the projected images must equal haf_search_batch_requests on the numpy clouds field for field; one
launch covers a whole batch.
"""
import ctypes as C
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import FEATURES, GOLDEN, RANGE

pytestmark = pytest.mark.gpu

GUARD_REL = 1e-5          # as test_gpu_batch_requests.py: many windows per context with the trained model
QNAN = np.uint32(0x7FC00000)
F32_CATALOGUE = np.array([0.0, -0.0, 1.0, 65535.0, -0.75, 1e-45, 3e-39, np.finfo(np.float32).max, -np.finfo(np.float32).max,
                          np.nan, np.inf, -np.inf, 0.5, 1.25, 2.0, 0.731], np.float32)
U16_CATALOGUE = np.array([0, 1, 65535, 700, 1234, 0, 2, 40000], np.uint16)


# ---------------------------------------------------------------------------------------------------------------------------
# numpy restatement of the contract
# ---------------------------------------------------------------------------------------------------------------------------
def restate(img, K, pose=None, scale=0.0):
    """float32 [H * W, 3] of one image: the formulas of include/hafgpu.h, one float32 rounding per operation"""
    u16 = img.dtype == np.uint16
    s = np.float32(scale) if scale != 0 else np.float32(0.001 if u16 else 1.0)
    kx, ky = np.float32(float(s) / K[0]), np.float32(float(s) / K[1])
    cxf, cyf = np.float32(K[2]), np.float32(K[3])
    H, W = img.shape
    v, u = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
    D = img.astype(np.float32)
    valid = (img != 0) if u16 else np.isfinite(img)
    with np.errstate(all="ignore"):
        x = ((u - cxf) * D) * kx
        y = ((v - cyf) * D) * ky
        z = D * s
        if pose is not None:
            m = np.asarray(pose, np.float32).reshape(4, 4)
            fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
            rows = [((m[r, 0] * x + m[r, 1] * y) + m[r, 2] * z) + m[r, 3] for r in range(3)]
            x, y, z = (np.where(fin, rows[r], c) for r, c in enumerate((x, y, z)))
    out = np.stack([x, y, z], -1).reshape(-1, 3).astype(np.float32)
    out.view(np.uint32)[~valid.reshape(-1)] = QNAN
    return out


def same(a, b):
    """bitwise equal, except that any NaN matches any NaN"""
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb]))


def look_at(target, height, tilt_deg=0.0):
    """camera -> base matrix of a camera `height` metres from `target`, looking down, tilted about the base x axis"""
    R = np.array([[1.0, 0, 0], [0, -1.0, 0], [0, 0, -1.0]])
    t = np.radians(tilt_deg)
    Rx = np.array([[1.0, 0, 0], [0, np.cos(t), -np.sin(t)], [0, np.sin(t), np.cos(t)]])
    R = Rx @ R
    M = np.eye(4)
    M[:3, :3] = R
    M[:3, 3] = np.asarray(target, np.float64) - height * R[:, 2]
    return M.astype(np.float32)


def render(xyz, pose, K, H, W):
    """U16 depth image (millimetres) of a base-frame cloud seen by the camera `pose` (nearest point per pixel)"""
    M = pose.astype(np.float64)
    c = (xyz.astype(np.float64) - M[:3, 3]) @ M[:3, :3]
    with np.errstate(all="ignore"):
        u = np.round(K[0] * c[:, 0] / c[:, 2] + K[2])
        v = np.round(K[1] * c[:, 1] / c[:, 2] + K[3])
    ok = (c[:, 2] > 0.05) & (u >= 0) & (u < W) & (v >= 0) & (v < H)
    depth = np.full(H * W, np.inf)
    np.minimum.at(depth, (v[ok] * W + u[ok]).astype(np.int64), c[ok, 2])
    return np.where(np.isfinite(depth), np.round(depth * 1000.0), 0).astype(np.uint16).reshape(H, W)


def heightfield(seed):
    """a synthetic scene (haf_grasping_b200.synth: a floor and eight Gaussian objects)"""
    from haf_grasping_b200 import synth
    return synth.synth_cloud(seed, 60000)


@pytest.fixture(scope="module")
def clouds():
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="module")
def trained_model(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("trained_depth") / "substitute_trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(p, "wb") as dst:
        dst.write(src.read())
    return p


@pytest.fixture(scope="module")
def gpu(hg, trained_model):
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, guard_rel=GUARD_REL)
    yield g
    g.close()


def _check(gpu, images, Ks, poses, scales):
    got = gpu.depth_to_xyz_batch_to_host(images, Ks, poses, scales)
    _, po = gpu.depth_to_xyz_batch(images, Ks, poses, scales)
    assert list(po) == list(np.cumsum([0] + [im.shape[0] * im.shape[1] for im in images]))
    for i, im in enumerate(images):
        want = restate(im, Ks[i], poses[i], scales[i])
        assert same(got[i], want), i


RIGID = look_at((0.05, -0.02, 0.0), 0.7, 30.0)
ZERO_ENTRIES = np.array([[0.0, 1.0, 0.0, 0.1], [0.0, 0.0, -1.0, 0.0], [-1.0, 0.0, 0.0, 0.8], [0, 0, 0, 1]], np.float32)
POSES = [None, np.eye(4, dtype=np.float32), RIGID, ZERO_ENTRIES]
INTRINSICS = [(525.0, 520.5, 319.5, 239.5), (300.0, 290.0, -3.25, 0.5), (61.7, 80.3, 700.0, -12.75), (1.0, 2.0, 0.0, 0.0)]


def _image(rng, enc, h, w):
    cat = U16_CATALOGUE if enc == np.uint16 else F32_CATALOGUE
    img = cat[rng.integers(0, len(cat), (h, w))]
    if enc == np.uint16:
        img = np.where(rng.random((h, w)) < 0.5, rng.integers(0, 65536, (h, w)), img).astype(np.uint16)
    else:
        img = np.where(rng.random((h, w)) < 0.5, rng.uniform(-0.5, 3.0, (h, w)), img).astype(np.float32)
    return img


def _padded(img, extra):
    """the same image in a buffer whose rows are `extra` elements longer (a strided view)"""
    buf = np.full((img.shape[0], img.shape[1] + extra), 7, img.dtype)
    buf[:, :img.shape[1]] = img
    return buf[:, :img.shape[1]]


@pytest.mark.parametrize("enc", [np.uint16, np.float32])
@pytest.mark.parametrize("scale", [0.0, 1.0 / 5000.0, 1.0])
def test_back_projection_matches_the_contract(gpu, enc, scale):
    rng = np.random.default_rng(3 + int(scale * 5000))
    images, Ks, poses, scales = [], [], [], []
    k = 0
    for w in (1, 2, 3, 31, 33, 640):
        for h in (1, 480):
            img = _image(rng, enc, h, w)
            for padded in (False, True):
                images.append(_padded(img, 1 + k % 3) if padded else img)
                Ks.append(INTRINSICS[k % len(INTRINSICS)])
                poses.append(POSES[k % len(POSES)])
                scales.append(scale)
                k += 1
    _check(gpu, images, Ks, poses, scales)


def test_mixed_batch_with_empty_images(gpu):
    rng = np.random.default_rng(21)
    images = [np.zeros((0, 5), np.uint16), _image(rng, np.uint16, 7, 9), np.zeros((4, 0), np.float32), _image(rng, np.float32, 5, 33),
              np.zeros((0, 0), np.uint16), _padded(_image(rng, np.uint16, 13, 31), 3), _image(rng, np.float32, 480, 640),
              np.zeros((0, 2), np.float32)]
    Ks = [INTRINSICS[i % 4] for i in range(len(images))]
    poses = [POSES[i % 4] for i in range(len(images))]
    scales = [0.0, 0.0002, 0.0, 0.5, 1.0, 1.0 / 5000.0, 0.0, 0.0]
    _check(gpu, images, Ks, poses, scales)


def test_sources_agree(gpu):
    """pageable below and above 4 MB (staging thread), pinned, CUDA tensor"""
    import torch
    rng = np.random.default_rng(5)
    K = INTRINSICS[0]
    for n in (3, 40):                                     # 0.6 MB and 8.2 MB of U16
        stack = np.stack([_image(rng, np.uint16, 320, 320) for _ in range(n)])
        want = [restate(im, K, RIGID) for im in stack]
        pinned = torch.empty(stack.shape, dtype=torch.int16, pin_memory=True)
        pinned.numpy()[:] = stack.view(np.int16)
        for src in (stack, list(stack), pinned, torch.from_numpy(stack.view(np.int16)).cuda()):
            got = gpu.depth_to_xyz_batch_to_host(src, K, RIGID)
            assert len(got) == n and all(same(g, w) for g, w in zip(got, want))
    f32 = np.stack([_image(rng, np.float32, 64, 48) for _ in range(5)])
    got = gpu.depth_to_xyz_batch_to_host(torch.from_numpy(f32).cuda(), K, None, 0.25)
    assert all(same(g, restate(im, K, None, 0.25)) for g, im in zip(got, f32))


def test_one_launch_per_call(gpu):
    rng = np.random.default_rng(6)
    for n in (1, 7, 512):
        imgs = [_image(rng, np.uint16, 8 + i % 5, 16 + i % 3) for i in range(n)]
        gpu.depth_to_xyz_batch(imgs, INTRINSICS[0])
        l0 = gpu.launch_count()
        gpu.depth_to_xyz_batch(imgs, INTRINSICS[0])
        assert gpu.launch_count() - l0 == 1, n
    empty = [np.zeros((0, 4), np.uint16), np.zeros((3, 0), np.float32)]
    l0 = gpu.launch_count()
    d, po = gpu.depth_to_xyz_batch(empty, INTRINSICS[0])
    assert gpu.launch_count() == l0 and d == 0 and list(po) == [0, 0, 0]


# ---------------------------------------------------------------------------------------------------------------------------
# search parity: images rendered from the bundled clouds and from synthetic heightfields
# ---------------------------------------------------------------------------------------------------------------------------
CAM = (300.0, 300.0, 159.5, 119.5)


def _scenes(clouds):
    names = ["pcd2", "plastic_mug2", "pcd12", "table1", "pcd3", "table2"]
    scenes = []
    for i, n in enumerate(names):
        xyz = clouds[n]
        target = (float(np.median(xyz[:, 0])), float(np.median(xyz[:, 1])), 0.0)
        scenes.append((xyz, look_at(target, 0.7, 30.0 * (i % 2))))
    for seed in (1, 2, 3):
        scenes.append((heightfield(seed), look_at((0.0, 0.0, 0.0), 0.7, 30.0 * (seed % 2))))
    imgs, poses, want = [], [], []
    for xyz, pose in scenes:
        img = render(xyz, pose, CAM, 240, 320)
        imgs.append(img)
        poses.append(pose)
        want.append(restate(img, CAM, pose))
        assert np.isfinite(want[-1]).all(1).sum() > 150          # every scene is seen by its camera
    return imgs, poses, want


def _requests(hg, want, per_image, seed):
    rng = np.random.default_rng(seed)
    reqs, ro = [], [0]
    tilted = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (0.0, -0.5, 0.8660254)]
    for c, xyz in enumerate(want):
        fin = xyz[np.isfinite(xyz).all(1)]
        centre = np.median(fin, 0) if len(fin) else np.zeros(3)
        for j in range(per_image[c]):
            reqs.append(hg.make_request(center=tuple(float(v) for v in centre + rng.uniform(-0.03, 0.03, 3)),
                                        approach=tilted[(c + j) % 3], width=1 + j % 2))
        ro.append(len(reqs))
    return reqs, ro


def _assert_same(a, b, keys):
    for k in keys:
        x, y = a[k], b[k]
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y), k
        else:
            assert len(x) == len(y), k
            for i in range(len(x)):
                assert bytes(x[i]) == bytes(y[i]), (k, i)


@pytest.mark.parametrize("shape", ["one", "three", "varying"])
def test_search_parity_with_numpy_clouds(gpu, hg, clouds, shape):
    imgs, poses, want = _scenes(clouds)
    n = len(imgs)
    per = {"one": [1] * n, "three": [3] * n, "varying": [1 + (c * 5) % 4 for c in range(n)]}[shape]
    reqs, ro = _requests(hg, want, per, seed=len(shape))
    xyz = np.concatenate(want)
    po = np.cumsum([0] + [len(w) for w in want])
    kw = dict(grasps=True, per_roll=True, per_roll_top=True)
    a = gpu.search_batch_depth(imgs, CAM, poses, 0.0, reqs, ro, **kw)
    b = gpu.search_batch_requests(xyz, po, reqs, ro, **kw)
    assert list(a["point_offsets"]) == list(po)
    _assert_same(a, b, ("best", "best_per_request", "grasp", "grasp_per_request", "grasp_per_roll", "per_roll_top"))


def _flat_bytes(x):
    return b"".join(_flat_bytes(e) for e in x) if isinstance(x, list) else bytes(x)


def test_single_goal_through_the_device_pointer(gpu, hg, clouds):
    imgs, poses, want = _scenes(clouds)
    for c in (0, 3, 7):
        reqs, _ = _requests(hg, [want[c]], [2], seed=c)
        d, po = gpu.depth_to_xyz_batch([imgs[c]], CAM, [poses[c]])
        a = gpu.search_grasps(d, reqs, per_roll=True, outputs=True, n_points=int(po[1]), stride_bytes=12)
        b = gpu.search_grasps(want[c], reqs, per_roll=True, outputs=True)
        for k in ("graspseval", "mask", "heights", "per_roll_top"):
            assert np.array_equal(a[k], b[k]), (c, k)
        assert bytes(a["best"]) == bytes(b["best"]) and bytes(a["grasp"]) == bytes(b["grasp"]), c
        for k in ("best_per_request", "grasp_per_request", "grasp_per_roll"):
            assert _flat_bytes(a[k]) == _flat_bytes(b[k]), (c, k)


def test_against_oracle(gpu, hg, oracle_lib, trained_model, clouds):
    """one rendered bundled scene: the record equals the oracle's on the valid points of the numpy cloud"""
    o = oracle_lib.Oracle(FEATURES, RANGE, trained_model)
    xyz = clouds["plastic_mug2"]
    pose = look_at((0.02, 0.0, 0.0), 0.7, 30.0)
    img = render(xyz, pose, CAM, 240, 320)
    cloud = restate(img, CAM, pose)
    fin = cloud[np.isfinite(cloud).all(1)]
    assert len(fin) > 500
    centre = tuple(float(v) for v in np.median(fin, 0))
    kws = [dict(center=centre), dict(center=centre, approach=(0.5, 0.0, 0.8660254), width=2)]
    res = gpu.search_batch_depth([img], CAM, [pose], 0.0, [hg.make_request(**kw) for kw in kws], [0, 2])
    for r, kw in enumerate(kws):
        orq = oracle_lib.make_request(**kw)
        ores = o.search(np.ascontiguousarray(fin), orq, full=True)
        b = ores["best"]
        assert res["best_per_request"][r].astuple() == b.astuple()
        p = o.transform_gp_in_wcs(orq, ores["heights"][max(b.roll, 0)], b.row, b.col, b.roll)
        rec = res["grasp_per_request"][r]
        assert np.array_equal(rec.as_array(), p)
        assert (rec.eval, rec.row, rec.col, rec.roll_index) == (b.eval, b.row, b.col, b.roll)


def test_candidates_on_the_device_pointer(gpu, hg, clouds):
    imgs, poses, want = _scenes(clouds)
    reqs, ro = _requests(hg, want, [2] * len(want), seed=8)
    d, po = gpu.depth_to_xyz_batch(imgs, CAM, poses)
    a = gpu.search_batch_candidates(d, po, reqs, ro, k=8, min_distance=0.02)
    b = gpu.search_batch_candidates(np.concatenate(want), po, reqs, ro, k=8, min_distance=0.02)
    assert bytes(a["candidates"]) == bytes(b["candidates"]) and np.array_equal(a["n_candidates"], b["n_candidates"])
    assert bytes(a["best"]) == bytes(b["best"]) and bytes(a["grasp"]) == bytes(b["grasp"])


def test_graphs_replay_new_images(hg, trained_model, clouds):
    imgs, poses, want = _scenes(clouds)
    reqs, ro = _requests(hg, want, [2] * len(want), seed=4)
    ref = hg.GraspSearch(FEATURES, RANGE, trained_model, guard_rel=GUARD_REL)
    g = hg.GraspSearch(FEATURES, RANGE, trained_model, use_graph=True, guard_rel=GUARD_REL)
    try:
        sets = []
        for shift in (0, 1):        # new images of the same shape: the scenes shifted by one pixel
            im = [np.roll(x, shift, axis=1) for x in imgs]
            sets.append((im, ref.search_batch_depth(im, CAM, poses, 0.0, reqs, ro, per_roll=True)))
        replays = []
        for _ in range(3):
            for im, want_res in sets:
                got = g.search_batch_depth(im, CAM, poses, 0.0, reqs, ro, per_roll=True)
                for k in ("best", "best_per_request", "grasp", "grasp_per_request", "grasp_per_roll"):
                    assert bytes(got[k]) == bytes(want_res[k]), k
                replays.append(g.timing().graph_replays)
        assert replays[-1] > replays[0]
    finally:
        g.close()
        ref.close()


def _bad_cases(hg):
    """(field edits, message fragment) of every validation rule"""
    return [(dict(width=1 << 24), "width and height"), (dict(height=-1), "width and height"), (dict(encoding=3), "encoding"),
            (dict(step=13), "step"), (dict(step=6), "step"), (dict(step=-8), "step"), ("span", "byte span"),
            (dict(fx=float("nan")), "fx"), (dict(cy=float("inf")), "fx"), (dict(fy=0.0), "fx"),
            (dict(depth_scale=1.5), "depth_scale"), (dict(depth_scale=-0.001), "depth_scale"), (dict(depth_scale=float("nan")), "depth_scale"),
            (dict(has_pose=2), "has_pose"), ("pose", "camera_to_base"), ("reserved", "reserved")]


def test_bad_arguments_name_the_lowest_image(gpu, hg):
    rng = np.random.default_rng(9)
    imgs = [_image(rng, np.uint16, 6, 4) for _ in range(5)]
    data, off, recs, n = gpu._depth_batch(imgs, INTRINSICS[0], RIGID, 0.0)
    good = gpu.depth_to_xyz_batch_to_host(imgs, INTRINSICS[0], RIGID)
    L = gpu.L
    for case, text in _bad_cases(hg):
        for bad_at in (3, 1):
            rs = (hg.haf_depth_image * n)()
            C.memmove(rs, recs, C.sizeof(rs))
            offs = (C.c_size_t * (n + 1))(*off)
            if case == "span":                   # images bad_at and 4 get one byte too many
                offs = (C.c_size_t * (n + 1))(*[int(o) + (k > bad_at) + (k > 4) for k, o in enumerate(off)])
            for i in (bad_at, 4):                # the lowest bad image is named
                r = rs[i]
                if case == "span":
                    pass
                elif case == "pose":
                    r.camera_to_base[5] = float("inf")
                elif case == "reserved":
                    r.reserved[1] = 1
                else:
                    for k, v in case.items():
                        setattr(r, k, v)
            po = (C.c_size_t * (n + 1))(*([12345] * (n + 1)))
            d = C.c_void_p(777)
            rc = L.haf_depth_to_xyz_batch(gpu.h, data.ctypes.data_as(C.c_void_p), offs, n, rs, C.byref(d), po)
            msg = (L.haf_last_error(gpu.h) or b"").decode()
            assert rc == -1 and msg.startswith("depth image %d: " % bad_at) and text in msg, (case, bad_at, msg)
            assert list(po) == [12345] * (n + 1) and d.value == 777, case
    got = gpu.debug_pcd_xyz(sum(im.size for im in imgs))
    assert same(got, np.concatenate(good))         # no device work was done
    rs = (hg.haf_depth_image * n)()
    C.memmove(rs, recs, C.sizeof(rs))
    rs[2].reserved[0] = 3
    with pytest.raises(hg.HafError) as e:
        gpu.search_batch_depth((data, off, rs))
    assert e.value.code == -1 and "depth image 2: " in str(e.value)


def test_two_gpus_equal_one(hg, gpu, trained_model, clouds):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    imgs, poses, want = _scenes(clouds)
    reqs, ro = _requests(hg, want, [1 + c % 3 for c in range(len(want))], seed=12)
    grp = hg.GraspSearch(FEATURES, RANGE, trained_model, devices=[0, 1], guard_rel=GUARD_REL)
    try:
        a = gpu.search_batch_depth(imgs, CAM, poses, 0.0, reqs, ro, per_roll=True, per_roll_top=True)
        b = grp.search_batch_depth(imgs, CAM, poses, 0.0, reqs, ro, per_roll=True, per_roll_top=True)
        _assert_same(a, b, ("best", "best_per_request", "grasp", "grasp_per_request", "grasp_per_roll", "per_roll_top", "point_offsets"))
        assert all(same(x, y) for x, y in zip(grp.depth_to_xyz_batch_to_host(imgs, CAM, poses), want))
    finally:
        grp.close()


def _write_pgm(path, img):
    h, w = img.shape
    path.write_bytes(b"P5\n# depth, mm\n%d %d\n65535\n" % (w, h) + img.astype(">u2").tobytes())


def _write_binary_pcd(path, xyz):
    hdr = ("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nCOUNT 1 1 1\nWIDTH %d\n"
           "HEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %d\nDATA binary\n" % (len(xyz), len(xyz)))
    path.write_bytes(hdr.encode() + np.ascontiguousarray(xyz, "<f4").tobytes())


def test_cli_depth_prints_what_pcd_prints(clouds, trained_model_path, tmp_path):
    from haf_grasping_b200 import build
    cli = build.build_cli()
    pose = look_at((0.0, 0.0, 0.0), 0.7, 30.0)
    depth_args, pcd_args = [], []
    for name in ("pcd2", "plastic_mug2", "pcd3"):
        img = render(clouds[name], pose, CAM, 240, 320)
        p = tmp_path / ("%s.pgm" % name)
        _write_pgm(p, img)
        depth_args += ["--depth", str(p)]
        q = tmp_path / ("%s.pcd" % name)
        _write_binary_pcd(q, restate(img, CAM, pose))
        pcd_args += ["--pcd", str(q)]
    base = [cli, "--features", FEATURES, "--range", RANGE, "--model", trained_model_path, "--center", "0", "0", "0.05"]
    cam = ["--camera"] + [repr(v) for v in CAM] + ["--camera-pose"] + [repr(float(v)) for v in pose.reshape(-1)]
    for extra in ([], ["--json"], ["--top", "4"], ["--top", "3", "--json", "--min-distance", "0.02"]):
        want = subprocess.run(base + pcd_args + extra, capture_output=True, text=True, check=True).stdout
        got = subprocess.run(base + depth_args + cam + extra, capture_output=True, text=True, check=True).stdout
        assert got == want, extra
        assert len(got.splitlines()) >= 3
