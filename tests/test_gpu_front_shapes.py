"""The front half of the search -- binning, integral image, window mask and compaction, and the tensor path's feature
staging -- against the CPU oracle at every shape and input its kernels branch on.

Reference, per unit: the oracle's generate_grid (with its clamp count), calc_intimage and pnt_in_box, on the unit's own
transform.  Heights are compared with == (the sign of a zero height is the only freedom: the device max is order-free, the
reference keeps the first zero it meets), integral images byte for byte, masks, the window set per unit and its count, and
the call's clamp count against the sum of the oracle's.

Every GPU case asserts, from the chunk record of haf_debug_chunk_copy_waits, the binning kernel, unit groups, units per
group, slices and integral variant it meant to reach.  The dispatch rule is restated in ``plan`` (hafgpu.cu, run_jobs_once)
so that the CPU check ``test_cases_cover_every_branch`` can show that the case list reaches every branch value; the GPU
cases compare the device's record with the restatement at the device's own SM count.

The point catalogue (``catalogue``) mixes non-finite coordinates, ulp ladders across the box edges, transformed z at -1,
just above it and around the -0.99 decode threshold, zeros, subnormals, a crowded cell, duplicates and a cloud whose height
overflows to +inf into single goals and batches.
"""
import math

import numpy as np
import pytest

from conftest import FEATURES, RANGE

SMEM_BIN = 200 * 1024          # dynamic shared memory of the whole-cloud binning kernel and the one-kernel integral image
MASK_CELLS = 4096              # cells per mask_windows_kernel CTA
FT_ROWS, FT_NW = 36, 64        # HAF_FT_ROWS, windows per features_tc_kernel CTA
B200_SMS = 148
FAST_TIER_REL, FAST_TIER_ABS = 5.5e-6, 5e-7   # tensor operands vs the exact scaled values (test_gpu_parity)
APPROACHES = [(0.0, 0.0, 1.0), (0.5, 0.0, 0.8660254), (-0.5, 0.0, 0.8660254), (0.0, 0.5, 0.8660254), (0.0, -0.5, 0.8660254),
              (0.3, 0.3, 0.9)]


# ---- the host's dispatch, restated -----------------------------------------------------------------------------------
def units_per_group_max(G):
    return min(16, SMEM_BIN // (G * G * 4))


def integral_variant(G):
    return 0 if G * (G + 1) * 8 <= SMEM_BIN else 1


def plan(G, sizes, units_per_cloud, sm_count, stride=12, bin_variant=0):
    """(kernel, unit groups, units per group, slices, integral variant) of one chunk, as run_jobs_once picks them"""
    n = len(sizes)
    GG = G * G
    upg = units_per_group_max(G)
    avg = sum(sizes) // max(1, n)
    if upg >= 1 and avg >= 8 * GG and n * 8 >= sm_count and bin_variant != 1:
        mu = max(units_per_cloud)
        ug = min(upg, max(1, mu))
        ngroups = -(-mu // ug)
        fixed = min(1.0, 4.2 * GG / max(avg, 1))
        best, slices = 0.0, 1
        for sl in range(1, 13):
            cost = math.ceil(n * ngroups * sl / sm_count) * (1.0 / sl + fixed)
            if sl == 1 or cost < best:
                best, slices = cost, sl
        return (1 if stride == 12 and bin_variant != 2 else 2, ngroups, ug, slices, integral_variant(G))
    return (0, 0, 0, 0, integral_variant(G))


def heads_tails(sizes, slices):
    """(head, tail) of every non-empty slice of the whole-cloud kernel's 16-byte loads (packed xyz on a 16-byte aligned base)"""
    out = set()
    off = 0
    for n in sizes:
        per = -(-n // slices) if n else 0
        for s in range(slices):
            p0, p1 = off + per * s, min(off + n, off + per * (s + 1))
            if p1 > p0:
                head = min((-p0) % 4, p1 - p0)
                out.add((head, (p1 - p0 - head) % 4))
        off += n
    return out


# ---- shape cases -------------------------------------------------------------------------------------------------------
# name, G, roll step, requests per cloud (approach indices), sizes (callable of the SM count), bin_variant, kernel meant,
# roll ranges (None or (begin, limit) per request), catalogue points mixed in
def _sizes_at(G, n_of_sm, total_of_sm=None, ragged=False, big_one=False):
    """cloud sizes: n clouds, average 8 G^2 (or the total given); ragged: empty and 1-7-point clouds at offsets that give every
    head and tail; big_one: one large cloud among tiny ones"""
    def f(sm):
        n = n_of_sm(sm)
        total = total_of_sm(sm) if total_of_sm else n * 8 * G * G
        if big_one:
            tiny = [1 + (i % 7) for i in range(n - 1)]
            return [total - sum(tiny)] + tiny
        if ragged:   # big, tiny, big, tiny, ..., then the remaining big clouds
            small = [0, 1, 2, 3, 5, 6, 7, 0, 4, 1, 3, 2][:max(0, n // 2 - 1)]
            rest = n - len(small)
            big = total - sum(small)
            per = [big // rest + (1 if i < big % rest else 0) for i in range(rest)]
            per[0] += 1; per[-1] -= 1   # odd offsets for what follows
            out = []
            for i in range(rest):
                out.append(per[i])
                if i < len(small):
                    out.append(small[i])
            return out
        base = total // n
        return [base + (1 if i < total - base * n else 0) for i in range(n)]
    return f


def _nwc(sm):
    return -(-sm // 8)       # fewest clouds that let the whole-cloud kernel run


CASES = [
    # binning kernels at G = 56
    dict(name="g56_point_parallel_natural", G=56, step=15, req=[0], sizes=lambda sm: [4000 + 37 * i for i in range(6)], kernel=0, cat=True),
    dict(name="g56_point_parallel_forced", G=56, step=15, req=[0], sizes=_sizes_at(56, _nwc), bin_variant=1, kernel=0, cat=True),
    dict(name="g56_whole_cloud_vec4_ragged", G=56, step=15, req=[0], sizes=_sizes_at(56, lambda sm: _nwc(sm) + 13, ragged=True), kernel=1, cat=True),
    dict(name="g56_whole_cloud_scalar", G=56, step=15, req=[0, 1, 2], sizes=_sizes_at(56, _nwc), bin_variant=2, kernel=2, cat=True),
    # the dispatch thresholds, exactly and one below
    dict(name="g56_threshold_exact", G=56, step=45, req=[0], sizes=_sizes_at(56, _nwc), kernel=1),
    dict(name="g56_threshold_clouds_minus_one", G=56, step=45, req=[0], sizes=_sizes_at(56, lambda sm: _nwc(sm) - 1), kernel=0),
    dict(name="g56_threshold_points_minus_one", G=56, step=45, req=[0], sizes=_sizes_at(56, _nwc, lambda sm: _nwc(sm) * 8 * 56 * 56 - 1), kernel=0),
    dict(name="g56_one_big_cloud_among_tiny", G=56, step=45, req=[0], sizes=_sizes_at(56, lambda sm: 2 * _nwc(sm), big_one=True), kernel=1),
    # units per cloud: 1, 16, 17, 60 (five approach vectors: row 2 changes inside a group), 72 (> HAF_BIN_MAXU)
    dict(name="g56_one_unit_per_cloud", G=56, step=180, req=[0], sizes=_sizes_at(56, _nwc), kernel=1),
    dict(name="g56_16_units_roll_ranges", G=56, step=45, req=[0, 1, 2, 3], ranges=[(0, 0), (1, 3), (0, 2), (3, 4)], sizes=_sizes_at(56, _nwc), kernel=1),
    dict(name="g56_17_units", G=56, step=11, req=[1], sizes=_sizes_at(56, _nwc), kernel=1),
    dict(name="g56_60_units_roll_ranges", G=56, step=15, req=[0, 1, 2, 3, 4], ranges=[(0, 0), (2, 9), (5, 7), (0, 0), (11, 12)], sizes=_sizes_at(56, _nwc), kernel=1, cat=True),
    dict(name="g56_72_units_point_parallel", G=56, step=15, req=[0, 1, 2, 3, 4, 5], ranges=[(0, 0), (3, 9), (0, 0), (0, 0), (1, 2), (0, 0)], sizes=lambda sm: [3000, 0, 2500, 7], kernel=0, cat=True),
    dict(name="g56_72_units_whole_cloud", G=56, step=15, req=[0, 1, 2, 3, 4, 5], ranges=[(0, 0), (3, 9), (0, 0), (0, 0), (1, 2), (0, 0)], sizes=_sizes_at(56, _nwc), kernel=1),
    # grid sides
    dict(name="g16_whole_cloud", G=16, step=15, req=[0, 1], sizes=_sizes_at(16, _nwc, ragged=True), kernel=1),
    dict(name="g58_whole_cloud_ug15", G=58, step=15, req=[0, 3], sizes=_sizes_at(58, _nwc), kernel=1),
    dict(name="g64_clamping_one_mask_cta", G=64, step=15, req=[0, 1], sizes=_sizes_at(64, _nwc), kernel=1, cat=True),
    dict(name="g64_clamping_point_parallel", G=64, step=15, req=[0, 1], sizes=lambda sm: [6000, 5, 4000], kernel=0, cat=True),
    dict(name="g66_two_mask_ctas", G=66, step=45, req=[0], sizes=lambda sm: [9000, 3], kernel=0),
    dict(name="g72_whole_cloud_ug9", G=72, step=45, req=[0, 1, 2], sizes=_sizes_at(72, _nwc), kernel=1),
    dict(name="g100_whole_cloud_ug5_clamping", G=100, step=45, req=[0, 1], sizes=_sizes_at(100, _nwc), kernel=1, cat=True),
    dict(name="g100_scalar_clamping", G=100, step=90, req=[1], sizes=_sizes_at(100, _nwc), bin_variant=2, kernel=2, cat=True),
    dict(name="g100_point_parallel_clamping", G=100, step=45, req=[1], sizes=lambda sm: [12000, 7, 1], kernel=0, cat=True),
    dict(name="g128_integral_one_row_pass", G=128, step=90, req=[0], sizes=lambda sm: [30000], kernel=0),
    dict(name="g130_integral_two_row_passes", G=130, step=90, req=[0], sizes=lambda sm: [30000, 2], kernel=0),
    dict(name="g158_last_small_integral", G=158, step=90, req=[0], sizes=lambda sm: [40000], kernel=0),
    dict(name="g160_first_two_kernel_integral", G=160, step=90, req=[0], sizes=lambda sm: [40000], kernel=0),
    dict(name="g162_whole_cloud_ug1", G=162, step=180, req=[0], sizes=_sizes_at(162, _nwc, big_one=True), kernel=1),
    dict(name="g226_whole_cloud_ug1", G=226, step=180, req=[0], sizes=_sizes_at(226, _nwc, big_one=True), kernel=1),
    dict(name="g228_point_parallel_always", G=228, step=180, req=[0], sizes=_sizes_at(228, _nwc, big_one=True), kernel=0),
    dict(name="g1024_one_cloud", G=1024, step=180, req=[0], sizes=lambda sm: [300000], kernel=0),
]
CATALOGUE_GRIDS = {56, 64, 100}


def case_plan(case, sm):
    sizes = case["sizes"](sm)
    R = 190 // case["step"]
    return sizes, plan(case["G"], sizes, [R * len(case["req"])] * len(sizes), sm, bin_variant=case.get("bin_variant", 0))


def clamping_grid(G):
    """a point a few ulps inside +r gets floor(100 (t + r)) == G at this side"""
    r = np.float32((0.5 * np.float32(G)) / 100.0)
    t = r
    for _ in range(64):
        t = np.nextafter(t, np.float32(0))
        if int(np.floor(np.float32(100) * np.float32(t + r))) >= G:
            return True
    return False


# ---- the point catalogue ---------------------------------------------------------------------------------------------------
def transform32(M, p):
    """pcl::transformPointCloud in float32, left to right, no FMA (numpy uses none): t [n, 3]"""
    m = np.asarray(M, np.float32).reshape(4, 4)
    p = np.asarray(p, np.float32).reshape(-1, 3)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    with np.errstate(over="ignore", invalid="ignore"):
        return np.stack([((m[i, 0] * x + m[i, 1] * y) + m[i, 2] * z) + m[i, 3] for i in range(3)], axis=1)


def ulps_around(v, k):
    """float32 values v - k ulps ... v + k ulps"""
    v = np.float32(v)
    i = np.array([v], np.float32).view(np.int32)[0].astype(np.int64)
    # monotone integer image of the floats
    key = i if i >= 0 else -(i & 0x7FFFFFFF)
    keys = key + np.arange(-k, k + 1)
    bits = np.where(keys >= 0, keys, (-keys) | 0x80000000).astype(np.uint32)
    return bits.view(np.float32)


def _solve(M, target):
    m = np.asarray(M, np.float64).reshape(4, 4)
    return np.linalg.solve(m[:3, :3], np.asarray(target, np.float64) - m[:3, 3]).astype(np.float32)


def _scan(M, base, row, k=1500, j=None):
    """points that step coordinate j (default: the one with the largest weight in `row` of M) by ulps around base"""
    m = np.asarray(M, np.float32).reshape(4, 4)
    j = int(np.argmax(np.abs(m[row, :3]))) if j is None else j
    pts = np.repeat(base[None, :], 2 * k + 1, axis=0)
    pts[:, j] = ulps_around(base[j], k)
    return pts, transform32(M, pts)


def edge_ladder(M, G, tz=0.05, n_ulps=64):
    """points whose transformed x (then y) lie within n_ulps ulps of -r and +r, the other coordinate well inside"""
    r = np.float32((0.5 * np.float32(G)) / 100.0)
    out = []
    for row in (0, 1):
        for edge in (-r, r):
            tgt = [0.0, 0.0, tz]
            tgt[row] = float(edge)
            tgt[1 - row] = 0.37 * float(r) * (1 if edge > 0 else -1)
            pts, t = _scan(M, _solve(M, tgt), row)
            near = np.isin(t[:, row], ulps_around(edge, n_ulps))
            out.append(pts[near])
    return np.concatenate(out)


def z_specials(M, G, where):
    """points inside the box whose transformed z is exactly -1, the first float above -1 the transform reaches (the translation
    of 0.15 leaves every other float near -1 out of reach), the floats around -0.99, and +0"""
    out = {}
    for name, want in (("z_minus_one", ulps_around(-1.0, 0)), ("z_above_minus_one", ulps_around(-1.0, 4)[5:]),
                       ("z_near_decode_threshold", ulps_around(np.float32(-0.99), 3)), ("z_zero", np.array([0.0], np.float32))):
        # every coordinate that enters z: the smaller its weight, the finer the steps of the transformed z
        m = np.asarray(M, np.float32).reshape(4, 4)
        scans = [_scan(M, _solve(M, [where[0], where[1], float(want[0])]), 2, k=4000, j=j) for j in range(3) if abs(m[2, j]) > 1e-3]
        pts, t = np.concatenate([p for p, _ in scans]), np.concatenate([q for _, q in scans])
        r = np.float32((0.5 * np.float32(G)) / 100.0)
        inside = (np.abs(t[:, 0]) < r) & (np.abs(t[:, 1]) < r)
        hit = pts[inside & np.isin(t[:, 2], want)]
        if name == "z_zero":
            hit = hit[np.signbit(t[inside & np.isin(t[:, 2], want)][:, 2]) == False][:2]   # noqa: E712 -- +0 only; see below
        if name == "z_above_minus_one" and len(hit):
            tz = transform32(M, hit)[:, 2]
            hit = hit[tz == tz.min()]
        out[name] = hit
    return out


def overflow_point(M, G):
    """a finite point whose x and z terms cancel exactly inside the box while its transformed z overflows to +inf, or None"""
    m = np.asarray(M, np.float32).reshape(4, 4)
    r = np.float32((0.5 * np.float32(G)) / 100.0)
    for x in np.linspace(1.72e38, 1.94e38, 12).astype(np.float32):
        with np.errstate(over="ignore", invalid="ignore"):
            if m[0, 1] == 0 or m[1, 2] == 0:
                return None
            y0 = np.float32(-(np.float64(m[0, 0] * x)) / np.float64(m[0, 1]))
            for y in ulps_around(y0, 8):
                s = np.float32(m[1, 0] * x) + np.float32(m[1, 1] * y)
                z0 = np.float32(-np.float64(s) / np.float64(m[1, 2]))
                zs = ulps_around(z0, 64)
                zs = zs[np.isfinite(zs)]
                t = transform32(M, np.stack([np.full(len(zs), x), np.full(len(zs), y), zs], axis=1))
                ok = (np.abs(t[:, 0]) < r) & (np.abs(t[:, 1]) < r) & np.isposinf(t[:, 2])
                if ok.any():
                    return np.array([x, y, zs[np.argmax(ok)]], np.float32)
    return None


NONFINITE = ["nan_x", "nan_y", "nan_z", "+inf_x", "-inf_x", "+inf_y", "-inf_y", "+inf_z", "-inf_z"]
FINITE = ["edge_ladder", "edge_ladder_below_z_minus_one", "z_minus_one", "z_above_minus_one", "z_near_decode_threshold", "z_zero",
          "signed_zero_inputs", "subnormals", "one_cell_many", "duplicates"]
CATALOGUE = NONFINITE + FINITE + ["overflow_to_inf"]


def catalogue(Ms, G, seed):
    """name -> float32 [k, 3] points for the unit transforms Ms (one ladder per unit).  Deterministic."""
    rng = np.random.default_rng(seed)
    r = float(np.float32((0.5 * np.float32(G)) / 100.0))
    cat = {k: [] for k in CATALOGUE}
    inner = _solve(Ms[0], [0.21 * r, -0.13 * r, 0.05])
    for i, name in enumerate(NONFINITE):
        p = np.repeat(inner[None, :], 3, axis=0)
        v = np.nan if name.startswith("nan") else (np.inf if name[0] == "+" else -np.inf)
        p[:, "xyz".index(name[-1])] = v
        cat[name].append(p)
    for u, M in enumerate(Ms):
        cat["edge_ladder"].append(edge_ladder(M, G))
        cat["edge_ladder_below_z_minus_one"].append(edge_ladder(M, G, tz=-1.5, n_ulps=8))
        where = (0.45 * r * np.cos(0.7 * u), 0.45 * r * np.sin(0.7 * u))
        for k, v in z_specials(M, G, where).items():
            cat[k].append(v)
        o = overflow_point(M, G)
        if o is not None:
            cat["overflow_to_inf"].append(o[None, :])
    zs = np.array([[0.0, 0.0, 0.0], [-0.0, 0.0, -0.0], [0.0, -0.0, 0.0], [-0.0, -0.0, -0.0]], np.float32)
    cat["signed_zero_inputs"].append(np.concatenate([zs, zs[::-1]]))
    sub = np.float32(1e-40)
    cat["subnormals"].append(np.array([[sub, -sub, 0.05], [-sub, sub, sub], [1e-45, 0.0, -1e-45], [sub, sub, -sub]], np.float32))
    c = _solve(Ms[0], [0.005 * r, 0.005 * r, 0.0])
    many = np.repeat(c[None, :], 3000, axis=0)
    many[:, 2] += rng.uniform(0.0, 0.2, 3000).astype(np.float32)
    cat["one_cell_many"].append(many)
    cat["duplicates"].append(np.repeat(many[:40], 8, axis=0))
    return {k: (np.concatenate(v).astype(np.float32) if v else np.zeros((0, 3), np.float32)) for k, v in cat.items()}


def base_cloud(seed, n, G):
    """smooth bumps over the box (heights that pass the mask's 0.03 threshold), cheap for millions of points"""
    rng = np.random.default_rng(seed)
    r = 0.5 * G / 100.0
    xy = rng.uniform(-0.98 * r, 0.98 * r, (n, 2)).astype(np.float32)
    c = rng.uniform(-0.6 * r, 0.6 * r, (4, 2))
    z = np.full(n, 0.02, np.float32)
    for k in range(4):
        z += np.float32(0.12) * np.exp(-((xy[:, 0] - c[k, 0]) ** 2 + (xy[:, 1] - c[k, 1]) ** 2) / (0.08 * r * r)).astype(np.float32)
    return np.concatenate([xy, z[:, None]], axis=1).astype(np.float32)


# ---- CPU: coverage of the case list --------------------------------------------------------------------------------------------
def test_cases_cover_every_branch():
    """the shape cases reach every branch value of binning, integral image and mask compaction (worked out for a 148-SM
    B200; the GPU cases re-check each against the device they run on)"""
    plans = {c["name"]: case_plan(c, B200_SMS) for c in CASES}
    for c in CASES:
        assert plans[c["name"]][1][0] == c["kernel"], c["name"]
    kernels = {p[0] for _, p in plans.values()}
    assert kernels == {0, 1, 2}
    ugs = {p[2] for _, p in plans.values() if p[0]}
    assert 16 in ugs and 1 in ugs and any(2 <= u <= 15 for u in ugs)
    assert any(units_per_group_max(c["G"]) == 0 for c in CASES)
    assert {units_per_group_max(G) for G in (58, 72, 100)} == {15, 9, 5}
    slices = {p[3] for _, p in plans.values() if p[0]}
    assert 1 in slices and 2 in slices and max(slices) >= 6, slices
    ht = set()
    for sizes, p in plans.values():
        if p[0] == 1:
            ht |= heads_tails(sizes, p[3])
    assert {h for h, _ in ht} == {0, 1, 2, 3} and {t for _, t in ht} == {0, 1, 2, 3}, ht
    Gs = {c["G"] for c in CASES}
    assert {p[4] for _, p in plans.values()} == {0, 1}
    assert any(integral_variant(G) == 0 and G > 128 for G in Gs) and integral_variant(158) == 0 and integral_variant(160) == 1
    assert {G % 8 for G in Gs} >= {0, 2, 4, 6} and any(G % 32 and integral_variant(G) for G in Gs)
    mask_ctas = {-(-G * G // MASK_CELLS) for G in Gs}
    assert 1 in mask_ctas and max(mask_ctas) > 1 and -(-64 * 64 // MASK_CELLS) == 1 and -(-66 * 66 // MASK_CELLS) == 2
    upc = {(190 // c["step"]) * len(c["req"]) for c in CASES}
    assert {1, 12, 16, 17, 60, 72} <= upc
    assert any((190 // c["step"]) * len(c["req"]) > 64 and plans[c["name"]][1][0] == 0 for c in CASES)
    assert any(c.get("ranges") and plans[c["name"]][1][0] for c in CASES)   # inactive units inside a whole-cloud group
    assert any(clamping_grid(c["G"]) and c.get("cat") for c in CASES) and not clamping_grid(56)
    cat_kernels = {(c["G"], plans[c["name"]][1][0]) for c in CASES if c.get("cat")}
    assert all((G, k) in cat_kernels for G in (56,) for k in (0, 1, 2)) and {G for G, _ in cat_kernels} == CATALOGUE_GRIDS
    # the thresholds: exactly at and one below
    nwc = _nwc(B200_SMS)
    assert len(plans["g56_threshold_exact"][0]) == nwc and sum(plans["g56_threshold_exact"][0]) // nwc == 8 * 56 * 56
    assert len(plans["g56_threshold_clouds_minus_one"][0]) == nwc - 1
    assert sum(plans["g56_threshold_points_minus_one"][0]) // nwc == 8 * 56 * 56 - 1


def test_catalogue_reaches_every_entry():
    """every catalogue entry exists at the catalogue's grid sides, for the default and a tilted approach vector; the ladder
    crosses both edges and, at a clamping side, reaches index G"""
    import haf_grasping_b200 as hg
    for G in sorted(CATALOGUE_GRIDS):
        r = np.float32((0.5 * np.float32(G)) / 100.0)
        reached = set()
        for av in (APPROACHES[0], APPROACHES[1]):
            Ms = [host_transform(hg, av, roll, 45) for roll in range(4)]
            cat = catalogue(Ms, G, 5)
            # (the default transform has z alone in row 2 and a translation of 0.15: z + 0.15 reaches every other float near
            # -1 only, and nothing cancels against an overflowing z; the tilted one reaches both)
            reached |= {k for k in CATALOGUE if len(cat[k])}
            t = transform32(Ms[0], cat["edge_ladder"])
            assert (t[:, 0] >= r).any() and (t[:, 0] < r).any() and (t[:, 0] <= -r).any() and (t[:, 0] > -r).any()
            ix = np.floor(np.float32(100) * (t[:, 0] + r))
            inside = (np.abs(t[:, 0]) < r) & (np.abs(t[:, 1]) < r)
            assert (ix[inside] >= G).any() == clamping_grid(G)
            if len(cat["overflow_to_inf"]):
                tz = np.concatenate([transform32(M, cat["overflow_to_inf"]) for M in Ms])
                assert np.isposinf(tz[:, 2]).any()
            if len(cat["z_minus_one"]):
                assert (transform32(Ms[0], cat["z_minus_one"])[:, 2] == -1).any() or len(Ms) > 1
        assert reached == set(CATALOGUE), (G, set(CATALOGUE) - reached)


def host_transform(hg, av, roll, step):
    return hg.build_transform(hg.make_request(approach=av), roll, step)


# ---- GPU ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def model(tmp_models):
    return tmp_models(64, seed=11)


@pytest.fixture(scope="module")
def orc(oracle_lib, model):
    return oracle_lib.Oracle(FEATURES, RANGE, model)


def _requests(hg, case):
    rq = []
    for k, a in enumerate(case["req"]):
        b, l = (case.get("ranges") or [(0, 0)] * len(case["req"]))[k]
        rq.append(dict(approach=APPROACHES[a], roll_begin=b, roll_limit=l))
    return rq


def _active(R, begin, limit):
    n = min(R, limit) if limit > 0 else R
    return range(max(0, min(begin, n)), n)


def build_batch(hg, case, sm):
    """packed clouds of the case: base points, with catalogue points at the catalogue's grid sides"""
    G, R = case["G"], 190 // case["step"]
    sizes = case["sizes"](sm)
    rqs = _requests(hg, case)
    Ms = [host_transform(hg, q["approach"], roll, case["step"]) for q in rqs for roll in range(R)]
    extra = None
    if case.get("cat"):
        cat = catalogue(Ms, G, 1234)
        extra = np.concatenate([cat[k] for k in NONFINITE + FINITE])
    clouds = []
    for c, n in enumerate(sizes):
        pts = base_cloud(1000 + c, n, G)
        if extra is not None and n >= 2000:   # replace points, so that sizes (and the plan) stay
            k = min(len(extra), n // 2)
            pts[-k:] = np.roll(extra, c * 997, axis=0)[:k]
        clouds.append(pts)
    return sizes, rqs, clouds


def check_front(gpu, orc, case, sizes, rqs, clouds, res):
    """heights, integral images, masks, windows, window counts and the clamp count of the last call against the oracle"""
    G, R, step = case["G"], 190 // case["step"], case["step"]
    nreq = len(rqs)
    U = len(sizes) * nreq * R
    M, _, _ = gpu.debug_unit_params(U, poses=False)
    heights = gpu.debug_heights(U)
    integral = gpu.debug_integral(U)
    win = gpu.debug_windows()
    clamped = 0
    for c in range(len(sizes)):
        for k, q in enumerate(rqs):
            j = c * nreq + k
            nwin = 0
            for roll in _active(R, q["roll_begin"], q["roll_limit"]):
                u = j * R + roll
                h, _, cl = orc.generate_grid(clouds[c], M[u], G, want_cells=True)
                clamped += cl
                assert np.array_equal(heights[u], h), (case["name"], c, k, roll, int((heights[u] != h).sum()))
                I = orc.calc_intimage(h)
                assert integral[u].tobytes() == I.tobytes(), (case["name"], c, k, roll)
                mask = orc.pnt_in_box(I, roll, (32, 44), step)
                cells = np.sort(win[win[:, 0] == u, 1])
                assert np.array_equal(cells, np.flatnonzero(mask.ravel())), (case["name"], c, k, roll)
                nwin += len(cells)
            assert res["best_per_request"][j].n_windows_scored == nwin, (case["name"], c, k)
    assert gpu.timing().n_clamped == clamped, (gpu.timing().n_clamped, clamped)
    return clamped


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_front_half_shapes(hg, orc, model, case):
    import torch
    gpu = hg.GraspSearch(FEATURES, RANGE, model, grid=case["G"], roll_step_deg=case["step"], bin_variant=case.get("bin_variant", 0))
    try:
        sm = gpu.info.sm_count
        sizes, rqs, clouds = build_batch(hg, case, sm)
        R = 190 // case["step"]
        want = plan(case["G"], sizes, [R * len(rqs)] * len(sizes), sm, bin_variant=case.get("bin_variant", 0))
        assert want[0] == case["kernel"], (want, "the case no longer reaches its kernel at %d SMs" % sm)
        off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        xyz = torch.from_numpy(np.concatenate(clouds) if sum(sizes) else np.zeros((0, 3), np.float32)).cuda()
        reqs = hg.make_requests(n=len(sizes) * len(rqs), approaches=[q["approach"] for q in rqs] * len(sizes),
                                roll_begin=[q["roll_begin"] for q in rqs] * len(sizes), roll_limit=[q["roll_limit"] for q in rqs] * len(sizes))
        ro = np.arange(len(sizes) + 1) * len(rqs)
        gpu.set_debug(True)
        res = gpu.search_batch_requests(xyz, off, reqs, ro, grasps=False)
        rec = gpu.debug_chunk_copy_waits()
        assert len(rec) == 1 and tuple(rec[0, 5:]) == want, (rec, want)
        n = check_front(gpu, orc, case, sizes, rqs, clouds, res)
        print("%s: plan %s, %d clamped points" % (case["name"], want, n))
    finally:
        gpu.close()


# ---- the catalogue through the whole search ---------------------------------------------------------------------------------
# what each catalogue cloud gets, per svm_mode: "equal" (the oracle's answer, grasp record bit for bit) or "unsupported"
# (HAF_ERR_UNSUPPORTED with a message).  The overflow cloud has one infinite height, so an integral image that is infinite
# below and right of that cell and fewer valid windows; every tier returns the oracle's answer for it, as for the others.
PINS = {(c, m): "equal" for c in ("finite", "nonfinite", "overflow") for m in ("tensor", "fp32", "fp64")}
MODES = {"tensor": 0, "fp64": 1, "fp32": 2}


def catalogue_clouds(hg, G, av, step):
    R = 190 // step
    cat = catalogue([host_transform(hg, av, roll, step) for roll in range(R)], G, 77)
    base = base_cloud(5, 20000, G)
    out = {"finite": np.concatenate([base] + [cat[k] for k in FINITE]),
           "nonfinite": np.concatenate([base] + [cat[k] for k in NONFINITE])}
    if len(cat["overflow_to_inf"]):
        out["overflow"] = np.concatenate([base, cat["overflow_to_inf"]])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
def test_catalogue_full_search(hg, oracle_lib, orc, model, mode):
    """every catalogue cloud, as a single goal and in a batch, at G = 56 and at the clamping G = 64, with the default and a
    tilted approach vector: the oracle's answer (best, windows, grasp record bit for bit) or HAF_ERR_UNSUPPORTED, as pinned"""
    step = 45
    for G in (56, 64):
        gpu = hg.GraspSearch(FEATURES, RANGE, model, grid=G, roll_step_deg=step, svm_mode=MODES[mode])
        try:
            for av in (APPROACHES[0], APPROACHES[1]):
                clouds = catalogue_clouds(hg, G, av, step)
                assert set(clouds) == ({"finite", "nonfinite", "overflow"} if av != APPROACHES[0] else {"finite", "nonfinite"})
                singles = {}
                for name, xyz in clouds.items():
                    grq, orq = hg.make_request(approach=av), oracle_lib.make_request(approach=av)
                    try:
                        gres = gpu.search_grasps(xyz, [grq], outputs=True)
                        got = "equal"
                    except hg.HafError as e:
                        assert e.code == -5 and str(e).strip(), e
                        got = "unsupported"
                    assert got == PINS[(name, mode)], (G, av, name, mode, got)
                    if got != "equal":
                        continue
                    ores = orc.search(xyz, orq, G=G, roll_step_deg=step)
                    assert np.isposinf(gres["heights"]).any() == (name == "overflow")
                    print("catalogue %s G=%d av=%s %s: best %s, %d windows" % (mode, G, av, name, gres["best"].astuple(), gres["best"].n_windows_scored))
                    ob, gb = ores["best"], gres["best"]
                    assert gb.astuple() == ob.astuple() and gb.n_windows_scored == ob.n_windows, (G, av, name, gb.astuple(), ob.astuple())
                    R = ob.rolls_done
                    assert np.array_equal(gres["heights"][0][:R], ores["heights"][:R]) and np.array_equal(gres["mask"][0][:R], ores["mask"][:R])
                    if ob.roll >= 0:
                        gp = orc.transform_gp_in_wcs(orq, ores["heights"][ob.roll], ob.row, ob.col, ob.roll, step)
                        assert gres["grasp"].as_array().tobytes() == gp.tobytes(), (G, av, name)
                    singles[name] = (gb.astuple(), gb.n_windows_scored)
                names = list(clouds)
                off = np.concatenate([[0], np.cumsum([len(clouds[k]) for k in names])])
                xyz = np.concatenate([clouds[k] for k in names])
                if all(k in singles for k in names):
                    best = gpu.search_batch_packed(xyz, off, hg.make_request(approach=av))
                    assert [(b.astuple(), b.n_windows_scored) for b in best] == [singles[k] for k in names]
                else:
                    with pytest.raises(hg.HafError) as e:
                        gpu.search_batch_packed(xyz, off, hg.make_request(approach=av))
                    assert e.value.code == -5
        finally:
            gpu.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [12, 16, 20])
def test_single_goal_strides_with_catalogue(hg, orc, model, stride):
    """single goals read points at a pitch of 12, 16 or 20 bytes (scalar loads at an odd pitch); heights and the clamp count
    at the clamping G = 64 equal the oracle's, with the catalogue mixed in"""
    G, step = 64, 45
    gpu = hg.GraspSearch(FEATURES, RANGE, model, grid=G, roll_step_deg=step)
    try:
        for av in (APPROACHES[0], APPROACHES[1]):
            xyz = np.concatenate([v for k, v in catalogue_clouds(hg, G, av, step).items() if k != "overflow"])
            padded = np.full((len(xyz), stride // 4), 7.0, np.float32)
            padded[:, :3] = xyz
            res = gpu.search(padded, [hg.make_request(approach=av)])
            assert res["best"].rolls_done == 190 // step
            clamped = 0
            for roll in range(190 // step):
                h, _, cl = orc.generate_grid(xyz, host_transform(hg, av, roll, step), G, want_cells=True)
                clamped += cl
                assert np.array_equal(res["heights"][0][roll], h), (stride, av, roll)
            assert gpu.timing().n_clamped == clamped > 0
    finally:
        gpu.close()


@pytest.mark.gpu
def test_staged_batch_mixes_binning_kernels(hg, model, monkeypatch):
    """a host-staged batch whose first chunk is under the SM threshold (point-parallel) and whose second is not (whole-cloud
    kernel): the chunk records name both, and the answers and the clamp count equal the one-pass device-resident run, from
    pinned and from pageable memory"""
    import torch
    G, step = 64, 45
    gpu = hg.GraspSearch(FEATURES, RANGE, model, grid=G, roll_step_deg=step)
    try:
        sm = gpu.info.sm_count
        n1, n2 = _nwc(sm) - 1, _nwc(sm) + 5
        cat = catalogue([host_transform(hg, APPROACHES[1], roll, step) for roll in range(190 // step)], G, 77)
        extra = np.concatenate([cat[k] for k in NONFINITE + FINITE])
        clouds = []
        for c in range(n1 + n2):
            pts = base_cloud(300 + c, 8 * G * G + 3 * c, G)
            pts[-len(extra):] = extra
            clouds.append(pts)
        off = np.concatenate([[0], np.cumsum([len(c) for c in clouds])])
        xyz = np.concatenate(clouds)
        rq = hg.make_request(approach=APPROACHES[1])
        ref = gpu.search_batch_packed(torch.from_numpy(xyz).cuda(), off, rq)
        t_ref = gpu.timing()
        assert t_ref.n_chunks == 1 and t_ref.n_clamped > 0
        assert gpu.debug_chunk_copy_waits()[0, 5] == 1
        want = [(b.astuple(), b.n_windows_scored) for b in ref]
        monkeypatch.setenv("HAF_STAGE_SCHED", "%d,%d" % (n1, n2))
        for src in (torch.from_numpy(xyz).pin_memory(), xyz):
            got = gpu.search_batch_packed(src, off, rq)
            rec = gpu.debug_chunk_copy_waits()
            assert [tuple(r[:2]) for r in rec] == [(0, n1), (n1, n1 + n2)]
            assert tuple(rec[0, 5:]) == plan(G, [len(c) for c in clouds[:n1]], [190 // step] * n1, sm)
            assert tuple(rec[1, 5:]) == plan(G, [len(c) for c in clouds[n1:]], [190 // step] * n2, sm)
            assert rec[0, 5] == 0 and rec[1, 5] == 1
            assert [(b.astuple(), b.n_windows_scored) for b in got] == want
            assert gpu.timing().n_clamped == t_ref.n_clamped and gpu.timing().n_windows == t_ref.n_windows
    finally:
        gpu.close()


# ---- feature staging of the tensor path ---------------------------------------------------------------------------------------
def cta_paths(win, G):
    """(path, stride class) of every features_tc_kernel CTA, from the window list in device order (kernels.cuh: 64 windows
    per CTA; staged as one unit, as two units, or read from global memory when they span three units or more than 36 rows)"""
    ld = G + 1
    out = []
    for w0 in range(0, len(win), FT_NW):
        blk = win[w0:w0 + FT_NW]
        u, cell = blk[:, 0], blk[:, 1]
        row, col = cell // G, cell % G
        uA, uB = u[0], u[-1]
        two = bool(np.all((u == uA) | (u == uB)))
        a = u == uA
        nA = row[a].max() - row[a].min() + 15
        nB = (row[~a].max() - row[~a].min() + 15) if uB != uA else 0
        ok = two and nA + nB <= FT_ROWS
        o = ld
        for t in range(0, len(blk), 32):   # the first row break of the first 32-lane group that has one
            lanes = range(t + 1, min(t + 32, len(blk)))
            brk = [i for i in lanes if u[i] == u[i - 1] and row[i] == row[i - 1] + 1]
            if brk:
                o = col[brk[0] - 1] + 1 - col[brk[0]]
                break
        path = ("two" if uB != uA else "one") if ok else ("three_units" if not two else "rows")
        out.append((path, (o - ld) % 32 if ok else 0))
    return out


@pytest.mark.gpu
def test_tensor_feature_staging_paths(hg, oracle_lib, orc, model):
    """the tensor path's operands (debug_tensor_inputs) against the exact scaled values per window, with mask shapes that put
    CTAs on every staging path: one unit, two units, three or more units (tiny areas) and more than 36 rows (tall, narrow
    areas), rotated at 15 and 45 degree steps; the exact values against the oracle on the first units"""
    paths, classes = set(), set()
    for G, step, areas in ((56, 15, [(32, 44), (14.9, 20), (16, 16), (60, 15)]), (100, 45, [(32, 44), (60, 15), (16, 16)]),
                           (158, 45, [(16, 16), (60, 15)]), (192, 45, [(32, 44), (60, 15)])):
        gpu = hg.GraspSearch(FEATURES, RANGE, model, grid=G, roll_step_deg=step)
        try:
            xyz = base_cloud(9, 12 * G * G, G)
            gpu.search(xyz, [hg.make_request(area=a) for a in areas], outputs=False)
            win = gpu.debug_windows()
            x = gpu.debug_tensor_inputs().astype(np.float64)
            raw, scaled = gpu.debug_features()
            err = np.abs(x - scaled)
            bad = err > FAST_TIER_REL * np.abs(scaled) + FAST_TIER_ABS
            assert not bad.any(), (G, int(bad.sum()), float(err.max()))
            cp = cta_paths(win, G)
            paths |= {p for p, _ in cp}
            classes |= {c for p, c in cp if p in ("one", "two")}
            # the exact tier against the oracle: the first request's first two rolls
            R = 190 // step
            integral = gpu.debug_integral(len(areas) * R)
            for roll in range(2):
                mask = orc.pnt_in_box(integral[roll], roll, (int(areas[0][0]), int(areas[0][1])), step)
                feats, rc = orc.calc_featurevectors(integral[roll], mask)
                sel = np.flatnonzero(win[:, 0] == roll)
                sel = sel[np.argsort(win[sel, 1])]
                assert np.array_equal(win[sel, 1], rc[:, 0] * G + rc[:, 1])
                assert raw[sel].tobytes() == feats.tobytes()
                assert scaled[sel].tobytes() == orc.scale(feats)[:, :gpu.D].tobytes()
        finally:
            gpu.close()
    print("staging paths %s, stride classes reached %s" % (sorted(paths), sorted(int(c) for c in classes)))
    assert paths == {"one", "two", "three_units", "rows"}, paths
    assert len(classes) >= 8, sorted(classes)


# ---- full searches at new grid sides ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("G", [16, 58, 130, 160, 226, 228])
def test_full_search_at_new_grid_sides(hg, oracle_lib, model, G):
    """heights, masks, integral images, windows, raw and scaled features, decisions, tops and best against the oracle in the
    default tensor mode (test_gpu_parity.check_search) on a synthetic cloud scaled to the grid"""
    from haf_grasping_b200 import synth
    from test_gpu_parity import Pair, check_search
    p = Pair(hg, oracle_lib, model, grid=G, roll_step_deg=90, roll_max_deg=190)
    try:
        xyz = synth.synth_cloud(31 + G, max(20000, 4 * G * G), r=0.98 * G / 200.0)
        check_search(p, xyz, hg, oracle_lib, model, area=(32.0, 44.0) if G < 100 else (60.0, 52.0))
    finally:
        p.close()
