"""The SVM contraction at every operand shape its kernels branch on, through the libsvm front end (SvmPredictor /
haf_svm_create_config), against a float64 restatement of the decision function; and the search path at feature counts
other than 323.

The tensor kernels (svm_tc.cuh) branch on the operand width -- Krow = round_up(Dsv + 6, 16) columns in KB k-blocks of 64,
the last one carrying last_slices 16-wide slices, the X tile resident only up to XK_MAX k-blocks, the six extra columns
where they fall -- on the support-vector tiles of 256 (sorted by the sign of coef, each sign group padded: one tile, odd
counts, an empty group, the coef table in global memory past TAB_SMEM_MAX), and on the rows (partial 128 / 256-row tiles
and the split of the SV tiles per work item, nsplit2, which can leave a work item an empty or a negative range).  The SIMT
kernel pads to Kpad / Spad, the FP64 DMMA guard tier to Dsv16, and the exact-order kernels stage the inputs of 8 windows in
shared memory.  CASES below covers each of those values; test_cases_cover_every_branch asserts that it does (on any
machine), and each GPU case asserts that the kernel and split the library reports (haf_info.reserved[2] / [3]) are the
ones the case was chosen for.

Reference: decision values sum_i coef_i exp(-gamma |x - sv_i|^2) - rho in float64 numpy; labels from that sign wherever
|dec| >= 1e-9 E, from libsvm's own summation order (the oracle's svm.cpp restatement) on the rows closer to 0.
"""
import math
import os
import re

import numpy as np
import pytest

from conftest import FEATURES, RANGE, ROOT
from model_io import check_decision_tolerance, coefK_sum, load_model_arrays

CSRC = os.path.join(ROOT, "haf_grasping_b200", "csrc")


def _const(fname, name):
    src = open(os.path.join(CSRC, fname)).read()
    m = re.search(r"(?:constexpr int %s\s*=|#define %s)\s*(\d+)" % (name, name), src)
    return int(m.group(1))


BK, BN, BM, NAUG = (_const("svm_tc.cuh", n) for n in ("BK", "BN", "BM", "NAUG"))
XK_MAX, TAB_SMEM_MAX = _const("svm_tc.cuh", "XK_MAX"), _const("svm_tc.cuh", "TAB_SMEM_MAX")
SVM_BK, SVM_BN, EXACT_WB = _const("kernels.cuh", "SVM_BK"), _const("kernels.cuh", "SVM_BN"), _const("kernels.cuh", "HAF_EXACT_WB")
B200_SMS = 148
SMEM_OPTIN = 227 * 1024      # opt-in shared memory per block of sm_100
MID_ROWS = B200_SMS // 2 * 2 * BM    # from here on a launch fills the GPU without splitting the SV tiles ("mid-sized" branch)
KERNEL_NAMES = {0: "FP64 exact", 1: "tc3", 2: "tc2", 3: "SIMT"}


def ru(a, b):
    return (a + b - 1) // b * b


def geometry(dsv, n_pos, n_neg):
    krow = ru(dsv + NAUG, 16)
    kb = -(-krow // BK)
    spadT = max(ru(n_pos, BN) + ru(n_neg, BN), BN)
    return dict(Krow=krow, KB=kb, last_slices=(krow - BK * (kb - 1)) // 16, Kpad=ru(dsv, SVM_BK), Dsv16=ru(dsv, 16),
                SpadT=spadT, n_ntiles=spadT // BN, Spad=ru(n_pos + n_neg, SVM_BN),
                aug_straddles=dsv // BK != (dsv + NAUG - 1) // BK, exact_smem=EXACT_WB * dsv * 8)


def nsplit2(rows, n_ntiles, sms):
    """the split of the SV tiles per work item that svm_stage (hafgpu.cu) picks for one pass over `rows` rows"""
    pairs = ru(rows, 2 * BM) // (2 * BM)
    if pairs < sms // 2:
        return min(n_ntiles, -(-sms // pairs))
    best, pick, ns = 0.0, 1, 1
    while ns <= n_ntiles and ns <= 8:
        if n_ntiles % ns == 0:
            rounds = pairs * ns / (sms // 2)
            eff = rounds / math.ceil(rounds)
            if eff > best + 0.02:
                best, pick = eff, ns
        ns *= 2
    return pick


def split_regime(rows, n_ntiles, sms):
    """'mid' (the launch fills the GPU), 'negative' (some work item starts past the last tile), 'empty' (one starts at it), else 'plain'"""
    if ru(rows, 2 * BM) // (2 * BM) >= sms // 2:
        return "mid"
    ns = nsplit2(rows, n_ntiles, sms)
    per = -(-n_ntiles // ns)
    starts = [sp * per for sp in range(ns)]
    if any(s > n_ntiles for s in starts):
        return "negative"
    if any(s == n_ntiles for s in starts):
        return "empty"
    return "plain"


def rows_for(regime, n_ntiles, sms):
    """a row count (with a partial last 256-row tile) that puts the launch in `regime`"""
    if regime == "mid":
        return (sms // 2) * 2 * BM + 3 * BM + 37
    for pairs in range(1, sms // 2):
        if split_regime(pairs * 2 * BM - 37, n_ntiles, sms) == regime:
            return pairs * 2 * BM - 37
    raise AssertionError("no row count gives a %s split for %d tiles on %d SMs" % (regime, n_ntiles, sms))


# (Dsv, (n_pos, n_neg), rows or split regime, probability run).  Each axis value of the issue at every mode; the risky
# ones paired (tail slices x odd KB x odd tile count x partial row tile); the heavy corners (Dsv 1000 / 1700 / 3700,
# 4200 SVs, the mid-sized launch) once each.
CASES = [
    (1, (1, 0), 1, False),
    (26, (0, 1), 2, False),
    (42, (256, 0), 127, False),
    (58, (257, 0), 128, True),
    (59, (255, 1), 129, False),
    (90, (300, 100), 255, False),
    (122, (1024, 768), 257, False),
    (123, (300, 100), 513, False),
    (323, (1024, 768), 129, True),
    (346, (255, 1), 255, False),
    (442, (1024, 768), 127, False),
    (506, (300, 100), 257, False),
    (507, (1024, 768), 129, False),
    (58, (1024, 1024), "empty", False),
    (90, (1024, 1024), "negative", False),
    (26, (300, 100), "mid", False),
    (122, (2100, 2100), 513, False),
    (1000, (257, 0), 129, False),
    (1700, (300, 100), 129, True),
    (3700, (255, 1), 33, True),       # the exact-order kernel's inputs of 8 windows exceed the opt-in shared memory
]
SMALL_W = (1, 2, 127, 128, 129, 255, 257, 513)


def _case_id(c):
    return "D%d-S%d+%d-W%s%s" % (c[0], c[1][0], c[1][1], c[2], "-prob" if c[3] else "")


def test_cases_cover_every_branch():
    """the sweep reaches every value the kernels branch on (worked out for a 148-SM B200; the GPU cases re-check the split
    regimes against the device they run on)"""
    geo = [geometry(d, p, n) for d, (p, n), _, _ in CASES]
    dsvs = {c[0] for c in CASES}
    assert dsvs >= {1, 26, 42, 58, 59, 90, 122, 123, 323, 346, 442, 506, 507, 1000, 1700}
    assert {g["last_slices"] for g in geo} == {1, 2, 3, 4}
    assert any(g["KB"] == 1 for g in geo)
    assert {g["KB"] for g in geo} >= {3, 7, 9, XK_MAX, XK_MAX + 1}
    assert any(g["aug_straddles"] for g in geo)
    assert any(g["Kpad"] != d for g, (d, *_) in zip(geo, CASES)) and any(g["Dsv16"] != d for g, (d, *_) in zip(geo, CASES))
    assert any(EXACT_WB * d * 8 > 100 * 1024 for d in dsvs)           # past the exact kernel's former 100 KB
    assert any(EXACT_WB * d * 8 > SMEM_OPTIN for d in dsvs)            # past the opt-in maximum: inputs read in place
    svs = {c[1] for c in CASES}
    assert svs >= {(1, 0), (0, 1), (256, 0), (257, 0), (255, 1), (300, 100), (1024, 768), (1024, 1024), (2100, 2100)}
    tiles = {g["n_ntiles"] for g in geo}
    assert 1 in tiles and 3 in tiles and 7 in tiles
    assert any(g["SpadT"] > TAB_SMEM_MAX for g in geo)
    assert any(g["Spad"] % SVM_BN == 0 and (p + n) % SVM_BN for g, (_, (p, n), _, _) in zip(geo, CASES))
    ws = {c[2] for c in CASES}
    assert ws >= set(SMALL_W) | {"empty", "negative", "mid"}
    for (d, (p, n), w, _), g in zip(CASES, geo):
        if not isinstance(w, int):
            rows = rows_for(w, g["n_ntiles"], B200_SMS)
            assert split_regime(rows, g["n_ntiles"], B200_SMS) == w
            assert rows % (2 * BM) != 0 and (w != "mid" or rows > MID_ROWS)
    # risky pairs: a tail of several slices with odd KB / odd tile counts / partial row tiles in one case
    assert any(g["KB"] % 2 == 1 and g["n_ntiles"] % 2 == 1 and isinstance(w, int) and w % BM
               for g, (_, _, w, _) in zip(geo, CASES))
    assert any(g["last_slices"] > 1 and g["n_ntiles"] % 2 == 1 and isinstance(w, int) and w % BM
               for g, (_, _, w, _) in zip(geo, CASES))


# ---------------------------------------------------------------------------------------------------------------- fixtures
def write_model(path, n_pos, n_neg, dims, gamma, rho, density, seed, prob=False):
    """a 2-class RBF C-SVC model in libsvm 3.12's text format with n_pos positive and n_neg negative coefficients (in that
    order, as libsvm stores the two classes); the last dimension is present in the first SV so that the model is `dims` wide"""
    rng = np.random.default_rng(seed)
    S = n_pos + n_neg
    sv = rng.uniform(-1.0, 1.0, (S, dims)) * (rng.random((S, dims)) < density)
    sv[0, dims - 1] = 0.5
    coef = rng.uniform(0.05, 1.0, S)
    coef[n_pos:] *= -1.0
    with open(path, "w") as fh:
        fh.write("svm_type c_svc\nkernel_type rbf\ngamma %.17g\nnr_class 2\ntotal_sv %d\nrho %.17g\nlabel 1 -1\n" % (gamma, S, rho))
        if prob:
            fh.write("probA -1.7\nprobB 0.2\n")
        fh.write("nr_sv %d %d\nSV\n" % (n_pos, n_neg))
        for i in range(S):
            fh.write("%.17g " % coef[i] + " ".join("%d:%.17g" % (d + 1, sv[i, d]) for d in np.nonzero(sv[i])[0]) + " \n")
    return path


def make_rows(model, W, dsv, density, seed):
    """W rows of width dsv (wider than the model where dsv > its width): first an SV itself (d^2 = 0: the tensor path's
    worst cancellation), the all-zero row, a row far from every SV (E below the FP32 range floor: FP64), a row with one
    value beyond the fp16 range (the exact path), then rows near an SV and uniform rows"""
    rng = np.random.default_rng(seed)
    sv = model["sv"]
    x = rng.uniform(-1.0, 1.0, (W, dsv)) * (rng.random((W, dsv)) < density)
    near = rng.random(W) < 0.5
    j = rng.integers(0, len(sv), W)
    x[near, :sv.shape[1]] = sv[j[near]] + rng.normal(0.0, 0.15, (int(near.sum()), sv.shape[1])) * (sv[j[near]] != 0)
    special = [np.pad(sv[0], (0, dsv - sv.shape[1])), np.zeros(dsv), np.full(dsv, 7.0), x[min(3, W - 1)].copy()]
    special[3][0] = 1.0e5
    for k, r in enumerate(special[:W]):
        x[k] = r
    return x


def reference(model, x):
    """float64 decision values, sum|coef|K and E per row"""
    sv, coef, g = model["sv"], model["coef"], model["gamma"]
    D = max(sv.shape[1], x.shape[1])
    svp = np.zeros((len(sv), D)); svp[:, :sv.shape[1]] = sv
    xp = np.zeros((len(x), D)); xp[:, :x.shape[1]] = x
    sn = (svp ** 2).sum(1)
    dec = np.zeros(len(x))
    for b in range(0, len(x), 2048):
        xb = xp[b:b + 2048]
        d2 = np.maximum((xb ** 2).sum(1)[:, None] + sn[None, :] - 2.0 * (xb @ svp.T), 0.0)
        dec[b:b + 2048] = np.exp(-g * d2) @ coef - model["rho"]
    plain, E = coefK_sum(model, x, with_E=True)
    return dec, plain, E


@pytest.fixture(scope="module")
def sms():
    """SMs of the device (each case checks it against haf_info.sm_count): the split regimes depend on it"""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _labels_reference(oracle_lib, model_path, model, x, dec, E):
    """libsvm's labels: the float64 sign where |dec| >= 1e-9 E, libsvm's own order (oracle) on the rows closer to 0"""
    lab = np.where(dec > 0, 1, -1)
    close = np.nonzero(np.abs(dec) < 1e-9 * E)[0]
    if len(close):
        o = oracle_lib.Oracle(FEATURES, RANGE, model_path)
        _, olab = o.svm_decision(x[close])
        lab[close] = olab
    return lab, len(close)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_svm_contraction_shapes(hg, oracle_lib, tmp_path, sms, case):
    dsv, (n_pos, n_neg), w, prob = case
    geo = geometry(dsv, n_pos, n_neg)
    W = w if isinstance(w, int) else rows_for(w, geo["n_ntiles"], sms)
    dims = dsv if dsv < 3 else dsv - 2                       # rows are 2 dimensions wider than the model (min_dims)
    density = 1.0 if dsv <= 128 else 0.5
    gamma = 2.0 / dsv
    path = str(tmp_path / "m.model")
    rng_seed = 1000 * dsv + n_pos + 7 * n_neg
    write_model(path, n_pos, n_neg, dims, gamma, 0.0, density, rng_seed, prob)
    model = load_model_arrays(path)
    x = make_rows(model, W, dsv, density, rng_seed + 1)
    # rho halfway between the two middle decision sums: both labels occur, many rows sit near 0, none at the rounding level
    dec0, _, _ = reference(model, x)
    s = np.sort(dec0)
    rho = float(0.5 * (s[len(s) // 2 - 1] + s[len(s) // 2])) if len(s) > 1 else 0.5 * float(s[0])
    write_model(path, n_pos, n_neg, dims, gamma, rho, density, rng_seed, prob)
    model = load_model_arrays(path)
    assert model["sv"].shape[1] == dims and model["rho"] == rho
    dec_ref, plain, E = reference(model, x)
    lab_ref, n_close = _labels_reference(oracle_lib, path, model, x, dec_ref, E)

    def run(**kw):
        p = hg.SvmPredictor(path, min_dims=dsv, **kw)
        try:
            lab, dec = p.predict(x)
            t = p.timing()
            info = p.info
            assert t.n_windows == W and info.sm_count == sms
            assert lab.astype(int).tolist() == lab_ref.tolist(), ("labels", kw, np.nonzero(lab.astype(int) != lab_ref)[0][:10])
            return dec, t, [info.reserved[k] for k in range(4)]
        finally:
            p.close()

    seen = set()
    report = []
    # calibrated tensor path and FP32 SIMT: the product tolerance
    for mode in (0, 2):
        dec, t, res = run(svm_mode=mode)
        check_decision_tolerance(model, x, dec, dec_ref)
        if mode == 2:
            assert res[2] == 3 and res[3] == 0
        else:
            seen.add(res[2])
            assert res[3] == nsplit2(W, geo["n_ntiles"], sms)
            report.append(("calibrated", t.tc_passes, t.escalations, KERNEL_NAMES[res[2]]))
    # forced products, both kernels, both coef-table places: within the context's own guard band
    for passes in (1, 2, 3):
        for variant in (0, 2):
            for table in (0, 1):
                dec, t, res = run(svm_mode=0, tc_passes=passes, tc_variant=variant, sv_table_global=table)
                band = res[1] * 1e-9 * (E + abs(rho))
                err = np.abs(dec - dec_ref)
                assert (err <= band).all(), ("forced products", passes, variant, table, float((err / (E + abs(rho))).max()), res[1])
                assert t.tc_passes >= passes
                assert res[3] == nsplit2(W, geo["n_ntiles"], sms)
                resident = t.tc_passes == 1 and variant == 0 and geo["KB"] <= XK_MAX
                assert res[2] == (1 if resident else 2), (passes, variant, table, res, t.tc_passes)
                seen.add(res[2])
                report.append((passes, variant, table, t.tc_passes, t.escalations, KERNEL_NAMES[res[2]]))
    if geo["KB"] <= XK_MAX:
        assert seen == {1, 2}, seen
    else:
        assert seen == {2}, seen
    if not isinstance(w, int):
        assert split_regime(W, geo["n_ntiles"], sms) == w
    # FP64 exact order
    dec, t, res = run(svm_mode=1)
    assert res[2] == 0
    assert (np.abs(dec - dec_ref) <= 1e-13 * plain + 1e-300).all(), float((np.abs(dec - dec_ref) / np.maximum(plain, 1e-300)).max())
    # every row through the FP64 guard tier 2: DMMA, and DFMA where its register tiles hold the model
    dfma_fits = (dsv * 16 + 16 + 8 * 16 * 2) * 8 <= 100 * 1024
    for gk in ((1, 2) if dfma_fits else (1,)):
        dec, t, res = run(svm_mode=0, guard_rel=1e6, guard_kernel=gk)
        assert t.n_guard == W
        assert (np.abs(dec - dec_ref) <= 1e-12 * plain + 1e-300).all(), ("tier 2", gk, float((np.abs(dec - dec_ref) / np.maximum(plain, 1e-300)).max()))
    if prob:
        p = hg.SvmPredictor(path, min_dims=dsv)
        try:
            lab, pr = p.predict_probability(x)
            assert p.timing().n_windows == W and p.info.reserved[2] == 0
        finally:
            p.close()
        o = oracle_lib.Oracle(FEATURES, RANGE, path)
        olab, opr = o.svm_predict_probability(x)
        assert np.array_equal(lab, olab)
        assert np.abs(pr - opr).max() <= 1e-10
    print(_case_id(case), "W", W, "near-zero rows", n_close, report)


# ---------------------------------------------------------------------------------------------------------------- search path
def _feature_files(tmp_path, D):
    """the first D lines of the bundled feature and range files; past 323, copies of the existing lines under new indices"""
    flines = [ln for ln in open(FEATURES).read().split("\n") if ln.strip()]
    rlines = open(RANGE).read().split("\n")
    head, rl = rlines[:2], [ln for ln in rlines[2:] if ln.strip()]
    fo = [flines[i % len(flines)] for i in range(D)]
    ro = []
    for i in range(D):
        _, lo, hi = rl[i % len(rl)].split()
        ro.append("%d %s %s" % (i + 1, lo, hi))
    fp, rp = str(tmp_path / ("features_%d.txt" % D)), str(tmp_path / ("range_%d" % D))
    open(fp, "w").write("\n".join(fo) + "\n\n")
    open(rp, "w").write("\n".join(head + ro) + "\n")
    return fp, rp


class _Pair:
    def __init__(self, hg, orc, features, range_path, model, nshaf=302, **kw):
        self.gpu = hg.GraspSearch(features, range_path, model, nr_features_without_shaf=nshaf, **kw)
        self.orc = orc.Oracle(features, range_path, model, nr_features_without_shaf=nshaf)
        self.G, self.step, self.rmax = 56, 15, 190

    def close(self):
        self.gpu.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D,mode,nshaf", [(58, 0, 302), (122, 0, 302), (127, 0, 302), (128, 0, 302), (129, 0, 302), (129, 2, 302),
                                          (200, 0, 150), (442, 0, 302), (507, 0, 302), (507, 2, 302)])
def test_search_at_other_feature_counts(hg, oracle_lib, tmp_path, D, mode, nshaf):
    """features_tc_kernel's 128-dimension passes and guard_inputs_kernel at feature counts around a pass boundary and past
    323: features, scaled inputs, graspseval, tops and the best grasp bit-exact, decision values within the product
    tolerance, labels identical"""
    from haf_grasping_b200 import synth
    from test_gpu_parity import check_search
    clouds = np.load(os.path.join(ROOT, "tests", "golden", "clouds.npz"))
    fp, rp = _feature_files(tmp_path, D)
    model = synth.write_synth_model(str(tmp_path / "m.model"), n_sv=300, dim=D, gamma=1.0 / D, seed=D)
    p = _Pair(hg, oracle_lib, fp, rp, model, nshaf=nshaf, svm_mode=mode)
    try:
        assert p.gpu.F == D + 1 and p.gpu.D <= D          # + the trailing blank line, as for the bundled file
        for name in ("pcd2", "table1"):
            gres, _, _ = check_search(p, clouds[name], hg, oracle_lib, model)
            assert gres["best"].n_windows_scored > 0
        import ctypes
        from haf_grasping_b200 import api
        info = api.haf_info()
        p.gpu.L.haf_get_info(p.gpu.h, ctypes.byref(info))
        resident = info.reserved[0] == 1 and geometry(D, 1, 1)["KB"] <= XK_MAX
        assert info.reserved[2] == (3 if mode == 2 else (1 if resident else 2))
    finally:
        p.close()
