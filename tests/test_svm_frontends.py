"""libsvm front ends (SURVEY 8f-3): svm-scale-b200 / svm-predict-b200 and the haf_svm_* / haf_scale_* C ABI they bind.

Parity here is pinned against the REFERENCE'S OWN PROGRAMS: oracle/_ref/svm-scale and oracle/_ref/svm-predict are
libsvm-3.12 compiled unmodified from the reference's sources; the GPU tests compare output files byte for byte.  Where
oracle/_ref is not built, the GPU tests compare with the restatements of tests/libsvm_programs.py instead, pinned first to
the committed outputs of those programs (tests/golden/svm_cli).
"""
import os
import subprocess

import numpy as np
import pytest

import libsvm_programs
from conftest import FEATURES, RANGE, ROOT

LIBDIR = os.path.join(ROOT, "haf_grasping_b200", "lib")
SVM_PREDICT = os.path.join(LIBDIR, "svm-predict-b200")
SVM_SCALE = os.path.join(LIBDIR, "svm-scale-b200")


@pytest.fixture(scope="module")
def tools():
    from haf_grasping_b200 import build
    if not (os.path.exists(SVM_PREDICT) and os.path.exists(SVM_SCALE)):
        build.build_svm_tools()
    return SVM_PREDICT, SVM_SCALE


# ---------------------------------------------------------------- CPU: host-side readers, loud failure without a GPU
def test_predict_reader_follows_svm_predicts_tokenisation(tools, tmp_path):
    f = tmp_path / "rows.txt"
    # blanks before an index, tab separators, a trailing blank before the newline (what svm-scale writes), no final newline
    f.write_text("+1 1:0.5  3:-2e-3\t7:1 \n-1 2:1e2 \n0\n1 4:4")
    out = subprocess.run([tools[0], "--parse-only", str(f)], capture_output=True, text=True, check=True).stdout.split()
    assert out[1] == "4" and out[3] == "5" and out[5] == "7" and out[7] == "0"
    assert float(out[9]) == 1 * 0.5 + 3 * -2e-3 + 7 * 1 + 2 * 1e2 + 4 * 4
    # what svm-predict.c:88-118 rejects: descending index, junk after a number, a value that sets errno (underflow), empty line
    for bad in ("1 3:1 2:1\n", "1 1:0.5x\n", "1 1:1e-400\n", "1 1:1\n\n1 2:2\n", "x 1:1\n"):
        f.write_text("1 1:1\n" + bad)
        out = subprocess.run([tools[0], "--parse-only", str(f)], capture_output=True, text=True, check=True).stdout.split()
        assert out[7] == ("3" if bad.startswith("1 1:1\n\n") else "2"), (bad, out)


def test_predict_reader_accepts_and_rejects_exactly_what_the_reference_program_does(tools, oracle_lib, tmp_models, tmp_path):
    """Fuzz: mutated rows go through the reference's own svm-predict (oracle/_ref, runs on the CPU) and through the B200
    front end's reader (--parse-only); the first rejected line ("Wrong input format at line N") must be the same."""
    _, ref_predict = _ref_bins(oracle_lib)
    rng = np.random.default_rng(2024)
    good = "1 1:0.5 2:-0.25 7:1e-3 12:3 40:-7.5e2 323:0.125"
    snippets = [";", ":", "::", " ", "  ", "\t", "x", "-", "+", "e", "E5", "nan", "inf", "-inf", "0x1p-3", "1e-400", "1e400", ".", "5.", "+.5",
                "99999999999999999999", "-3", "0", "7", "12:", ":3", "1 :2", "3: 4", "#", ",", "\r", "1e", "--1", "1:2:3", "٣"]
    model = tmp_models(256)
    checked = rejected = 0
    for trial in range(120):
        lines = []
        for k in range(4):
            ln = good
            if rng.random() < 0.22:
                for _ in range(int(rng.integers(1, 3))):
                    pos = int(rng.integers(0, len(ln) + 1))
                    snip = snippets[int(rng.integers(0, len(snippets)))]
                    ln = ln[:pos] + snip + ln[pos + (int(rng.integers(0, 3)) if rng.random() < 0.5 else 0):]
            lines.append(ln)
        src = tmp_path / ("fuzz_%d.txt" % trial)
        src.write_bytes(("\n".join(lines) + "\n").encode("utf-8"))
        a = subprocess.run([ref_predict, str(src), model, str(tmp_path / "ref.out")], capture_output=True)
        want = 0
        if a.returncode != 0:
            assert a.stderr.startswith(b"Wrong input format at line "), a.stderr
            want = int(a.stderr.split()[-1])
        out = subprocess.run([tools[0], "--parse-only", str(src)], capture_output=True, text=True, check=True).stdout.split()
        assert int(out[7]) == want, (trial, lines, a.stderr, out)
        checked += 1
        rejected += want > 0
    assert checked == 120 and 15 < rejected < 105     # the fuzz exercises both outcomes


def test_scale_reader_follows_svm_scales_sscanf_pairs(tools, tmp_path):
    f = tmp_path / "rows.txt"
    f.write_text("-1 1:0.5 2:3 10:1e-3\n+1  4: 2.5 junk 6:1\n3\n")   # "%d:%lf" skips blanks before the value; a row ends at junk
    out = subprocess.run([tools[1], "--parse-only", str(f)], capture_output=True, text=True, check=True).stdout.split()
    assert out[1] == "3" and out[3] == "4" and out[5] == "10"
    assert float(out[7]) == 1 * 0.5 + 2 * 3 + 10 * 1e-3 + 4 * 2.5


def test_front_ends_fail_loudly_without_a_gpu(tools, tmp_models, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    f = tmp_path / "rows.txt"
    f.write_text("1 1:0.5 2:1\n")
    r = subprocess.run([tools[0], str(f), tmp_models(256), str(tmp_path / "out.txt")], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stderr
    r = subprocess.run([tools[1], "-r", RANGE, str(f)], capture_output=True, text=True)
    assert r.returncode == 1 and "no CUDA device" in r.stderr and r.stdout == ""
    import haf_grasping_b200 as h
    with pytest.raises(h.HafError) as e:
        h.SvmPredictor(tmp_models(256))
    assert e.value.code == -4


def _ref_bins(oracle_lib):
    if not oracle_lib.ref_available():
        pytest.skip("oracle/_ref (the reference's libsvm programs compiled in place) is not on this box")
    return os.path.join(oracle_lib.REF_DIR, "svm-scale"), os.path.join(oracle_lib.REF_DIR, "svm-predict")


# ---------------------------------------------------------------- committed golden outputs of the reference's programs
GOLDEN_CLI = os.path.join(ROOT, "tests", "golden", "svm_cli")


def _golden_models(tmp_path, tmp_models):
    import gzip
    from conftest import GOLDEN
    trained = str(tmp_path / "trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(trained, "wb") as dst:
        dst.write(src.read())
    return {"trained": trained, "synth": tmp_models(256)}


def test_golden_cli_fixtures_are_what_the_reference_programs_print(oracle_lib, tmp_path, tmp_models):
    """Pins tests/golden/svm_cli (made by tests/golden/make_svm_cli_golden.py) against oracle/_ref where that exists."""
    import json
    ref_scale, ref_predict = _ref_bins(oracle_lib)
    g = lambda n: os.path.join(GOLDEN_CLI, n)  # noqa: E731
    r = subprocess.run([ref_scale, "-r", RANGE, g("features.txt")], capture_output=True, check=True)
    assert r.stdout == open(g("scaled_ref.txt"), "rb").read()
    for k, args in enumerate(json.load(open(g("manifest.json")))["fit_args"]):
        r = subprocess.run([ref_scale] + args + ["-s", str(tmp_path / "r.range"), g("sparse.txt")], capture_output=True, check=True)
        assert r.stdout == open(g("fit_%d_ref.txt" % k), "rb").read() and r.stderr == open(g("fit_%d_ref.stderr" % k), "rb").read()
        assert open(tmp_path / "r.range", "rb").read() == open(g("fit_%d_ref.range" % k), "rb").read()
    for name, model in _golden_models(tmp_path, tmp_models).items():
        r = subprocess.run([ref_predict, g("scaled_ref.txt"), model, str(tmp_path / "o.txt")], capture_output=True, check=True)
        assert open(tmp_path / "o.txt", "rb").read() == open(g("out_%s_ref.txt" % name), "rb").read()
        assert r.stdout == open(g("out_%s_ref.stdout" % name), "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("svm_mode", [0, 1, 2])
def test_front_ends_reproduce_the_committed_reference_outputs(tools, tmp_path, tmp_models, svm_mode):
    """The same comparison as the tests below, against the committed outputs of the reference programs: runs on a box
    that has neither /root/reference nor oracle/_ref."""
    import json
    g = lambda n: os.path.join(GOLDEN_CLI, n)  # noqa: E731
    r = subprocess.run([tools[1], "-r", RANGE, g("features.txt")], capture_output=True, check=True)
    assert r.stdout == open(g("scaled_ref.txt"), "rb").read()
    if svm_mode == 0:
        for k, args in enumerate(json.load(open(g("manifest.json")))["fit_args"]):
            r = subprocess.run([tools[1]] + args + ["-s", str(tmp_path / "r.range"), g("sparse.txt")], capture_output=True, check=True)
            assert r.stdout == open(g("fit_%d_ref.txt" % k), "rb").read() and r.stderr == open(g("fit_%d_ref.stderr" % k), "rb").read()
            assert open(tmp_path / "r.range", "rb").read() == open(g("fit_%d_ref.range" % k), "rb").read()
    for name, model in _golden_models(tmp_path, tmp_models).items():
        r = subprocess.run([tools[0], "--svm-mode", str(svm_mode), g("scaled_ref.txt"), model, str(tmp_path / "o.txt")], capture_output=True, check=True)
        assert open(tmp_path / "o.txt", "rb").read() == open(g("out_%s_ref.txt" % name), "rb").read()
        assert r.stdout == open(g("out_%s_ref.stdout" % name), "rb").read()


# ---------------------------------------------------------------- GPU: byte-exact against the reference's programs
@pytest.fixture(scope="module")
def roll_files(oracle_lib, tmp_path_factory, tmp_models):
    """/tmp/features.txt of roll 3 of pcd2 as the reference's feature class writes it ("-1 k:%.4g ..."), and the file
    svm-scale -r makes of it ("%g" of every non-zero value, a blank after each pair), both written from the oracle's
    values.  Their first 20 rows must equal the committed output of the reference's own class and svm-scale
    (tests/golden/svm_cli); the rest rely on the oracle's text pinned by test_oracle_vs_ref.py."""
    import gzip
    from conftest import GOLDEN
    wd = tmp_path_factory.mktemp("rollfiles")
    trained = str(wd / "trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(trained, "wb") as dst:
        dst.write(src.read())
    clouds = np.load(os.path.join(GOLDEN, "clouds.npz"))
    o = oracle_lib.Oracle(FEATURES, RANGE, trained)
    ores = o.search(clouds["pcd2"], oracle_lib.make_request())
    feats, _ = o.calc_featurevectors(ores["integral"][3], ores["mask"][3])
    rows = ["-1" + "".join(" %d:%.4g" % (k + 1, v) for k, v in enumerate(f)) + "\n" for f in feats]
    scaled = ["-1 " + "".join("%d:%g " % (k + 1, v) for k, v in enumerate(s) if v != 0) + "\n" for s in o.scale(feats)]
    for lines, committed in ((rows, "features.txt"), (scaled, "scaled_ref.txt")):
        with open(os.path.join(GOLDEN_CLI, committed)) as fh:
            assert "".join(lines[:20]) == fh.read(), committed
    files = {"features": str(wd / "features.txt"), "scaled": str(wd / "features.txt.scale")}
    for key, lines in (("features", rows), ("scaled", scaled)):
        with open(files[key], "w") as fh:
            fh.write("".join(lines))
    return dict(files, dir=wd, trained=trained, synth=tmp_models(256))


@pytest.fixture(scope="module")
def programs(oracle_lib, roll_files, tmp_path_factory):
    """(scale_fit(args, src, range_out) -> (stdout, stderr), predict(src, model, out) -> (returncode, stdout, stderr)):
    the reference's own svm-scale / svm-predict where oracle/_ref holds them, else the restatements, pinned first to the
    committed outputs of the reference programs"""
    if not oracle_lib.ref_available():
        libsvm_programs.check_against_committed_outputs(oracle_lib, {k: roll_files[k] for k in ("trained", "synth")},
                                                        tmp_path_factory.mktemp("restated"))
        return libsvm_programs.svm_scale_fit, lambda src, model, out: libsvm_programs.svm_predict(src, model, out, oracle_lib)
    ref_scale, ref_predict = _ref_bins(oracle_lib)

    def scale_fit(args, src, range_out):
        r = subprocess.run([ref_scale] + args + ["-s", range_out, src], capture_output=True, check=True)
        return r.stdout, r.stderr

    def predict(src, model, out):
        r = subprocess.run([ref_predict, src, model, out], capture_output=True)
        return r.returncode, r.stdout, r.stderr
    return scale_fit, predict


def test_restated_programs_reproduce_the_committed_reference_outputs(oracle_lib, tmp_path, tmp_models):
    """the stand-ins of the reference programs (used where oracle/_ref is absent) print what the programs printed"""
    libsvm_programs.check_against_committed_outputs(oracle_lib, _golden_models(tmp_path, tmp_models), tmp_path)


@pytest.mark.gpu
def test_svm_scale_restore_mode_is_byte_identical_to_the_reference_program(tools, roll_files, oracle_lib, tmp_path):
    mine = subprocess.run([tools[1], "-r", RANGE, roll_files["features"]], capture_output=True, check=True)
    ref = open(roll_files["scaled"], "rb").read()
    assert len(ref) > 100000
    assert mine.stdout == ref


@pytest.mark.gpu
@pytest.mark.parametrize("args", [[], ["-l", "0", "-u", "1"], ["-y", "-3", "5"], ["-l", "-2.5", "-u", "0.75", "-y", "0", "1"]])
def test_svm_scale_fit_and_save_mode_matches_the_reference_program(tools, roll_files, programs, tmp_path, args):
    """No -r: min / max come from the data (pass 2 on the GPU, absent entries = 0); the saved range file and the scaled
    text must both equal the reference program's."""
    # a sparser, smaller file: drop every value with |v| < 0.02 and keep 60 rows -> absent entries matter
    rows = []
    for k, ln in enumerate(open(roll_files["features"]).read().split("\n")[:60]):
        t = ln.split()
        if not t:
            continue
        rows.append(" ".join([str(k % 3 - 1)] + [a for a in t[1:] if abs(float(a.split(":")[1])) >= 0.02]))
    src = tmp_path / "sparse.txt"
    src.write_text("\n".join(rows) + "\n")
    a_stdout, a_stderr = programs[0](args, str(src), str(tmp_path / "ref.range"))
    b = subprocess.run([tools[1]] + args + ["-s", str(tmp_path / "mine.range"), str(src)], capture_output=True, check=True)
    assert open(tmp_path / "ref.range", "rb").read() == open(tmp_path / "mine.range", "rb").read()
    assert a_stdout == b.stdout
    assert a_stderr == b.stderr     # the "#nonzeros" warning


@pytest.mark.gpu
@pytest.mark.parametrize("svm_mode", [0, 1, 2])
@pytest.mark.parametrize("which", ["trained", "synth"])
def test_svm_predict_output_file_is_byte_identical_to_the_reference_program(tools, roll_files, programs, tmp_path, svm_mode, which):
    model = roll_files[which]
    ref_out, my_out = tmp_path / "ref.out", tmp_path / "mine.out"
    a_rc, a_stdout, _ = programs[1](roll_files["scaled"], model, str(ref_out))
    b = subprocess.run([tools[0], "--svm-mode", str(svm_mode), roll_files["scaled"], model, str(my_out)], capture_output=True, check=True)
    assert a_rc == 0
    assert open(ref_out, "rb").read() == open(my_out, "rb").read()
    assert a_stdout == b.stdout     # "Accuracy = ...% (c/n) (classification)"


@pytest.mark.gpu
def test_svm_predict_stops_at_a_malformed_line_like_the_reference_program(tools, roll_files, programs, tmp_path):
    lines = open(roll_files["scaled"]).read().split("\n")[:20]
    lines[12] = lines[12].replace(" 7:", " 7;")
    src = tmp_path / "broken.txt"
    src.write_text("\n".join(lines) + "\n")
    a_rc, _, a_stderr = programs[1](str(src), roll_files["synth"], str(tmp_path / "ref.out"))
    b = subprocess.run([tools[0], str(src), roll_files["synth"], str(tmp_path / "mine.out")], capture_output=True)
    assert a_rc == b.returncode == 1
    assert a_stderr == b.stderr == b"Wrong input format at line 13\n"
    assert open(tmp_path / "ref.out", "rb").read() == open(tmp_path / "mine.out", "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("svm_mode,rtol", [(0, 1e-5), (1, 1e-13), (2, 1e-5)])
def test_haf_svm_predict_decision_values_against_libsvm_in_process(roll_files, oracle_lib, programs, svm_mode, rtol):
    """C ABI: decision values of every row against svm_predict_values of the reference's own svm.cpp (oracle/_ref; where
    that is not built, the oracle's restatement of it, whose labels `programs` pinned to the committed outputs of the
    reference's svm-predict), labels identical.  Includes rows wider than the model (indices beyond the model's largest)
    and an all-zero row."""
    import haf_grasping_b200 as h
    rows = []
    for ln in open(roll_files["scaled"]).read().split("\n")[:150]:
        t = ln.split()
        if t:
            x = np.zeros(330)
            for a in t[1:]:
                i, v = a.split(":")
                x[int(i) - 1] = float(v)
            rows.append(x)
    rows[5][:] = 0.0
    rows[6][327] = 0.125           # beyond the model's 323 dimensions: contributes x^2 to every distance (svm.cpp:356-364)
    x = np.array(rows)
    if oracle_lib.ref_available():
        ref = oracle_lib.Ref(FEATURES, RANGE, roll_files["trained"])
        want = [ref.svm_predict(r) for r in x]
    else:
        dec, lab = oracle_lib.Oracle(FEATURES, RANGE, roll_files["trained"]).svm_decision(x)
        want = list(zip(dec.tolist(), lab.tolist()))
    p = h.SvmPredictor(roll_files["trained"], svm_mode=svm_mode, min_dims=330)
    try:
        labels, dec = p.predict(x)
        scale = sum(abs(float(ln.split()[0])) for ln in open(roll_files["trained"]).read().split("SV\n")[1].split("\n") if ln.strip())
        assert np.abs(dec - np.array([w[0] for w in want])).max() <= rtol * scale
        assert labels.astype(int).tolist() == [w[1] for w in want]
        assert p.timing().n_windows == len(x)
    finally:
        p.close()


@pytest.mark.gpu
def test_svm_predict_empty_file_and_rows_without_features(tools, roll_files, programs, tmp_path):
    for name, text in (("empty.txt", ""), ("bare.txt", "1\n-1 \n+1 3:0.25\n")):
        src = tmp_path / name
        src.write_text(text)
        a_rc, a_stdout, _ = programs[1](str(src), roll_files["synth"], str(tmp_path / "ref.out"))
        b = subprocess.run([tools[0], str(src), roll_files["synth"], str(tmp_path / "mine.out")], capture_output=True)
        assert a_rc == b.returncode == 0
        assert a_stdout == b.stdout
        assert open(tmp_path / "ref.out", "rb").read() == open(tmp_path / "mine.out", "rb").read()


@pytest.mark.gpu
def test_haf_svm_predict_chunking_is_invisible(roll_files):
    """More rows than one pass holds (512 MB of densified doubles): results of a row must not depend on the chunk or the
    tile it lands in -- a subset predicted on its own gives the same decision values: bit-identical outside the guard band
    (the FP64 FMA tier sums its support-vector slices in arrival order, so band rows may differ in the last bits)."""
    import haf_grasping_b200 as h
    rng = np.random.default_rng(11)
    n, width = 230000, 330                      # 230 000 x 330 doubles = 607 MB -> two chunks
    nnz_per_row = 4
    idx = np.sort(rng.integers(1, width + 1, size=(n, nnz_per_row)), axis=1)
    idx[:, 1:] += (idx[:, 1:] <= idx[:, :-1]).cumsum(axis=1)  # make strictly ascending (may exceed width: clip below)
    idx = np.minimum(idx, width - nnz_per_row + np.arange(nnz_per_row) + 1)
    for k in range(1, nnz_per_row):
        idx[:, k] = np.maximum(idx[:, k], idx[:, k - 1] + 1)
    val = rng.uniform(-1, 1, size=(n, nnz_per_row))
    rp = np.arange(0, (n + 1) * nnz_per_row, nnz_per_row, dtype=np.int64)
    p = h.SvmPredictor(roll_files["synth"], min_dims=width + nnz_per_row)
    try:
        lab, dec = p.predict((rp, idx.reshape(-1).astype(np.int32), val.reshape(-1)))
        assert p.timing().n_chunks == 2
        sel = np.concatenate([np.arange(0, 700), np.arange(n - 900, n), rng.integers(0, n, 500)])
        rp2 = np.arange(0, (len(sel) + 1) * nnz_per_row, nnz_per_row, dtype=np.int64)
        lab2, dec2 = p.predict((rp2, idx[sel].reshape(-1).astype(np.int32), val[sel].reshape(-1)))
        assert np.array_equal(lab[sel], lab2)
        assert np.abs(dec[sel] - dec2).max() <= 1e-9
        assert (dec[sel] == dec2).mean() >= 0.99
    finally:
        p.close()


@pytest.mark.gpu
def test_haf_scale_abi_matches_numpy_restatement(roll_files):
    """haf_scale_minmax / haf_scale_apply against a direct numpy restatement of svm-scale.c:165-198 and :333-353."""
    import haf_grasping_b200 as h
    rng = np.random.default_rng(3)
    x = rng.normal(size=(500, 40)) * (rng.random((500, 40)) < 0.6)
    x[:, 7] = 0.0                    # never present -> min == max == 0 -> skipped
    x[:, 9] = 2.5                    # single-valued
    fmin, fmax = h.scale_minmax(x, 40)
    assert np.array_equal(fmin[1:], x.min(0)) and np.array_equal(fmax[1:], x.max(0))
    out = h.scale_apply(x, 40, fmin, fmax, lower=-1.0, upper=1.0)
    mn, mx = x.min(0), x.max(0)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = -1.0 + (1.0 - -1.0) * (x - mn) / (mx - mn)
    want = np.where(x == mn, -1.0, np.where(x == mx, 1.0, want))
    want[:, mx == mn] = 0.0
    assert np.array_equal(out, want)
