"""What libsvm-3.12's svm-scale (fit-and-save mode) and svm-predict print, restated in Python on top of the oracle.

The front-end tests compare svm-scale-b200 / svm-predict-b200 with the original programs.  Where those are not built
(oracle/_ref), these restatements stand in for them; `check_against_committed_outputs` pins them byte for byte to the
committed outputs of the original programs (tests/golden/svm_cli) before a test relies on them.

They restate what those tests feed the programs (well-formed files, a malformed pair, empty and feature-less rows);
the fuzzed inputs of the reader test still need the original svm-predict.

svm-scale: svm-scale.c:120-229 (passes 1-3, the saved range file, the #nonzeros warning) and output_target / output
(:300-353).  svm-predict: svm-predict.c:82-150 (strtok / strtol / strtod reader, "%g" label per line, the accuracy line)
and exit_input_error (:20-24); decision values from the oracle's restatement of svm_predict_values.
"""
import json
import math
import os
import re

import numpy as np

from conftest import FEATURES, GOLDEN, RANGE

GOLDEN_CLI = os.path.join(GOLDEN, "svm_cli")


def _g(v):
    """C's "%g" of a double, x86 glibc spelling of NaN included (0.0 / 0 is the negative default NaN there)"""
    return "-nan" if math.isnan(v) else "%g" % v


def _pairs(line):
    """svm-scale's pair scan: strtok(NULL, ":") / strtok(NULL, " \\t") after the label"""
    toks = line.split(None, 1)
    rest = toks[1] if len(toks) > 1 else ""
    out = []
    for m in re.finditer(r"\s*([^:\s]+):\s*(\S+)", rest):
        out.append((int(m.group(1)), float(m.group(2))))
    return float(toks[0]), out


def svm_scale_fit(args, src, range_out):
    """svm-scale [-l L] [-u U] [-y YL YU] -s range_out src -> (stdout bytes, stderr bytes); writes range_out"""
    lower, upper, y_scaling, y_lower, y_upper = -1.0, 1.0, False, 0.0, 0.0
    i = 0
    while i < len(args):
        if args[i] == "-l":
            lower, i = float(args[i + 1]), i + 2
        elif args[i] == "-u":
            upper, i = float(args[i + 1]), i + 2
        elif args[i] == "-y":
            y_scaling, y_lower, y_upper, i = True, float(args[i + 1]), float(args[i + 2]), i + 3
        else:
            raise ValueError(args[i])
    rows = [_pairs(ln) for ln in open(src).read().split("\n") if ln.strip()]
    max_index = max((k for _, p in rows for k, _ in p), default=0)
    num_nonzeros = sum(len(p) for _, p in rows)
    fmax = [-math.inf] * (max_index + 1)
    fmin = [math.inf] * (max_index + 1)
    y_max, y_min = -math.inf, math.inf
    for target, pairs in rows:
        if y_scaling:
            y_max, y_min = max(y_max, target), min(y_min, target)
        present = dict(pairs)
        for k in range(1, max_index + 1):
            v = present.get(k, 0.0)
            fmax[k], fmin[k] = max(fmax[k], v), min(fmin[k], v)
    with open(range_out, "w") as fh:
        if y_scaling:
            fh.write("y\n%.16g %.16g\n%.16g %.16g\n" % (y_lower, y_upper, y_min, y_max))
        fh.write("x\n%.16g %.16g\n" % (lower, upper))
        for k in range(1, max_index + 1):
            if fmin[k] != fmax[k]:
                fh.write("%d %.16g %.16g\n" % (k, fmin[k], fmax[k]))
    out, new_num_nonzeros = [], 0
    for target, pairs in rows:
        if y_scaling:
            if target == y_min:
                target = y_lower
            elif target == y_max:
                target = y_upper
            else:
                target = y_lower + (y_upper - y_lower) * (target - y_min) / (y_max - y_min)
        line = [_g(target) + " "]
        present = dict(pairs)
        for k in range(1, max_index + 1):
            if fmax[k] == fmin[k]:
                continue
            v = present.get(k, 0.0)
            if v == fmin[k]:
                v = lower
            elif v == fmax[k]:
                v = upper
            else:
                v = lower + (upper - lower) * (v - fmin[k]) / (fmax[k] - fmin[k])
            if v != 0:
                line.append("%d:%s " % (k, _g(v)))
                new_num_nonzeros += 1
        out.append("".join(line) + "\n")
    err = ""
    if new_num_nonzeros > num_nonzeros:
        err = ("WARNING: original #nonzeros %d\n         new      #nonzeros %d\nUse -l 0 if many original feature values are zeros\n"
               % (num_nonzeros, new_num_nonzeros))
    return "".join(out).encode(), err.encode()


def _strtok(s, pos, delims):
    while pos < len(s) and s[pos] in delims:
        pos += 1
    if pos >= len(s):
        return None, pos
    end = pos
    while end < len(s) and s[end] not in delims:
        end += 1
    return s[pos:end], min(end + 1, len(s))


_INT = re.compile(r"[ \t\n\v\f\r]*[+-]?[0-9]+")
_FLOAT = re.compile(r"[ \t\n\v\f\r]*[+-]?(?:[0-9]+\.?[0-9]*|\.[0-9]+)(?:[eE][+-]?[0-9]+)?")


def _predict_rows(path):
    """svm-predict's reader: (target labels, rows as [(index, value)], 1-based number of the first bad line or 0)"""
    targets, rows = [], []
    text = open(path).read()
    lines = text.split("\n")
    if text.endswith("\n") or not text:
        lines.pop()
    for n, line in enumerate(lines, 1):
        label, pos = _strtok(line, 0, " \t\n")
        if label is None:
            return targets, rows, n
        m = _FLOAT.match(label)
        if not m or m.end() != len(label):
            return targets, rows, n
        pairs, last = [], -1
        while True:
            idx, pos2 = _strtok(line, pos, ":")
            val, pos3 = _strtok(line, pos2, " \t") if idx is not None else (None, pos2)
            if val is None:
                break
            pos = pos3
            mi, mv = _INT.match(idx), _FLOAT.match(val)
            if not mi or mi.end() != len(idx) or int(idx) <= last:
                return targets, rows, n
            if not mv or (mv.end() != len(val) and not val[mv.end()].isspace()):
                return targets, rows, n
            last = int(idx)
            pairs.append((last, float(mv.group())))
        targets.append(float(label))
        rows.append(pairs)
    return targets, rows, 0


def svm_predict(src, model, out_path, oracle_lib):
    """svm-predict src model out_path -> (returncode, stdout bytes, stderr bytes); writes out_path"""
    targets, rows, bad = _predict_rows(src)
    o = oracle_lib.Oracle(FEATURES, RANGE, model)
    labels = []
    if rows:
        dim = max([k for p in rows for k, _ in p] + [1])
        x = np.zeros((len(rows), dim))
        for r, pairs in enumerate(rows):
            for k, v in pairs:
                x[r, k - 1] = v
        labels = o.svm_decision(x)[1].tolist()
    with open(out_path, "w") as fh:
        fh.write("".join("%g\n" % lab for lab in labels))
    if bad:
        return 1, b"", ("Wrong input format at line %d\n" % bad).encode()
    correct = sum(int(lab == t) for lab, t in zip(labels, targets))
    total = len(labels)
    acc = correct / total * 100 if total else math.nan
    return 0, ("Accuracy = %s%% (%d/%d) (classification)\n" % (_g(acc), correct, total)).encode(), b""


def check_against_committed_outputs(oracle_lib, models, tmp_path):
    """both restatements reproduce every committed output of the original programs, byte for byte"""
    g = lambda n: os.path.join(GOLDEN_CLI, n)  # noqa: E731
    for k, args in enumerate(json.load(open(g("manifest.json")))["fit_args"]):
        rng = str(tmp_path / "restated.range")
        out, err = svm_scale_fit(args, g("sparse.txt"), rng)
        assert out == open(g("fit_%d_ref.txt" % k), "rb").read(), args
        assert err == open(g("fit_%d_ref.stderr" % k), "rb").read(), args
        assert open(rng, "rb").read() == open(g("fit_%d_ref.range" % k), "rb").read(), args
    for name, model in models.items():
        out = str(tmp_path / "restated.out")
        rc, stdout, _ = svm_predict(g("scaled_ref.txt"), model, out, oracle_lib)
        assert rc == 0 and stdout == open(g("out_%s_ref.stdout" % name), "rb").read(), name
        assert open(out, "rb").read() == open(g("out_%s_ref.txt" % name), "rb").read(), name
