import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
FEATURES = os.path.join(GOLDEN, "refdata", "Features.txt")
RANGE = os.path.join(GOLDEN, "refdata", "range21062012_allfeatures")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "ref: needs the in-place compiled reference (oracle/_ref)")


def _sm100_device_present() -> bool:
    """True when the CUDA runtime sees a device of compute capability 10.x (what libhafgpu is built for)."""
    try:
        import torch
        return torch.cuda.is_available() and torch.cuda.get_device_capability(0)[0] == 10
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a box without a B200 skips the gpu tests instead of erroring in their fixtures; tests marked
    `ref` are skipped where the in-place compiled reference (oracle/_ref) is absent and cannot be built."""
    have_gpu = None
    ref_ok = os.path.isdir("/root/reference") or all(
        os.path.exists(os.path.join(ROOT, "oracle", "_ref", f)) for f in ("libhaf_ref.so", "svm-scale", "svm-predict"))
    for item in items:
        if "gpu" in item.keywords:
            if have_gpu is None:
                have_gpu = _sm100_device_present()
            if not have_gpu:
                item.add_marker(pytest.mark.skip(reason="no sm_100 CUDA device (libhafgpu has no CPU fallback)"))
        if "ref" in item.keywords and not ref_ok:
            item.add_marker(pytest.mark.skip(reason="oracle/_ref not built and /root/reference absent"))


@pytest.fixture(scope="session")
def tmp_models(tmp_path_factory):
    """Substitute libsvm models generated on the fly (deterministic), keyed by n_sv."""
    from haf_grasping_b200 import synth

    d = tmp_path_factory.mktemp("models")
    cache = {}

    def get(n_sv=256, seed=7, labels=(1, -1), rho=0.0, gamma=1.0 / 323.0):
        key = (n_sv, seed, labels, rho, gamma)
        if key not in cache:
            p = str(d / ("synth_%d_%d_%d_%d_%g_%g.model" % (n_sv, seed, labels[0], labels[1], rho, gamma)))
            synth.write_synth_model(p, n_sv=n_sv, seed=seed, labels=labels, rho=rho, gamma=gamma)
            cache[key] = p
        return cache[key]

    return get


@pytest.fixture(scope="session")
def oracle_lib():
    from oracle import orc

    orc.build(ref=os.path.isdir("/root/reference"))
    return orc


@pytest.fixture(scope="session")
def hg():
    import haf_grasping_b200 as h
    return h


@pytest.fixture(scope="session")
def clouds_npz():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "clouds.npz"))


@pytest.fixture(scope="session")
def trained_model_path(tmp_path_factory):
    import gzip
    p = str(tmp_path_factory.mktemp("trained_s") / "substitute_trained.model")
    with gzip.open(os.path.join(GOLDEN, "substitute_trained.model.gz"), "rb") as src, open(p, "wb") as dst:
        dst.write(src.read())
    return p
