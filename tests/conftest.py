import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (select with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _engine_options_from_env():
    """B200MP_ATTN_STAGED / B200MP_MULTI_TUNE select a kernel variant for the whole session (GPU box only), so the same
    parity tests can be run against every variant that benchmarks compare."""
    import torch
    if torch.cuda.is_available():
        from pytorch_geometric_b200 import ops
        for env, opt in (("B200MP_ATTN_STAGED", "attn_staged"), ("B200MP_MULTI_TUNE", "multi_tune")):
            if os.environ.get(env) is not None:
                ops.set_option(opt, int(os.environ[env]))
    yield


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture
def golden():
    return load_golden


def assert_close(a, b, rtol=1e-5, atol=1e-6, msg=""):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{msg} shape {a.shape} vs {b.shape}"
    err = np.abs(a - b)
    tol = atol + rtol * np.abs(b)
    bad = err > tol
    assert not bad.any(), f"{msg} max err {err.max():.3e} at {np.argwhere(bad)[:5].tolist()}"


def reference_path():
    """Where the UNMODIFIED reference package can be imported from: oracle/_ref, installed by build() from the
    reference checkout (oracle/install_ref.sh)."""
    cand = os.path.join(ROOT, "oracle", "_ref")
    return cand if os.path.isdir(os.path.join(cand, "torch_geometric")) else None


@pytest.fixture
def tg():
    """The reference package (`import torch_geometric`); the test is skipped where it is not installed."""
    path = reference_path()
    if path is None:
        pytest.skip("the reference package is not installed (oracle/install_ref.sh)")
    if path not in sys.path:
        sys.path.insert(0, path)
    import torch_geometric
    return torch_geometric
