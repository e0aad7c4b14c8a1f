import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The reference's vendored FAISS (oracle/_ref, tests/cpp/dropin_ivf_check) runs OpenMP teams of one thread per visible CPU; under a
# cgroup quota (16 of 128 cores on the GPU boxes) the spinning teams starve each other.  Bound the checker's teams, not the product.
os.environ.setdefault("OMP_NUM_THREADS", "8")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _build_once():
    """Build the product library and the CPU checkers once per session (cheap no-op when up to date)."""
    import __graft_entry__ as g

    if not os.path.exists(os.path.join(ROOT, "reindexer_b200", "librxgpu.so")) or not os.path.exists(
            os.path.join(ROOT, "oracle", "liboracle_port.so")):
        g.build()


@pytest.fixture
def ref_tape(request):
    """the reference's outputs for this test (helpers.RefTape): replayed from tests/golden/ref_tapes/, recorded, or asked of the
    reference itself where no tape is stored"""
    from helpers import RefTape

    name = f"{request.module.__name__}.{request.node.name}".replace("[", "-").replace("]", "")
    tape = RefTape(name)
    if tape.live and not os.path.isdir(os.path.join(ROOT, "oracle", "_ref")):
        pytest.skip(f"no stored reference answers for {name} and oracle/_ref is not built")
    yield tape
    tape.save()


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "knn_golden.npz"))


GOLDEN_SYNTH_CASES = ["l2_small", "ip_small", "cos_small", "l2_odd_dim", "ip_768", "cos_k_gt_n"]
GOLDEN_TIE_CASES = ["tie_l2", "tie_ip", "dup_rows_cos"]
