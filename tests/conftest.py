import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


def pytest_sessionfinish(session, exitstatus):
    """After a GPU run with MMX_PARITY_REPORT=<file>: per test, per tensor, the plain relative error and which clause of
    check_close passed it.  Opt-in, so that a test run never rewrites a committed file or needs a writable tree."""
    import json
    from tests import golden_util
    path = os.environ.get("MMX_PARITY_REPORT")
    if not path:
        return
    try:
        import torch
        on_gpu = torch.cuda.is_available()
    except Exception:
        on_gpu = False
    if not golden_util.REPORT or not on_gpu:
        return
    by_clause = {}
    for r in golden_util.REPORT:
        by_clause[r["passed_by"].split(" (")[0]] = by_clause.get(r["passed_by"].split(" (")[0], 0) + 1
    worst = sorted(golden_util.REPORT, key=lambda r: -r["rel_err"] / max(r["rtol"], 1e-30))[:25]
    with open(path, "w") as f:
        json.dump({"exitstatus": int(exitstatus), "n_checks": len(golden_util.REPORT), "by_clause": by_clause,
                   "worst_relative_to_tolerance": worst, "checks": golden_util.REPORT}, f, indent=1)
