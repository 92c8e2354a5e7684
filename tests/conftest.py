import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_report_header(config):
    try:
        from oracle import blst_ref  # noqa: F401
        return "oracle: BLST (oracle/_ref)"
    except RuntimeError:
        return ("oracle: oracle/replay.py (oracle/_ref not built): pyref for group operations, decoders, partials and "
                "final exponentiation; the answer table tests/golden/oracle_answers.json.gz for verdicts, GT, MSM, "
                "hash_to_G2, combine and aggregate verify")


def _gpu_available():
    try:
        import nim_blscurve_b200 as bg
        return bg.lib().blsgpu_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    """A plain `pytest tests` on a machine without a CUDA device skips the gpu-marked tests instead of erroring in
    their fixtures (the product has no CPU path, so there is nothing for them to run on)."""
    if _gpu_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device / libblsgpu.so: gpu tests need the B200 box (no CPU fallback exists)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def srb():
    import hashlib
    return hashlib.sha256(b"Mr F was here").digest()   # tests/t_batch_verifier.nim:60


@pytest.fixture(scope="session")
def br():
    """BLST itself when oracle/_ref is built; otherwise oracle/replay.py, which rebuilds the same inputs and answers
    from the stored results (tests/golden/oracle_answers.json.gz)."""
    try:
        from oracle import blst_ref
        return blst_ref
    except RuntimeError:
        from oracle import replay
        return replay


@pytest.fixture(scope="session")
def cache():
    import nim_blscurve_b200 as bg
    c = bg.BatchedBLSVerifierCache(max_sets=4096, device=0)
    yield c
    c.close()
