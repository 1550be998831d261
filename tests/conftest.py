import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    # a fresh checkout has no built artefacts (they are git-ignored): build them once; never rebuild what is there
    need = [os.path.join(ROOT, "lfbm5d_b200", "_lib", f) for f in ("liblfbm5d_cuda.so", "liblfbm5d_host.so", "LFBM5Ddenoising", "LFBM3Ddenoising")]
    need.append(os.path.join(ROOT, "oracle", "liblfbm5d_oracle.so"))
    if not all(os.path.exists(f) for f in need):
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def oracle():
    import oracleapi
    oracleapi.lib()
    return oracleapi


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference's values: live from oracle/_ref where it is built, stored digests elsewhere (refapi.Pinned)."""
    import refapi
    pins = refapi.Pinned()
    yield pins
    if pins.record:
        pins.save()
