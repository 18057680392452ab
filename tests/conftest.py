import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # a fresh checkout has no built artefacts: build the C-ABI library (nvcc cross-compiles without a GPU)
    # and the oracle once, exactly as __graft_entry__.build() does
    lib = os.path.join(ROOT, "singlecarrier_b200", "libsinglecarrier_b200.so")
    if not os.path.exists(lib) or not os.path.exists(os.path.join(ROOT, "oracle", "libsc_oracle.so")):
        import subprocess
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=ROOT, check=True,
                       stdout=subprocess.DEVNULL)


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle as po
    po.build()
    return po.Oracle()


@pytest.fixture(scope="session")
def ref():
    """The reference's own objects when oracle/_ref/libsc_ref.so is built, else their outputs recorded in
    tests/golden/ref_replay.npz (tools/make_golden.py) for the same inputs."""
    from oracle import pyoracle as po
    return po.Reference() if po.have_ref() else po.RecordedReference()


@pytest.fixture(scope="session")
def gold():
    def load(name):
        path = os.path.join(GOLDEN, name)
        if name.endswith(".npz"):
            return dict(np.load(path))
        return np.fromfile(path, dtype="<i2")
    return load


def bits_equal_where_valid(a_bits, b_bits, valid):
    v = np.asarray(valid).astype(bool)
    return bool((a_bits[v] == b_bits[v]).all())


def f32_bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)
