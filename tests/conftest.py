import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    """golden_v1.npz as a dict.  Inputs made by synth_inputs are stored as their call ("<name>_cfg2": M, N, seed, block;
    "<name>_cfg4": shape..., seed, block) and a digest: they are regenerated here and must match the digest."""
    from oracle import oracle as O
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz")))
    for key in [k for k in g if k.endswith(("_cfg2", "_cfg4"))]:
        name, p = key[:-5], [int(v) for v in g.pop(key)]
        x = O.gen_cfg2(p[0], p[1], seed=p[2], block=p[3]) if key.endswith("_cfg2") else O.gen_cfg4(tuple(p[:-2]), seed=p[-2], block=p[-1])
        assert digest(x) == g.pop(name + "_digest"), "generated input %s differs from the one the reference solved" % name
        g[name] = x
    return g


@pytest.fixture(scope="session")
def refcheck():
    """What the unmodified reference computed on the tests' seeded inputs (tests/golden/make_golden.py reference_checks):
    digests where a test demands bit-identical results, values (sampled at full size) where it allows a tolerance."""
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_checks.npz"))


@pytest.fixture(scope="session")
def port():
    from oracle import oracle as O
    return O.Port()


def digest(a):
    """64-bit digest of an array's shape and values (float64, or bits for a boolean array): equal digests <=> identical arrays
    (up to a 2^-64 collision)."""
    import hashlib
    a = np.asarray(a)
    data = np.packbits(a).tobytes() if a.dtype == bool else np.ascontiguousarray(a, dtype="<f8").tobytes()
    h = hashlib.blake2b(np.asarray(a.shape, dtype="<i8").tobytes() + data, digest_size=8)
    return np.frombuffer(h.digest(), dtype="<u8")[0]


@pytest.fixture(scope="session")
def ptv():
    import proxtv_b200
    proxtv_b200.require_device()
    return proxtv_b200


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def jumps(x, tol=0.0):
    x = np.asarray(x).ravel()
    return np.nonzero(np.abs(np.diff(x)) > tol)[0]
