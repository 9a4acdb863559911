"""Inverse-CDF sampling (qipb200_state_sample) validated without a GPU: a CPU model of the whole algorithm
(tests/native/sample_model.cpp: same chunk layout, the decision rules of rustqip_b200/csrc/sample.cuh, W emulated
ranks) against the reference's serial scan (oracle: soft_measure, measurement_ops.rs:153-176)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import qip_oracle as qo
from rustqip_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "native", "_build", "libsample_model.so")
SRCS = [os.path.join(HERE, "native", "sample_model.cpp"), os.path.join(ROOT, "rustqip_b200", "csrc", "sample.cuh")]
EPS = 1e-12   # draws closer than this to a serial-CDF boundary may land on either neighbour


@pytest.fixture(scope="module")
def model():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in SRCS):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", SO,
                               SRCS[0]])
    L = C.CDLL(SO)
    L.sample_model.restype = C.c_int
    L.sample_model.argtypes = [C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64,
                               C.c_void_p]
    return L


def run_model(L, n, W, psi, indices, draws):
    psi = np.ascontiguousarray(psi, dtype=np.complex128)
    idx = np.ascontiguousarray(indices, dtype=np.uint64)
    r = np.ascontiguousarray(draws, dtype=np.float64)
    out = np.zeros(len(r), dtype=np.uint64)
    assert L.sample_model(n, W, psi.ctypes.data, idx.ctypes.data, len(idx), r.ctypes.data, len(r), out.ctypes.data) == 0
    return out


def serial_index(cdf, r):
    """First index whose inclusive cumulative probability is >= r; None when there is none (-> index 0)."""
    i = int(np.searchsorted(cdf, r, side="left"))
    return i if i < len(cdf) else None


def states(n):
    rng = np.random.default_rng(1000 + n)
    psi = rng.standard_normal(1 << n) + 1j * rng.standard_normal(1 << n)
    psi /= np.linalg.norm(psi)
    yield "random", psi
    basis = np.zeros(1 << n, dtype=np.complex128)
    basis[(0x2D5A >> 1) % (1 << n)] = 1.0
    yield "basis", basis
    ghz = np.zeros(1 << n, dtype=np.complex128)
    ghz[0] = ghz[-1] = np.sqrt(0.5)
    yield "ghz", ghz
    yield "norm0.9", psi * np.sqrt(0.9)


def draws_for(n, cdf):
    rng = np.random.default_rng(7 * n)
    special = [0.0, 1.0 - 2.0 ** -53, 1.0, 0.5, 0.9]
    # the CDF boundaries themselves and points just beside them
    bounds = cdf[rng.integers(0, len(cdf), 8)]
    near = np.concatenate([bounds, np.nextafter(bounds, 2.0), np.nextafter(bounds, -1.0)])
    return np.concatenate([special, near, rng.random(150)]).clip(0.0, 1.0)


@pytest.mark.parametrize("n", range(1, 15))
def test_model_matches_serial_scan(model, n):
    all_q = list(range(n))
    lists = [[n // 2], all_q[::-1], all_q]
    for name, psi in states(n):
        cdf = np.cumsum(np.abs(psi) ** 2)
        draws = draws_for(n, cdf)
        want = {tuple(ix): [qo.soft_measure(n, ix, psi, r) for r in draws] for ix in lists}
        for W in (1, 2, 4, 8):
            if W > (1 << n):
                continue
            # indices [n-1, ..., 0] make the outcome the drawn index itself
            got_index = run_model(model, n, W, psi, all_q[::-1], draws)
            for ix in lists:
                got = run_model(model, n, W, psi, ix, draws)
                bitpos = [n - 1 - q for q in ix]
                for j, r in enumerate(draws):
                    i = int(got_index[j])
                    assert int(got[j]) == sum(((i >> b) & 1) << k for k, b in enumerate(bitpos))
                    d = np.min(np.abs(cdf - r))
                    if d > EPS:
                        assert int(got[j]) == want[tuple(ix)][j], (name, W, ix, r)
                        continue
                    lo, hi = serial_index(cdf, r - EPS), serial_index(cdf, r + EPS)
                    ok = (lo is not None and lo <= i and (hi is None or i <= hi)) or (hi is None and i == 0)
                    assert ok, (name, W, r, i, lo, hi)
            if name == "norm0.9":
                above = draws > 0.9 + EPS
                assert above.any() and np.all(got_index[above] == 0)


def test_sample_entry_rejects_null_state():
    L = _lib.lib()
    idx = np.zeros(1, dtype=np.uint64)
    r = np.zeros(1)
    out = np.zeros(1, dtype=np.uint64)
    st = L.qipb200_state_sample(None, idx.ctypes.data, 1, r.ctypes.data, 1, out.ctypes.data)
    assert st == 1  # QIPB200_ERR_INVALID_ARG
    assert b"sample" in L.qipb200_last_error(None)
