"""Inverse-CDF sampling on the device (qipb200_state_sample / State.sample): per-draw parity with the reference's
serial scan (measurement_ops.rs:153-176), read-only behaviour, statistics, the BASELINE sizes, the rotated layout,
and sharded states (one-process multi-device context and one process per GPU)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import qip_oracle as qo
from rustqip_b200 import circuits, gates
from rustqip_b200.builder import B200Builder
from rustqip_b200.errors import CircuitError
from rustqip_b200.state import Context, State

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPECIAL = [0.0, 1.0 - 2.0 ** -53, 1.0, 0.5]


def serial_indices(psi, draws):
    """Index the serial scan selects for each draw (first inclusive cumulative probability >= r; none -> 0), and the
    distance of each draw to the nearest CDF boundary (the scan's own rounding lives within that distance)."""
    cdf = np.cumsum(np.abs(psi.astype(np.complex128)) ** 2)
    i = np.searchsorted(cdf, draws, side="left")
    idx = np.where(i < len(cdf), i, 0).astype(np.uint64)
    lo = np.clip(i, 0, len(cdf) - 1)
    dist = np.minimum(np.abs(cdf[lo] - draws), np.abs(cdf[np.clip(i - 1, 0, len(cdf) - 1)] - draws))
    return idx, dist


def outcomes(index, n, indices):
    out = np.zeros_like(index)
    for j, q in enumerate(indices):
        out |= ((index >> np.uint64(n - 1 - q)) & np.uint64(1)) << np.uint64(j)
    return out


def check_parity(psi, n, got_index, draws, margin, sub=256, got_sub=None, sub_indices=None):
    """Every draw farther than `margin` from a boundary matches the serial scan; returns how many were excluded.
    The first `sub` draws are also checked against the oracle's own scan call (got_sub: outcomes on sub_indices)."""
    want, dist = serial_indices(psi, draws)
    far = dist > margin
    bad = np.nonzero(far & (got_index != want))[0]
    assert len(bad) == 0, [(float(draws[k]), int(got_index[k]), int(want[k])) for k in bad[:5]]
    if got_sub is not None:
        p128 = np.ascontiguousarray(psi.astype(np.complex128))
        for k in range(min(sub, len(draws))):
            if far[k]:
                assert int(got_sub[k]) == qo.soft_measure(n, sub_indices, p128, float(draws[k])), float(draws[k])
    return int((~far).sum())


@pytest.mark.parametrize("dtype", [np.complex128, np.complex64])
@pytest.mark.parametrize("n", [1, 5, 12, 20])
def test_sample_matches_serial_scan(ctx, n, dtype):
    rng = np.random.default_rng(100 + n)
    draws = np.concatenate([SPECIAL, rng.random(4096)])
    all_rev = list(range(n))[::-1]          # outcome == drawn index
    mixed = list(dict.fromkeys([n - 1, 0, n // 2]))
    kinds = ["random"] + (["circuit"] if n >= 5 else [])
    excluded = 0
    for kind in kinds:
        with State(n, dtype, ctx) as st:
            if kind == "random":
                st.upload(circuits.random_state(n, 7 + n, dtype))
            else:
                st.set_basis(0)
                st.apply_schedule(circuits.random_circuit(n, 8, 40 + n, "H,T,CNOT"))
            psi = st.download()
            got = st.sample(all_rev, draws)
            got_mixed = st.sample(mixed, draws)
            one_by_one = [st.soft_measure(mixed, float(r)) for r in draws[:64]]
        assert got.dtype == np.uint64 and got.shape == draws.shape
        assert np.array_equal(got_mixed, outcomes(got, n, mixed))
        assert list(got_mixed[:64]) == one_by_one
        excluded += check_parity(psi, n, got, draws, 1e-10, got_sub=got_mixed, sub_indices=mixed)
    # 1 - 2^-53 and 1.0 sit at the state's total; random draws within 1e-10 of one of 2^n boundaries are rare
    assert excluded <= 2 * len(kinds) + 8, excluded


def test_sample_is_read_only(ctx):
    n = 14
    with State(n, np.complex128, ctx) as st:
        st.set_basis(3)
        st.apply_schedule(circuits.random_circuit(n, 6, 9, "H,T,CNOT"))
        before = st.download()
        nrm = st.norm2()
        st.sample(list(range(n)), np.random.default_rng(1).random(10000))
        after = st.download()
        assert before.tobytes() == after.tobytes()
        assert abs(st.norm2() - nrm) < 1e-13   # norm2 itself reduces with atomics: equal up to summation order


def test_sample_validation(ctx):
    with State(4, np.complex128, ctx) as st:
        st.set_basis(0)
        assert st.sample([0], []).shape == (0,)
        for bad in ([0.5, 1.5], [-0.1], [float("nan")]):
            with pytest.raises(CircuitError, match="not in"):
                st.sample([0], bad)
        with pytest.raises(CircuitError):
            st.sample([4], [0.5])
        with pytest.raises(CircuitError):
            st.sample([1, 1], [0.5])
        # soft_measure keeps accepting any draw: above the total -> index 0, below 0 -> the first index
        st.set_basis(5)
        assert st.soft_measure([0, 1, 2, 3], 1.5) == 0
        assert st.soft_measure([3, 2, 1, 0], -1.0) == 0


def test_sample_statistics(ctx):
    from scipy import stats
    n, indices, K = 24, [0, 5, 11, 23], 1 << 20
    with State(n, np.complex128, ctx) as st:
        st.set_basis(0)
        st.apply_schedule(circuits.random_circuit(n, 12, 77, "H,T,CNOT"))
        probs = st.measure_probs(indices)
        got = st.sample(indices, np.random.default_rng(2024).random(K))
    counts = np.bincount(got.astype(np.int64), minlength=1 << len(indices))
    live = probs > 1e-12
    assert counts[~live].sum() == 0
    f_exp = probs[live] / probs[live].sum() * K
    p = stats.chisquare(counts[live], f_exp).pvalue
    print("chi-square over %d bins: p = %.3g" % (int(live.sum()), p))
    assert p > 1e-6, (counts, probs)


@pytest.mark.parametrize("dtype,margin", [(np.complex128, 1e-9), (np.complex64, 1e-5)])
def test_sample_baseline_size_n30(ctx, dtype, margin):
    n, K = 30, 1 << 16
    rng = np.random.default_rng(30)
    draws = np.concatenate([SPECIAL, rng.random(K)])
    qubits = list(range(n))
    with State(n, dtype, ctx) as st:
        # GHZ: r <= 1/2 -> |0...0>, above -> |1...1>
        st.set_basis(0)
        st.apply_schedule([gates.h(0)] + [gates.cnot(0, q) for q in range(1, n)])
        got = st.sample(qubits, draws)
        ones = (1 << n) - 1
        assert set(np.unique(got).tolist()) <= {0, ones}
        assert np.all(got[draws < 0.5 - margin] == 0)
        assert np.all(got[(draws > 0.5 + margin) & (draws < 1.0 - margin)] == ones)
        # product of Ry(theta_q): the inverse CDF is a bit-by-bit descent from qubit 0 (the top index bit)
        theta = rng.uniform(0.4, 2.7, n)
        c, s = np.cos(theta / 2), np.sin(theta / 2)
        st.set_basis(0)
        st.apply_schedule([gates.mat([q], np.array([c[q], -s[q], s[q], c[q]], dtype=np.complex128)) for q in range(n)])
        got = st.sample(qubits, draws)
    # a draw within `margin` of a boundary at level d (qubit d) is only checked on the bits above that level
    r, mass = draws.copy(), np.ones_like(draws)
    want = np.zeros(len(draws), dtype=np.uint64)
    depth = np.full(len(draws), n)
    for q in range(n):
        m0 = mass * c[q] ** 2
        depth = np.where((depth == n) & ((np.abs(r - m0) < margin) | (np.abs(r - mass) < margin)), q, depth)
        one = r > m0
        want |= one.astype(np.uint64) << np.uint64(q)
        r = np.where(one, r - m0, r)
        mass = np.where(one, mass * s[q] ** 2, m0)
    checked = (np.uint64(1) << depth.astype(np.uint64)) - np.uint64(1)
    bad = np.nonzero((got ^ want) & checked)[0]
    full = int((depth == n).sum())
    print("n=30 %s: %d of %d draws checked on all 30 bits, mean checked depth %.1f (margin %.0e)" % (
        np.dtype(dtype).name, full, len(draws), float(depth.mean()), margin))
    assert len(bad) == 0, [(float(draws[k]), int(got[k]), int(want[k]), int(depth[k])) for k in bad[:5]]
    assert depth.mean() >= (25 if dtype == np.complex128 else 10)


def test_builder_sample_with_init(ctx):
    b = B200Builder()
    q = b.qubit()
    ra = b.register(3)
    b.h(q)
    b.cnot(q, ra)
    shots = b.sample_with_init([(ra, 0)], b.merge_two_registers(q, ra), 4096, rng=np.random.default_rng(5), ctx=ctx)
    assert set(np.unique(shots).tolist()) == {0, 15}
    b.measure(q)
    with pytest.raises(CircuitError, match="measurement"):
        b.sample_with_init([], q, 10, ctx=ctx)


_ROTATE_WORKER = r"""
import numpy as np
from oracle import qip_oracle as qo
from rustqip_b200 import circuits
from rustqip_b200.state import Context, State

with Context(0) as ctx:
    for n, dtype in [(16, np.complex128), (18, np.complex64)]:
        a = circuits.random_circuit(n, 10, 11, "H,T,CNOT")
        b = circuits.qft(n)[:60] + circuits.random_circuit(n, 5, 12, "H,CZ,CNOT")
        draws = np.random.default_rng(n).random(2048)
        idx = [n - 1, 0, 3]
        with State(n, dtype, ctx) as st:
            st.set_basis(5)
            st.apply_schedule(a)
            st.apply_schedule(b)
            got = st.sample(idx, draws)                 # on the layout the rotating schedules left behind
            psi = st.download().astype(np.complex128)
        with State(n, dtype, ctx) as st:
            st.set_basis(5)
            st.apply_schedule(a)
            st.apply_schedule(b)
            m = st.soft_measure(idx, float(draws[0]))   # the one-draw case, also on the permuted layout
        cdf = np.cumsum(np.abs(psi) ** 2)
        ok = [got[k] == qo.soft_measure(n, idx, psi, float(r)) for k, r in enumerate(draws) if np.min(np.abs(cdf - r)) > 1e-10]
        assert all(ok), (n, ok.count(False))
        assert m == got[0], (m, got[0])
        print("rotate sample n=%d %s: %d draws OK" % (n, np.dtype(dtype).name, len(ok)))
"""


@pytest.mark.xfail(reason="opt-in path written after the round's GPU budget was spent: never run on hardware", strict=False)
def test_sample_after_rotating_schedule():
    env = dict(os.environ, QIPB200_ROTATE="1", QIPB200_JIT="sync", PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-c", _ROTATE_WORKER], cwd=ROOT, env=env, capture_output=True, text=True, timeout=420)
    sys.stdout.write(p.stdout[-3000:])
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]


def _gpu_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sample_multi_device_context(world):
    if _gpu_count() < world:
        pytest.skip("needs %d GPUs" % world)
    g = (world - 1).bit_length()
    with Context(list(range(world))) as mctx:
        for n, dtype in [(17, np.complex128), (16, np.complex64)]:
            draws = np.concatenate([SPECIAL, np.random.default_rng(n).random(4096)])
            with State(n, dtype, mctx) as st:
                st.set_basis(5)
                st.apply_schedule(circuits.sharded_parity_circuit(n, g))   # leaves migrated qubits behind
                got = st.sample(list(range(n))[::-1], draws)               # restores the layout on every shard
                m = st.soft_measure([0, 2], 0.4)
                psi = st.download()
            excluded = check_parity(psi, n, got, draws, 1e-10)
            assert m == qo.soft_measure(n, [0, 2], psi.astype(np.complex128), 0.4)
            assert excluded <= 8, excluded
            print("multi-device world=%d n=%d %s: %d draws, %d at a boundary" % (world, n, np.dtype(dtype).name, len(draws), excluded))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sample_one_process_per_gpu(world):
    if _gpu_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29670 + world), os.path.join(ROOT, "tests", "sample_dist_worker.py")]
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    sys.stdout.write(p.stdout[-4000:])
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


def test_sample_host_example():
    exe = os.path.join(ROOT, "examples", "sample_host")
    p = subprocess.run([exe], cwd=ROOT, capture_output=True, text=True, timeout=300)
    sys.stdout.write(p.stdout)
    assert p.returncode == 0, p.stdout + p.stderr
