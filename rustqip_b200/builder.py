"""Host-side mirror of the slice of ``LocalBuilder`` that reaches the hot path.

Reference: qip/src/builder.rs (pipeline of ``(indices, object)`` entries :23-28,
``apply_circuit_object`` :376-398, ``calculate_state_with_init`` :400-519, conditioned
decomposition :664-814) and qip/src/builder_traits.rs (register bookkeeping, Clifford+T
helpers :398-476, Toffoli network :505-568).

Only what is needed to *produce the gate schedule* is mirrored -- circuit construction is
host-only bookkeeping that stays Rust in a real integration (SURVEY.md section 2 rows 10-13).
``calculate_state_with_init`` is the in-scope entry: it translates the pipeline with the
reference's gate table and runs it on the B200 through the C ABI.
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import gates
from .errors import CircuitError
from .ops import MatrixOp


class Register:
    """qip ``Qudit``: an ordered set of qubit indices (qip/src/builder.rs:33-105)."""

    def __init__(self, indices: Sequence[int]):
        self.indices = list(indices)

    def n(self) -> int:
        return len(self.indices)


class B200Builder:
    """Drop-in for ``LocalBuilder<P>`` on the path BASELINE.json names."""

    def __init__(self, dtype=np.complex128):
        self.dtype = dtype
        self._n = 0
        self.pipeline: List[Tuple[List[int], str, object]] = []  # (indices, kind, payload)
        self._temps: List[int] = []

    # ---- register bookkeeping (builder_traits.rs:61-222, builder.rs:300-375) -------------
    def n(self) -> int:
        return self._n

    def qubit(self) -> Register:
        return self.register(1)

    def register(self, n: int) -> Register:
        if n <= 0:
            raise CircuitError("register size must be positive (NonZeroUsize)")
        r = Register(range(self._n, self._n + n))
        self._n += n
        return r

    def merge_two_registers(self, a: Register, b: Register) -> Register:
        return Register(a.indices + b.indices)

    def merge_registers(self, rs: Iterable[Register]) -> Register:
        out: List[int] = []
        for r in rs:
            out += r.indices
        return Register(out)

    def split_all_register(self, r: Register) -> List[Register]:
        return [Register([i]) for i in r.indices]

    def pipeline_depth(self) -> int:
        return len(self.pipeline)

    # ---- apply_circuit_object (builder.rs:376-398): 1-qubit objects broadcast over a register
    def _push1(self, r: Register, kind: str, payload=None) -> Register:
        for i in r.indices:
            self.pipeline.append(([i], kind, payload))
        return r

    def x(self, r): return self._push1(r, "X")
    def y(self, r): return self._push1(r, "Y")
    def z(self, r): return self._push1(r, "Z")
    def h(self, r): return self._push1(r, "H")
    def s(self, r): return self._push1(r, "S")
    def t(self, r): return self._push1(r, "T")
    def rz(self, r, theta: float): return self._push1(r, "RZ", float(theta))

    def s_dagger(self, r):  # builder_traits.rs:419-422
        return self.s(self.z(r))

    def t_dagger(self, r):  # builder_traits.rs:408-411
        return self.t(self.s_dagger(r))

    def cnot(self, cr: Register, r: Register):  # builder_traits.rs:425-451
        if cr.n() > 1:
            raise CircuitError("Clifford CNOT can only have a single control qubit.")
        for i in r.indices:
            self.pipeline.append(([cr.indices[0], i], "CNOT", None))
        return cr, r

    def swap(self, ra: Register, rb: Register):  # builder_traits.rs:454-480: three CNOTs per pair
        if ra.n() != rb.n():
            raise CircuitError("Swap must be between registers of the same size.")
        for a, b in zip(ra.indices, rb.indices):
            qa, qb = Register([a]), Register([b])
            self.cnot(qa, qb)
            self.cnot(qb, qa)
            self.cnot(qa, qb)
        return ra, rb

    def apply_matrix(self, r: Register, data) -> Register:  # MAT, builder.rs:468-470
        data = np.asarray(data).reshape(-1)
        if data.shape[0] != 1 << (2 * r.n()):
            raise CircuitError("Matrix has incorrect N and cannot be broadcast")
        self.pipeline.append((list(r.indices), "MAT", data))
        return r

    def apply_swap_object(self, ra: Register, rb: Register):  # UnitaryMatrixObject::SWAP, builder.rs:471-478
        self.pipeline.append((ra.indices + rb.indices, "SWAP", None))
        return ra, rb

    def measure(self, r: Register):  # builder_traits.rs:622-628 (recorded; executed by calculate_state)
        self.pipeline.append((list(r.indices), "MEASURE", None))
        return r, len([1 for p in self.pipeline if p[1] == "MEASURE"]) - 1

    # ---- Toffoli network (builder_traits.rs:505-568) ------------------------------------------
    def basic_toffoli(self, cr: Register, r: Register):
        if cr.n() != 2:
            raise CircuitError("Basic Toffoli can only be applied to two control qubits.")
        cra, crb = Register([cr.indices[0]]), Register([cr.indices[1]])
        self.h(r)
        self.cnot(crb, r)
        self.t_dagger(r)
        self.cnot(cra, r)
        self.t(r)
        self.cnot(crb, r)
        self.t_dagger(r)
        self.cnot(cra, r)
        self.t(crb)
        self.t(r)
        self.cnot(cra, crb)
        self.h(r)
        self.t(cra)
        self.t_dagger(crb)
        self.cnot(cra, crb)
        return cr, r

    def toffoli(self, cr: Register, r: Register):
        if cr.n() == 1:
            return self.cnot(cr, r)
        if cr.n() == 2:
            return self.basic_toffoli(cr, r)
        raise CircuitError("more than two controls need the ancilla ladder (builder_traits.rs:552-563): not mirrored")

    # ---- condition_with (conditioning.rs:12-85, builder.rs:664-764 for X / CNOT / swap) -----------
    def condition_with(self, cr: Register) -> "Conditioned":
        return Conditioned(self, cr)

    # ---- the in-scope entry ---------------------------------------------------------------------
    def unitary_ops(self) -> List[MatrixOp]:
        """Gate table of calculate_state_with_init (builder.rs:439-498) for the unitary entries."""
        ops = []
        for indices, kind, payload in self.pipeline:
            if kind == "MEASURE":
                continue
            if kind == "X": ops.append(gates.x(indices[0]))
            elif kind == "Y": ops.append(gates.y(indices[0]))
            elif kind == "Z": ops.append(gates.z(indices[0]))
            elif kind == "H": ops.append(gates.h(indices[0]))
            elif kind == "S": ops.append(gates.s(indices[0]))
            elif kind == "T": ops.append(gates.t(indices[0]))
            elif kind == "RZ": ops.append(gates.rz(indices[0], payload))
            elif kind == "CNOT": ops.append(gates.cnot(indices[0], indices[1]))
            elif kind == "MAT": ops.append(gates.mat(indices, payload))
            elif kind == "SWAP":
                half = len(indices) // 2
                ops.append(gates.swap(indices[:half], indices[half:]))
            else:  # pragma: no cover
                raise CircuitError("unknown pipeline entry %r" % kind)
        return ops

    def initial_index(self, init: Sequence[Tuple[Register, int]]) -> int:
        """builder.rs:409-420: bit i of a register's value goes to its i-th qubit."""
        n = self._n
        idx = 0
        for reg, value in init:
            for i, q in enumerate(reg.indices):
                idx |= ((value >> i) & 1) << (n - 1 - q)
        return idx

    def calculate_state_with_init(self, init: Sequence[Tuple[Register, int]] = (), ctx=None, fusion: bool = True,
                                  measured: Optional[Sequence[int]] = None, rng=None):
        """LocalBuilder::calculate_state_with_init (builder.rs:400-519) on the B200.

        Returns (state, measurements); measurements is a list of (value, probability).  The
        reference draws the outcome with rand::random (quirk Q8); pass `measured` to force
        outcomes or `rng` (anything with .random()) to draw them."""
        from .state import State
        measurements = []
        forced = list(measured) if measured is not None else None
        with State(self._n, self.dtype, ctx) as st:
            st.set_basis(self.initial_index(init))
            batch: List[Tuple[List[int], str, object]] = []

            def flush():
                if batch:
                    sub = B200Builder(self.dtype)
                    sub._n, sub.pipeline = self._n, list(batch)
                    st.apply_schedule(sub.unitary_ops(), fusion=fusion)
                    batch.clear()

            for entry in self.pipeline:
                if entry[1] != "MEASURE":
                    batch.append(entry)
                    continue
                flush()
                indices = entry[0]
                if forced:
                    m = forced.pop(0)
                else:
                    r = rng.random() if rng is not None else float(np.random.random())
                    m = st.soft_measure(indices, r)
                p = st.measure_prob(m, indices)
                st.collapse(indices, m, p)
                measurements.append((m, p))
            flush()
            return st.download(), measurements


    def sample_with_init(self, init: Sequence[Tuple[Register, int]], indices, shots: int, rng=None, ctx=None,
                         fusion: bool = True) -> np.ndarray:
        """Run the unitary pipeline once from the initial registers and draw `shots` outcomes of the qubits
        `indices` (a Register or qubit indices; bit i of an outcome from the i-th qubit) from the final state
        (soft_measure, measurement_ops.rs:153-176, once per shot).  `rng`: a numpy Generator for the draws.
        A pipeline with a measurement entry is refused: shots after a mid-circuit collapse are not independent."""
        from .state import State
        if any(kind == "MEASURE" for _, kind, _ in self.pipeline):
            raise CircuitError("sample_with_init: the pipeline contains a measurement; shots need a unitary pipeline")
        qubits = indices.indices if isinstance(indices, Register) else list(indices)
        draws = (rng if rng is not None else np.random.default_rng()).random(int(shots))
        with State(self._n, self.dtype, ctx) as st:
            st.set_basis(self.initial_index(init))
            st.apply_schedule(self.unitary_ops(), fusion=fusion)
            return st.sample(qubits, draws)


class Conditioned:
    """conditioning.rs:29-85 restricted to what LocalBuilder can decompose without ancillas."""

    def __init__(self, parent: B200Builder, cr: Register):
        self.parent, self.cr = parent, cr

    def x(self, r: Register) -> Register:  # builder.rs:672
        for i in r.indices:
            self.parent.toffoli(self.cr, Register([i]))
        return r

    def cnot(self, cr: Register, r: Register):  # builder.rs:754-764: controls merged, then toffoli
        for i in r.indices:
            self.parent.toffoli(self.parent.merge_two_registers(self.cr, cr), Register([i]))
        return cr, r

    def swap(self, ra: Register, rb: Register):  # CliffordTBuilder::swap on the conditioned builder
        if ra.n() != rb.n():
            raise CircuitError("Swap must be between registers of the same size.")
        for a, b in zip(ra.indices, rb.indices):
            qa, qb = Register([a]), Register([b])
            self.cnot(qa, qb)
            self.cnot(qb, qa)
            self.cnot(qa, qb)
        return ra, rb

    def dissolve(self) -> Register:
        return self.cr


def readme_cswap_circuit(dtype=np.complex128):
    """The README example (README.md:26-63) = BASELINE.json configs[0]: 7 qubits,
    H(q); controlled swap(ra, rb) on q; H(q); measure q; init ra=0b000, rb=0b001."""
    b = B200Builder(dtype)
    q = b.qubit()
    ra = b.register(3)
    rb = b.register(3)
    q = b.h(q)
    cb = b.condition_with(q)
    ra, rb = cb.swap(ra, rb)
    q = cb.dissolve()
    q = b.h(q)
    q, handle = b.measure(q)
    return b, q, ra, rb, handle
