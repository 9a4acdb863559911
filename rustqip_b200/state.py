"""Device context and device-resident state handles (thin RAII over the C ABI).

``State`` plays the role of the two ``Vec<Complex<P>>`` owned by
``LocalBuilder::calculate_state_with_init`` (qip/src/builder.rs:406-407): the
amplitudes stay in HBM between gates; only explicit download copies them out.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._abi import QIP_F32, QIP_F64, cdtype, marshal_op, marshal_ops, prec_of
from .errors import B200Unavailable, CircuitError
from .ops import MatrixOp


class Context:
    """One CUDA device + stream (qipb200_ctx).  One process per GPU."""

    def __init__(self, device=0):
        """device: one CUDA device id, or a list of ids (a power-of-two count): ONE context over several devices
        of this process (qipb200_init_multi) whose states are sharded over them inside the library."""
        self._h = C.c_void_p()
        L = _lib.lib()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            st = L.qipb200_init_multi(C.byref(self._h), len(device), ids)
            self.device = int(device[0])
            self.devices = [int(d) for d in device]
        else:
            st = L.qipb200_init(C.byref(self._h), int(device))
            self.device = int(device)
            self.devices = [int(device)]
        if st != 0:
            msg = L.qipb200_last_error(None).decode("utf-8", "replace")
            raise B200Unavailable(msg)

    @property
    def handle(self):
        return self._h

    def stream_handle(self) -> int:
        """Raw cudaStream_t of this context (for CUDA-event timing by the caller)."""
        sp = C.c_void_p()
        _lib.check(_lib.lib().qipb200_stream_handle(self._h, C.byref(sp)), self._h)
        return int(sp.value or 0)

    def launch_stats(self):
        """dict(all, tile_passes, exchanges, fused_gates) -- cumulative counters of this context."""
        out = (C.c_uint64 * 4)()
        _lib.check(_lib.lib().qipb200_launch_stats(self._h, out), self._h)
        return {"all": int(out[0]), "tile_passes": int(out[1]), "exchanges": int(out[2]), "fused_gates": int(out[3])}

    def jit_stats(self, wait: bool = False):
        """Generated-kernel statistics; wait=True blocks until the background NVRTC compilations are done."""
        out = (C.c_double * 4)()
        note = C.create_string_buffer(512)
        _lib.check(_lib.lib().qipb200_jit_stats(self._h, 1 if wait else 0, out, note, 512), self._h)
        return {"jit_passes": int(out[0]), "tile_passes": int(out[1]), "programs_compiled": int(out[2]),
                "compile_ms_total": out[3], "note": note.value.decode("utf-8", "replace")}

    def profile(self, on: bool):
        """Bracket every fused tile pass / NVLink exchange with CUDA events on the context's stream."""
        _lib.check(_lib.lib().qipb200_profile_enable(self._h, 1 if on else 0), self._h)

    def profile_read(self):
        """dict(tile_ms, tile_passes, exchange_ms, exchanges) since the previous read (synchronises the stream)."""
        out = (C.c_double * 4)()
        _lib.check(_lib.lib().qipb200_profile_read(self._h, out), self._h)
        return {"tile_ms": out[0], "tile_passes": int(out[1]), "exchange_ms": out[2], "exchanges": int(out[3])}

    def kernel_launches(self) -> int:
        return int(_lib.lib().qipb200_kernel_launches(self._h))

    def close(self):
        if self._h:
            _lib.lib().qipb200_shutdown(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def _ptr(a: np.ndarray):
    return a.ctypes.data


class State:
    """Device-resident 2^n amplitudes (or one rank's shard of them)."""

    def __init__(self, n: int, dtype=np.complex128, ctx: Optional[Context] = None, rank: int = 0,
                 world_size: int = 1):
        self.ctx = ctx or default_context()
        self.n = int(n)
        self.prec = prec_of(dtype)
        self.dtype = cdtype(self.prec)
        self.rank, self.world_size = int(rank), int(world_size)
        self._h = C.c_void_p()
        L = _lib.lib()
        if world_size == 1:
            st = L.qipb200_state_new(self.ctx.handle, self.prec, self.n, C.byref(self._h))
        else:
            st = L.qipb200_state_new_sharded(self.ctx.handle, self.prec, self.n, self.rank,
                                             self.world_size, C.byref(self._h))
        _lib.check(st, self.ctx.handle)
        g = (self.world_size - 1).bit_length()
        self.local_len = 1 << (self.n - g)

    # -- lifecycle ------------------------------------------------------------
    def free(self):
        if self._h:
            _lib.lib().qipb200_state_free(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.free()

    def __del__(self):  # pragma: no cover
        try:
            self.free()
        except Exception:
            pass

    def _chk(self, st):
        _lib.check(st, self.ctx.handle)

    # -- builder.rs:409-421 ---------------------------------------------------
    def set_basis(self, index: int):
        self._chk(_lib.lib().qipb200_state_set_basis(self._h, int(index)))

    def upload(self, host: np.ndarray, offset: int = 0):
        host = np.ascontiguousarray(host, dtype=self.dtype)
        self._chk(_lib.lib().qipb200_state_upload(self._h, _ptr(host), int(offset), host.shape[0]))

    def download(self, out: Optional[np.ndarray] = None, offset: int = 0, length: Optional[int] = None):
        if length is None:
            length = (out.shape[0] if out is not None else self.local_len - offset)
        if out is None:
            out = np.empty(length, dtype=self.dtype)
        assert out.dtype == self.dtype and out.flags.c_contiguous
        self._chk(_lib.lib().qipb200_state_download(self._h, _ptr(out), int(offset), int(length)))
        return out

    def download_ptr(self, host_ptr: int, length: int, offset: int = 0):
        """Download into raw host memory (e.g. a pinned torch tensor's data_ptr())."""
        self._chk(_lib.lib().qipb200_state_download(self._h, C.c_void_p(host_ptr), int(offset), int(length)))

    # -- builder.rs:499,514 ---------------------------------------------------
    def apply_op(self, op: MatrixOp):
        cop, keep = marshal_op(op, self.prec)
        self._chk(_lib.lib().qipb200_state_apply_op(self._h, C.byref(cop)))

    def apply_schedule(self, ops: Sequence[MatrixOp], fusion: bool = True):
        arr, keep = marshal_ops(ops, self.prec)
        self.apply_marshalled(arr, len(ops), fusion)

    def apply_marshalled(self, arr, n_ops: int, fusion: bool = True):
        flags = _lib.SCHED_DEFAULT if fusion else _lib.SCHED_NO_FUSION
        self._chk(_lib.lib().qipb200_state_apply_schedule(self._h, arr, n_ops, flags))

    def norm2(self) -> float:
        v = C.c_double()
        self._chk(_lib.lib().qipb200_state_norm2(self._h, C.byref(v)))
        return v.value

    def sync(self):
        self._chk(_lib.lib().qipb200_state_sync(self._h))

    def max_abs_diff(self, other: "State") -> float:
        """max over amplitudes of max(|d re|, |d im|) against another state of the same shape (on the device)."""
        v = C.c_double()
        self._chk(_lib.lib().qipb200_state_max_abs_diff(self._h, other._h, C.byref(v)))
        return v.value

    # -- N3: QIPA state files through the C ABI (checkpoint / resume) ----------------
    def save(self, path: str):
        self._chk(_lib.lib().qipb200_state_save(self._h, str(path).encode()))

    def load(self, path: str):
        self._chk(_lib.lib().qipb200_state_load(self._h, str(path).encode()))

    # -- measurement_ops.rs ---------------------------------------------------
    def measure_probs(self, indices: Sequence[int]) -> np.ndarray:
        idx = np.ascontiguousarray(np.asarray(list(indices), dtype=np.uint64))
        out = np.zeros(1 << len(idx), dtype=np.float64)
        self._chk(_lib.lib().qipb200_state_measure_probs(self._h, _ptr(idx), len(idx), _ptr(out)))
        return out

    def measure_prob(self, measured: int, indices: Sequence[int]) -> float:
        idx = np.ascontiguousarray(np.asarray(list(indices), dtype=np.uint64))
        v = C.c_double()
        self._chk(_lib.lib().qipb200_state_measure_prob(self._h, int(measured), _ptr(idx), len(idx), C.byref(v)))
        return v.value

    def soft_measure(self, indices: Sequence[int], r: float) -> int:
        idx = np.ascontiguousarray(np.asarray(list(indices), dtype=np.uint64))
        m = C.c_uint64()
        self._chk(_lib.lib().qipb200_state_soft_measure(self._h, _ptr(idx), len(idx), float(r), C.byref(m)))
        return int(m.value)

    def sample(self, indices: Sequence[int], draws) -> np.ndarray:
        """soft_measure for every draw in `draws` (floats in [0, 1]) from one read of the state; the state is unchanged.
        Returns the outcomes as uint64, bit i from indices[i]."""
        idx = np.ascontiguousarray(np.asarray(list(indices), dtype=np.uint64))
        r = np.ascontiguousarray(np.asarray(draws, dtype=np.float64).reshape(-1))
        out = np.empty(max(1, r.shape[0]), dtype=np.uint64)
        self._chk(_lib.lib().qipb200_state_sample(self._h, _ptr(idx), len(idx), _ptr(r) if r.shape[0] else _ptr(out),
                                                  r.shape[0], _ptr(out)))
        return out[: r.shape[0]]

    def collapse(self, indices: Sequence[int], measured: int, prob: float):
        idx = np.ascontiguousarray(np.asarray(list(indices), dtype=np.uint64))
        self._chk(_lib.lib().qipb200_state_collapse(self._h, _ptr(idx), len(idx), int(measured), float(prob)))

    # -- multi-GPU --------------------------------------------------------------
    def ipc_export(self):
        a = (C.c_ubyte * _lib.IPC_HANDLE_BYTES)()
        f = (C.c_ubyte * _lib.IPC_HANDLE_BYTES)()
        self._chk(_lib.lib().qipb200_state_ipc_export(self._h, a, f))
        return bytes(a), bytes(f)

    def ipc_import(self, amp_handles: bytes, flag_handles: bytes):
        assert len(amp_handles) == self.world_size * _lib.IPC_HANDLE_BYTES
        a = C.create_string_buffer(amp_handles, len(amp_handles))
        f = C.create_string_buffer(flag_handles, len(flag_handles))
        self._chk(_lib.lib().qipb200_state_ipc_import(self._h, a, f))

    def qubit_map(self):
        m = np.zeros(self.n, dtype=np.uint32)
        self._chk(_lib.lib().qipb200_state_qubit_map(self._h, _ptr(m)))
        return m

    def exchange_bytes(self) -> int:
        v = C.c_uint64()
        self._chk(_lib.lib().qipb200_state_exchange_bytes(self._h, C.byref(v)))
        return int(v.value)


def validate_op(op: MatrixOp, n: int, dtype=np.complex128):
    """make_*_op checks + index range at the ABI; needs no GPU."""
    prec = prec_of(dtype)
    cop, keep = marshal_op(op, prec)
    _lib.check(_lib.lib().qipb200_validate_op(None, prec, int(n), C.byref(cop)), None)


def plan_exchanges(ops: Sequence[MatrixOp], n: int, world_size: int, dtype=np.complex128):
    prec = prec_of(dtype)
    arr, keep = marshal_ops(ops, prec)
    out = np.zeros(max(1, len(ops)), dtype=np.uint32)
    _lib.check(_lib.lib().qipb200_plan_exchanges(prec, int(n), int(world_size), arr, len(ops), _ptr(out)), None)
    return out[: len(ops)]
