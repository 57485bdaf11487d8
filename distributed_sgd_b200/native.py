"""ctypes binding of libdsgd.so (the C ABI in include/dsgd.h) and libdsgd_host.so (data preparation).

This is the only place the Python host touches native code.  There is no fallback: if libdsgd.so is
missing or no B200 is usable, the call raises (NativeLibraryMissing / DsgdError) -- nothing in this
package computes the hot path on the CPU.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
from typing import Optional, Tuple

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libdsgd.so")
HOST_LIB_PATH = os.path.join(_PKG, "libdsgd_host.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "dsgd.h")

UNIQUE_ID_BYTES = 128
MAX_MODELS = 32
IPC_HANDLE_BYTES = 64
FLAG_ASYNC = 1
REPLICA_SELF, REPLICA_MASTER = 0, 1

OK, ERR_INVALID, ERR_STATE, ERR_EMPTY, ERR_RANGE, ERR_CUDA, ERR_NCCL, ERR_NOMEM, ERR_TIMEOUT = 0, -1, -2, -3, -4, -5, -6, -7, -8


class NativeLibraryMissing(ImportError):
    pass


class DsgdError(RuntimeError):
    """A failing C-ABI call.  `.code` is the DSGD_ERR_* value."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[dsgd {code}] {msg}")
        self.code = code


class DsgdInvalid(DsgdError, ValueError):  # the reference's require(...) -> IllegalArgumentException
    pass


class DsgdState(DsgdError):  # "slave is in synchronous mode", "already running"
    pass


class DsgdEmpty(DsgdError, ValueError):  # Vec.sum on an empty list (math/Vec.scala:129)
    pass


class DsgdRange(DsgdError, IndexError):  # ArrayIndexOutOfBoundsException on data(idx)
    pass


_EXC = {ERR_INVALID: DsgdInvalid, ERR_STATE: DsgdState, ERR_EMPTY: DsgdEmpty, ERR_RANGE: DsgdRange}


def build(verbose: bool = False) -> None:
    """Compile libdsgd.so (nvcc, sm_100a) and libdsgd_host.so (gcc) in-tree."""
    r = subprocess.run(["make", "-C", os.path.join(_PKG, "csrc"), "all"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
        print(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("building libdsgd.so failed")


_lib = None
_host = None

_vp, _i32, _i64, _f64, _u32, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_uint32, C.c_uint64

# name -> argtypes; every function returns int unless listed in _RESTYPE
ABI = {
    "dsgd_create": [C.POINTER(_vp), C.c_int, _i32, _f64, C.c_int, C.c_int, _u32],
    "dsgd_destroy": [_vp],
    "dsgd_last_error": [_vp],
    "dsgd_info": [_vp],
    "dsgd_set_stream": [_vp, _vp],
    "dsgd_synchronize": [_vp],
    "dsgd_timer_start": [_vp],
    "dsgd_timer_stop": [_vp, C.POINTER(C.c_float)],
    "dsgd_launch_count": [_vp, C.POINTER(_i64)],
    "dsgd_profile_begin": [_vp, _i32],
    "dsgd_profile_end": [_vp, C.POINTER(C.c_float), C.POINTER(_i64)],
    "dsgd_load_csr": [_vp, _i64, _i64, _vp, _vp, _vp, _vp],
    "dsgd_set_dim_sparsity": [_vp, _vp],
    "dsgd_compute_dim_sparsity": [_vp, _i64, _vp],
    "dsgd_set_weights": [_vp, _vp],
    "dsgd_get_weights": [_vp, _vp],
    "dsgd_forward": [_vp, _vp, _vp, _i64, _vp],
    "dsgd_gradient": [_vp, _vp, _vp, _i64, _vp, C.POINTER(_f64)],
    "dsgd_eval": [_vp, _vp, _i64, _i64, C.POINTER(_f64), C.POINTER(_f64)],
    "dsgd_eval_counts": [_vp, _vp, _i64, _i64, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_f64)],
    "dsgd_comm_unique_id": [_vp],
    "dsgd_comm_init": [_vp, _vp],
    "dsgd_xchg_export": [_vp, _vp],
    "dsgd_xchg_import": [_vp, C.c_int, _vp],
    "dsgd_xchg_attach": [_vp, C.c_int, _vp],
    "dsgd_xchg_stats": [_vp, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)],
    "dsgd_debug_timeline": [_vp, _vp],
    "dsgd_set_grid_limit": [_vp, _i32],
    "dsgd_reserve": [_vp, _i64, _i64],
    "dsgd_set_workers": [_vp, _i32, _vp, _i32],
    "dsgd_sync_step": [_vp, _vp, _i64, _f64, C.POINTER(_f64)],
    "dsgd_sync_steps": [_vp, _vp, _i64, _i64, _f64, _vp],
    "dsgd_stage_samples": [_vp, _vp, _i64],
    "dsgd_sync_steps_staged": [_vp, _i64, _i64, _i64, _f64, C.c_int],
    "dsgd_read_losses": [_vp, _vp, _i64],
    "dsgd_models_set": [_vp, _i32, _vp, _vp, _vp],
    "dsgd_models_shape": [_vp, C.POINTER(_i32), C.POINTER(_i32)],
    "dsgd_models_get_weights": [_vp, _vp],
    "dsgd_models_steps": [_vp, _vp, _i64, _i64, _vp, _vp],
    "dsgd_models_eval_counts": [_vp, _i32, _i64, _i64, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_f64)],
    "dsgd_async_host_master": [_vp, _vp],
    "dsgd_ipc_export": [_vp, C.c_int, _vp],
    "dsgd_ipc_import": [_vp, C.c_int, _vp],
    "dsgd_peer_attach": [_vp, C.c_int, _vp, C.c_int],
    "dsgd_async_replay": [_vp, _vp, _vp, _i32, _i64, _f64],
    "dsgd_async_running": [_vp, C.POINTER(C.c_int)],
    "dsgd_async_master_weights": [_vp, _vp],
    "dsgd_async_outbox_enable": [_vp],
    "dsgd_async_outbox_read": [_vp, _vp],
    "dsgd_async_elapsed_ms": [_vp, C.POINTER(C.c_float)],
    "dsgd_start_async": [_vp, _vp, _vp, _i64, _i32, _f64, _i32, _i64, _u64],
    "dsgd_stop_async": [_vp],
    "dsgd_update_grad": [_vp, _vp, _vp, _i64],
    "dsgd_async_updates": [_vp, C.POINTER(_i64)],
}
_RESTYPE = {"dsgd_last_error": C.c_char_p, "dsgd_info": C.c_char_p}


def lib():
    """Load libdsgd.so; raises NativeLibraryMissing if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback for the hot path.")
        l = C.CDLL(LIB_PATH)
        for name, args in ABI.items():
            fn = getattr(l, name)  # AttributeError here == header and library disagree
            fn.argtypes = args
            fn.restype = _RESTYPE.get(name, C.c_int)
        _lib = l
    return _lib


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_rows", C.c_int64), ("dim", C.c_int32), ("mean_nnz", C.c_double),
                ("sigma", C.c_double), ("max_nnz", C.c_int32), ("zipf_s", C.c_double), ("zipf_q", C.c_double),
                ("label_noise", C.c_double)]


def host_lib():
    global _host
    if _host is None:
        if not os.path.exists(HOST_LIB_PATH):
            raise NativeLibraryMissing(f"{HOST_LIB_PATH} not found: run __graft_entry__.build()")
        h = C.CDLL(HOST_LIB_PATH)
        h.dsgd_synth_row_ptr.restype = C.c_int64
        h.dsgd_synth_row_ptr.argtypes = [C.POINTER(SynthParams), _vp]
        h.dsgd_synth_fill.argtypes = [C.POINTER(SynthParams), _vp, _vp, _vp, _vp, _vp]
        h.dsgd_rcv1_count.argtypes = [C.c_char_p, C.POINTER(_i64), C.POINTER(_i64)]
        h.dsgd_rcv1_parse.argtypes = [C.c_char_p, _i32, _i64, _i64, _vp, _vp, _vp, _vp]
        h.dsgd_rcv1_labels.argtypes = [C.c_char_p, _vp, _i64, _vp]
        h.dsgd_rcv1_write.argtypes = [C.c_char_p, C.c_char_p, _i64, _vp, _vp, _vp, _vp, _i64]
        h.dsgd_draw_epoch.restype = C.c_int64
        h.dsgd_draw_epoch.argtypes = [C.c_uint64, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _i64]
        h.dsgd_feistel_pos.restype = C.c_uint32
        h.dsgd_feistel_pos.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64]
        _host = h
    return _host


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _arr(a, dtype, n: Optional[int] = None, what: str = "array") -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=dtype).reshape(-1)
    if n is not None and a.size != n:
        raise DsgdInvalid(ERR_INVALID, f"{what}: expected {n} elements, got {a.size}")
    return a


class NativeCtx:
    """One dsgd_ctx == one GPU worker (a reference Slave with its SparseSVM)."""

    def __init__(self, device: int, dim: int, lam: float, rank: int = 0, world: int = 1, is_async: bool = False):
        self._l = lib()
        self._h = C.c_void_p()
        self.dim, self.lam, self.rank, self.world, self.device = int(dim), float(lam), int(rank), int(world), int(device)
        rc = self._l.dsgd_create(C.byref(self._h), device, dim, lam, rank, world, FLAG_ASYNC if is_async else 0)
        if rc != OK:
            msg = (self._l.dsgd_last_error(None) or b"").decode()
            self._h = C.c_void_p()
            raise _EXC.get(rc, DsgdError)(rc, msg)
        self.n_rows = 0

    # -- plumbing --
    def _ck(self, rc: int):
        if rc != OK:
            raise _EXC.get(rc, DsgdError)(rc, (self._l.dsgd_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._l.dsgd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def info(self) -> dict:
        return json.loads(self._l.dsgd_info(self._h).decode())

    def set_stream(self, cuda_stream: Optional[int]):
        self._ck(self._l.dsgd_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def synchronize(self):
        self._ck(self._l.dsgd_synchronize(self._h))

    def timer_start(self):
        self._ck(self._l.dsgd_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self._ck(self._l.dsgd_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        n = C.c_int64()
        self._ck(self._l.dsgd_launch_count(self._h, C.byref(n)))
        return n.value

    def profile_begin(self, sample_every: int = 1):
        self._ck(self._l.dsgd_profile_begin(self._h, sample_every))

    def profile_end(self) -> Tuple[float, int]:
        """(mean duration in ms of the sampled gradient-kernel launches, number sampled)."""
        ms, n = C.c_float(), C.c_int64()
        self._ck(self._l.dsgd_profile_end(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # -- data / model --
    def load_csr(self, row_ptr, col, val, label):
        row_ptr = _arr(row_ptr, np.int64)
        n_rows = row_ptr.size - 1
        nnz = int(row_ptr[-1]) if row_ptr.size else 0
        col, val, label = _arr(col, np.int32), _arr(val, np.float32), _arr(label, np.int8, n_rows, "label")
        if col.size != val.size or col.size < nnz:
            raise DsgdInvalid(ERR_INVALID, "load_csr: col/val shorter than row_ptr[-1]")
        self._ck(self._l.dsgd_load_csr(self._h, n_rows, nnz, _ptr(row_ptr), _ptr(col), _ptr(val), _ptr(label)))
        self.n_rows = n_rows

    def set_dim_sparsity(self, d):
        d = _arr(d, np.float64, self.dim, "dim_sparsity")
        self._ck(self._l.dsgd_set_dim_sparsity(self._h, _ptr(d)))

    def compute_dim_sparsity(self, n_train: int) -> np.ndarray:
        out = np.zeros(self.dim, dtype=np.float64)
        self._ck(self._l.dsgd_compute_dim_sparsity(self._h, n_train, _ptr(out)))
        return out

    def set_weights(self, w):
        w = _arr(w, np.float64, self.dim, "weights")
        self._ck(self._l.dsgd_set_weights(self._h, _ptr(w)))

    def get_weights(self) -> np.ndarray:
        out = np.zeros(self.dim, dtype=np.float64)
        self._ck(self._l.dsgd_get_weights(self._h, _ptr(out)))
        return out

    # -- requests --
    def _w(self, w):
        return None if w is None else _arr(w, np.float64, self.dim, "weights")

    def forward(self, samples, w=None) -> np.ndarray:
        samples = _arr(samples, np.int32)
        out = np.zeros(samples.size, dtype=np.float64)
        w = self._w(w)
        self._ck(self._l.dsgd_forward(self._h, _ptr(w), _ptr(samples), samples.size, _ptr(out)))
        return out

    def gradient(self, samples, w=None, want_loss: bool = False):
        samples = _arr(samples, np.int32)
        out = np.zeros(self.dim, dtype=np.float64)
        loss = C.c_double()
        w = self._w(w)
        self._ck(self._l.dsgd_gradient(self._h, _ptr(w), _ptr(samples), samples.size, _ptr(out),
                                       C.byref(loss) if want_loss else None))
        return (out, loss.value) if want_loss else out

    def eval(self, row_begin: int, row_end: int, w=None) -> Tuple[float, float]:
        loss, acc = C.c_double(), C.c_double()
        w = self._w(w)
        self._ck(self._l.dsgd_eval(self._h, _ptr(w), row_begin, row_end, C.byref(loss), C.byref(acc)))
        return loss.value, acc.value

    def eval_counts(self, row_begin: int, row_end: int, w=None) -> Tuple[int, int, float]:
        """(hinge sum, correct count, ||w||^2) over rows [row_begin, row_end) -- exact shardable form."""
        h, c, n2 = C.c_int64(), C.c_int64(), C.c_double()
        w = self._w(w)
        self._ck(self._l.dsgd_eval_counts(self._h, _ptr(w), row_begin, row_end, C.byref(h), C.byref(c), C.byref(n2)))
        return h.value, c.value, n2.value

    # -- sync --
    def set_workers(self, counts, k_total: int = 0):
        """Logical workers on this ctx: counts[v] samples each per step; k_total = Vec.mean divisor."""
        counts = _arr(counts, np.int32)
        self._ck(self._l.dsgd_set_workers(self._h, counts.size, _ptr(counts) if counts.size else None, k_total))

    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * UNIQUE_ID_BYTES)()
        rc = lib().dsgd_comm_unique_id(C.cast(buf, C.c_void_p))
        if rc != OK:
            raise DsgdError(rc, (lib().dsgd_last_error(None) or b"").decode())
        return bytes(buf)

    def comm_init(self, uid: bytes):
        assert len(uid) == UNIQUE_ID_BYTES
        buf = (C.c_uint8 * UNIQUE_ID_BYTES).from_buffer_copy(uid)
        self._ck(self._l.dsgd_comm_init(self._h, C.cast(buf, C.c_void_p)))

    def xchg_export(self) -> bytes:
        buf = (C.c_uint8 * IPC_HANDLE_BYTES)()
        self._ck(self._l.dsgd_xchg_export(self._h, C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def xchg_import(self, peer_rank: int, handle: bytes):
        buf = (C.c_uint8 * IPC_HANDLE_BYTES).from_buffer_copy(handle)
        self._ck(self._l.dsgd_xchg_import(self._h, peer_rank, C.cast(buf, C.c_void_p)))

    def xchg_attach(self, peer_rank: int, peer: "NativeCtx"):
        self._ck(self._l.dsgd_xchg_attach(self._h, peer_rank, peer._h))

    def setup_peer_exchange(self, group) -> None:
        """One process per GPU: swap exchange-block handles through the process group and map every peer's block
        (the fused multi-GPU sync step then needs no NCCL)."""
        handles = group.all_gather_bytes(self.xchg_export())
        for r, h in enumerate(handles):
            if r != self.rank:
                self.xchg_import(r, h)
        group.barrier()

    def xchg_stats(self) -> Tuple[int, int, int]:
        """(value words, bitmap words) this rank stored into EACH peer so far, and the SGD steps of those launches."""
        v, b, n = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self._l.dsgd_xchg_stats(self._h, C.byref(v), C.byref(b), C.byref(n)))
        return v.value, b.value, n.value

    def reserve(self, n_samples: int, n_steps: int):
        """Allocate the sync path's device buffers now (see dsgd_reserve: needed when several ctxs share one GPU)."""
        self._ck(self._l.dsgd_reserve(self._h, n_samples, n_steps))

    def set_grid_limit(self, n_ctas: int):
        """CTAs of the persistent sync kernel (0: one per SM) -- lets several ranks share one GPU in tests."""
        self._ck(self._l.dsgd_set_grid_limit(self._h, n_ctas))

    TIMELINE_WORDS = 256 * 16 + 4 * 160 * 4

    def debug_timeline(self) -> np.ndarray:
        """Phase stamps of the last persistent launch (needs DSGD_PERSIST_TIMELINE in the environment)."""
        out = np.zeros(self.TIMELINE_WORDS, dtype=np.int64)
        self._ck(self._l.dsgd_debug_timeline(self._h, _ptr(out)))
        return out

    def sync_step(self, samples, lr: float, want_loss: bool = True):
        samples = _arr(samples, np.int32)
        loss = C.c_double()
        self._ck(self._l.dsgd_sync_step(self._h, _ptr(samples), samples.size, lr, C.byref(loss) if want_loss else None))
        return loss.value if want_loss else None

    def sync_steps(self, samples, n_per_step: int, n_steps: int, lr: float, want_losses: bool = True):
        samples = _arr(samples, np.int32, n_per_step * n_steps, "samples")
        losses = np.zeros(n_steps, dtype=np.float64) if want_losses else None
        self._ck(self._l.dsgd_sync_steps(self._h, _ptr(samples), n_per_step, n_steps, lr, _ptr(losses)))
        return losses

    def stage_samples(self, samples):
        samples = _arr(samples, np.int32)
        self._ck(self._l.dsgd_stage_samples(self._h, _ptr(samples), samples.size))

    def sync_steps_staged(self, first: int, n_per_step: int, n_steps: int, lr: float, want_losses: bool = False):
        self._ck(self._l.dsgd_sync_steps_staged(self._h, first, n_per_step, n_steps, lr, 1 if want_losses else 0))

    def read_losses(self, n_steps: int) -> np.ndarray:
        out = np.zeros(n_steps, dtype=np.float64)
        self._ck(self._l.dsgd_read_losses(self._h, _ptr(out), n_steps))
        return out

    # -- model sets: several (lambda, learning rate) settings trained on the same draws --
    def models_set(self, lambdas, learning_rates, w0=None):
        """Replace the model set (an empty one frees it).  w0: [n_models, dim] or [dim] for all, or None (zeros)."""
        lam = _arr(lambdas, np.float64)
        lr = _arr(learning_rates, np.float64, lam.size, "learning_rates")
        if w0 is not None:
            w0 = np.asarray(w0, dtype=np.float64)
            if w0.ndim == 1:
                w0 = np.tile(_arr(w0, np.float64, self.dim, "weights"), lam.size)
            w0 = _arr(w0, np.float64, lam.size * self.dim, "weights")
        self._ck(self._l.dsgd_models_set(self._h, lam.size, _ptr(lam), _ptr(lr), _ptr(w0)))
        self.n_models = lam.size

    def models_shape(self) -> Tuple[int, int]:
        n, d = C.c_int32(), C.c_int32()
        self._ck(self._l.dsgd_models_shape(self._h, C.byref(n), C.byref(d)))
        return n.value, d.value

    def models_get_weights(self) -> np.ndarray:
        """[n_models, dim] resident weights of the set."""
        n, d = self.models_shape()
        out = np.zeros(n * d, dtype=np.float64)
        self._ck(self._l.dsgd_models_get_weights(self._h, _ptr(out)))
        return out.reshape(n, d)

    def models_steps(self, samples, n_per_step: int, n_steps: int, active=None, want_losses: bool = True):
        """n_steps steps of every active model on the same samples; returns [n_steps, n_models] losses (NaN: frozen)."""
        n, _ = self.models_shape()
        samples = _arr(samples, np.int32, n_per_step * n_steps, "samples")
        act = None if active is None else _arr(np.asarray(active, dtype=bool), np.uint8, n, "active")
        losses = np.zeros(n_steps * n, dtype=np.float64) if want_losses else None
        self._ck(self._l.dsgd_models_steps(self._h, _ptr(samples), n_per_step, n_steps, _ptr(act), _ptr(losses)))
        return None if losses is None else losses.reshape(n_steps, n)

    def models_eval_counts(self, m: int, row_begin: int, row_end: int) -> Tuple[int, int, float]:
        """eval_counts for model m's resident weights."""
        h, c, n2 = C.c_int64(), C.c_int64(), C.c_double()
        self._ck(self._l.dsgd_models_eval_counts(self._h, m, row_begin, row_end, C.byref(h), C.byref(c), C.byref(n2)))
        return h.value, c.value, n2.value

    # -- async --
    def async_host_master(self, w0):
        """Host the master's replica (GradState.grad + update counter) on this GPU."""
        w0 = _arr(w0, np.float64, self.dim, "weights")
        self._ck(self._l.dsgd_async_host_master(self._h, _ptr(w0)))

    def ipc_export(self, which: int = REPLICA_SELF) -> bytes:
        buf = (C.c_uint8 * IPC_HANDLE_BYTES)()
        self._ck(self._l.dsgd_ipc_export(self._h, which, C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def peer_attach(self, peer_rank: int, peer: "NativeCtx", which: int = REPLICA_SELF):
        """Same-process peer (several ctxs driven by one host process)."""
        self._ck(self._l.dsgd_peer_attach(self._h, peer_rank, peer._h, which))

    def async_replay(self, w0, samples, batch: int, lr: float):
        w0 = _arr(w0, np.float64, self.dim, "weights")
        samples = _arr(samples, np.int32)
        if samples.size % batch:
            raise DsgdInvalid(ERR_INVALID, "async_replay: len(samples) is not a multiple of batch")
        self._ck(self._l.dsgd_async_replay(self._h, _ptr(w0), _ptr(samples), batch, samples.size // batch, lr))

    def async_running(self) -> bool:
        r = C.c_int()
        self._ck(self._l.dsgd_async_running(self._h, C.byref(r)))
        return bool(r.value)

    def async_elapsed_ms(self) -> float:
        ms = C.c_float()
        self._ck(self._l.dsgd_async_elapsed_ms(self._h, C.byref(ms)))
        return ms.value

    def async_master_weights(self) -> np.ndarray:
        out = np.zeros(self.dim, dtype=np.float64)
        self._ck(self._l.dsgd_async_master_weights(self._h, _ptr(out)))
        return out

    def async_outbox_enable(self):
        """One more target of every delta of this worker: the accumulator a host relay forwards to colleagues that are not GPU
        peers (core/Slave.scala:104-105).  Call before start_async."""
        self._ck(self._l.dsgd_async_outbox_enable(self._h))

    def async_outbox_read(self) -> np.ndarray:
        """Sum of -delta since async_outbox_enable (safe while the loop runs)."""
        out = np.zeros(self.dim, dtype=np.float64)
        self._ck(self._l.dsgd_async_outbox_read(self._h, _ptr(out)))
        return out

    def ipc_import(self, peer_rank: int, handle: bytes):
        buf = (C.c_uint8 * IPC_HANDLE_BYTES).from_buffer_copy(handle)
        self._ck(self._l.dsgd_ipc_import(self._h, peer_rank, C.cast(buf, C.c_void_p)))

    def start_async(self, w0, assigned, batch: int, lr: float, concurrency: int = 1, max_updates: int = 0, seed: int = 0):
        w0 = None if w0 is None else _arr(w0, np.float64, self.dim, "weights")
        assigned = _arr(assigned, np.int32)
        self._ck(self._l.dsgd_start_async(self._h, _ptr(w0), _ptr(assigned), assigned.size, batch, lr, concurrency,
                                          max_updates, seed))

    def stop_async(self):
        self._ck(self._l.dsgd_stop_async(self._h))

    def update_grad(self, idx, val):
        idx, val = _arr(idx, np.int32), _arr(val, np.float64)
        if idx.size != val.size:
            raise DsgdInvalid(ERR_INVALID, "update_grad: idx and val differ in length")
        self._ck(self._l.dsgd_update_grad(self._h, _ptr(idx), _ptr(val), idx.size))

    def async_updates(self) -> int:
        n = C.c_int64()
        self._ck(self._l.dsgd_async_updates(self._h, C.byref(n)))
        return n.value
