"""ctypes binding of the C ABI in include/machineboss_b200.h.

This is plumbing for tests, bench.py and the Python convenience layer; the product is the shared
library.  There is no fallback: if the library is missing it is built with nvcc, and if that
fails, or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

from . import build as _build

ENGINE_GENERIC, ENGINE_JIT, ENGINE_WIDE = 0, 1, 2

_lib = None

# every symbol include/machineboss_b200.h declares
SYMBOLS = ["mb_last_error", "mb_version", "mb_set_kernel_cache_dir", "mb_device_count", "mb_set_device", "mb_set_engine", "mb_set_option", "mb_machine_set_option",
           "mb_machine_create", "mb_machine_update_weights", "mb_machine_info", "mb_machine_destroy",
           "mb_batch_create", "mb_batch_destroy", "mb_batch_trim", "mb_batch_set_envelopes", "mb_forward", "mb_backward", "mb_viterbi",
           "mb_viterbi_paths", "mb_viterbi_paths_narrow", "mb_viterbi_paths_start", "mb_batch_wait", "mb_counts", "mb_matrix", "mb_last_kernel_ms", "mb_last_redo", "mb_jit_compile_check", "mb_jit_host_tables", "mb_lane_emulate", "mb_col_emulate",
           "mb_shard_pairs", "mb_group_create", "mb_group_info", "mb_group_destroy", "mb_group_machine_create", "mb_group_machine_update_weights",
           "mb_group_machine_set_option", "mb_group_machine_info", "mb_group_machine_destroy", "mb_group_batch_create", "mb_group_batch_set_envelopes",
           "mb_group_batch_shard", "mb_group_batch_destroy", "mb_group_forward", "mb_group_backward", "mb_group_viterbi", "mb_group_viterbi_paths",
           "mb_group_viterbi_paths_narrow", "mb_group_counts", "mb_group_last_loglike", "mb_group_last_kernel_ms"]


class MachineBossError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        path = _build.build()
        L = ctypes.CDLL(path)
        P, I32, I64, D = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double
        L.mb_last_error.restype = ctypes.c_char_p
        L.mb_last_error.argtypes = []
        L.mb_version.restype = ctypes.c_int
        L.mb_set_kernel_cache_dir.argtypes = [ctypes.c_char_p]
        L.mb_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
        L.mb_set_device.argtypes = [ctypes.c_int]
        L.mb_set_engine.argtypes = [ctypes.c_int]
        L.mb_set_option.argtypes = [ctypes.c_char_p, I32]
        L.mb_machine_set_option.argtypes = [P, ctypes.c_char_p, I32]
        L.mb_machine_create.argtypes = [ctypes.POINTER(P), I32, I32, I32, I64, P, P, P, P, P]
        L.mb_machine_update_weights.argtypes = [P, P]
        L.mb_machine_info.argtypes = [P, ctypes.POINTER(I32), ctypes.POINTER(I64), ctypes.POINTER(I32)]
        L.mb_machine_destroy.argtypes = [P]
        L.mb_machine_destroy.restype = None
        L.mb_batch_create.argtypes = [ctypes.POINTER(P), I64, P, P, P, P]
        L.mb_batch_destroy.argtypes = [P]
        L.mb_batch_destroy.restype = None
        L.mb_batch_trim.argtypes = [P]
        L.mb_batch_set_envelopes.argtypes = [P, P, P, P]
        L.mb_forward.argtypes = [P, P, P]
        L.mb_backward.argtypes = [P, P, P]
        L.mb_viterbi.argtypes = [P, P, P, P]
        L.mb_viterbi_paths.argtypes = [P, P, P]
        L.mb_viterbi_paths_narrow.argtypes = [P, P, I32, P]
        L.mb_viterbi_paths_start.argtypes = [P, P, I32, P]
        L.mb_batch_wait.argtypes = [P]
        L.mb_counts.argtypes = [P, P, P, P]
        L.mb_matrix.argtypes = [P, P, I64, I32, P]
        L.mb_jit_compile_check.argtypes = [I32, I32, I32, I64, P, P, P, P, ctypes.c_char_p, I64]
        L.mb_jit_host_tables.argtypes = [I32, I32, I32, I64, P, P, P, P, P, I32, P, I64, ctypes.POINTER(I64)]
        L.mb_lane_emulate.argtypes = [I32, I32, I32, I64, P, P, P, P, P, P, I64, I32, ctypes.POINTER(D), P, P]
        L.mb_col_emulate.argtypes = [I32, I32, I32, I64, P, P, P, P, P, P, I64, I32, ctypes.POINTER(D), P, ctypes.c_char_p, I64, P, I64, ctypes.POINTER(I64)]
        L.mb_last_redo.argtypes = [P, ctypes.POINTER(I64)]
        L.mb_last_kernel_ms.argtypes = [P, ctypes.POINTER(D), ctypes.POINTER(I64)]
        L.mb_shard_pairs.argtypes = [I64, P, P, I32, P]
        L.mb_group_create.argtypes = [ctypes.POINTER(P), P, I32]
        L.mb_group_info.argtypes = [P, ctypes.POINTER(I32), P, ctypes.POINTER(I32)]
        L.mb_group_destroy.argtypes = [P]
        L.mb_group_destroy.restype = None
        L.mb_group_machine_create.argtypes = [P, ctypes.POINTER(P), I32, I32, I32, I64, P, P, P, P, P]
        L.mb_group_machine_update_weights.argtypes = [P, P]
        L.mb_group_machine_set_option.argtypes = [P, ctypes.c_char_p, I32]
        L.mb_group_machine_info.argtypes = [P, ctypes.POINTER(I32), ctypes.POINTER(I64), ctypes.POINTER(I32)]
        L.mb_group_machine_destroy.argtypes = [P]
        L.mb_group_machine_destroy.restype = None
        L.mb_group_batch_create.argtypes = [P, ctypes.POINTER(P), I64, P, P, P, P]
        L.mb_group_batch_set_envelopes.argtypes = [P, P, P, P]
        L.mb_group_batch_shard.argtypes = [P, P, P]
        L.mb_group_batch_destroy.argtypes = [P]
        L.mb_group_batch_destroy.restype = None
        L.mb_group_forward.argtypes = [P, P, P]
        L.mb_group_backward.argtypes = [P, P, P]
        L.mb_group_viterbi.argtypes = [P, P, P, P]
        L.mb_group_viterbi_paths.argtypes = [P, P, P]
        L.mb_group_viterbi_paths_narrow.argtypes = [P, P, I32, P]
        L.mb_group_counts.argtypes = [P, P, P, P]
        L.mb_group_last_loglike.argtypes = [P, ctypes.POINTER(D)]
        L.mb_group_last_kernel_ms.argtypes = [P, ctypes.POINTER(D), ctypes.POINTER(I64)]
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise MachineBossError(lib().mb_last_error().decode())


def device_count() -> int:
    n = ctypes.c_int(0)
    _check(lib().mb_device_count(ctypes.byref(n)))
    return n.value


def set_device(d: int) -> None:
    _check(lib().mb_set_device(d))


def set_engine(e: int) -> None:
    _check(lib().mb_set_engine(e))


OPTION_UNSET = -2147483648


def set_kernel_cache_dir(path) -> None:
    """Keep / look up the run-time compiled modules in this directory (None: no cache)."""
    _check(lib().mb_set_kernel_cache_dir(path.encode() if path else None))


def set_option(name: str, value) -> None:
    """Default of a tuning knob for machines this thread creates afterwards (None: the built-in choice)."""
    _check(lib().mb_set_option(name.encode(), OPTION_UNSET if value is None else int(value)))


def jit_compile_check(n_states, n_in, n_out, src, dst, tin, tout) -> str:
    """NVRTC-compile the specialised kernels of a machine structure (no device needed); returns the log."""
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
    buf = ctypes.create_string_buffer(1 << 16)
    _check(lib().mb_jit_compile_check(int(n_states), int(n_in), int(n_out), int(arrs[0].shape[0]),
                                      *[_ptr(a) for a in arrs], buf, len(buf)))
    return buf.value.decode()


def jit_host_tables(n_states, n_in, n_out, src, dst, tin, tout, log_weight, which: int) -> np.ndarray:
    """The tables the generated score kernels read for these weights (no device needed); see mb_jit_host_tables."""
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
    lw = np.ascontiguousarray(log_weight, dtype=np.float64)
    n = ctypes.c_int64(0)
    _check(lib().mb_jit_host_tables(int(n_states), int(n_in), int(n_out), int(lw.shape[0]), *[_ptr(a) for a in arrs], _ptr(lw), int(which), None, 0, ctypes.byref(n)))
    out = np.zeros(max(n.value, 1), dtype=np.float64)
    _check(lib().mb_jit_host_tables(int(n_states), int(n_in), int(n_out), int(lw.shape[0]), *[_ptr(a) for a in arrs], _ptr(lw), int(which), out.ctypes.data, n.value, ctypes.byref(n)))
    return out[: n.value]


def lane_emulate(n_states, n_in, n_out, src, dst, tin, tout, log_weight, y, op: int, back_pointers: bool = False):
    """The lane engine's windowed program run for one read on the host; returns (result, info[8][, back-pointers])."""
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
    lw = np.ascontiguousarray(log_weight, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.uint8)
    res = ctypes.c_double(0)
    info = np.zeros(8, dtype=np.int32)
    bp = np.zeros((len(y) + 1) * int(n_states), dtype=np.uint32) if back_pointers else None
    _check(lib().mb_lane_emulate(int(n_states), int(n_in), int(n_out), int(lw.shape[0]), *[_ptr(a) for a in arrs], _ptr(lw),
                                 _ptr(y), len(y), int(op), ctypes.byref(res), info.ctypes.data, bp.ctypes.data if back_pointers else None))
    return (res.value, info, bp) if back_pointers else (res.value, info)


def col_emulate(n_states, n_in, n_out, src, dst, tin, tout, log_weight, y, op: int, compile_log: bool = False, path: bool = False):
    """The column engine's program for a periodic generator run for one read on the host; returns (result, info[12][, NVRTC log]
    [, Viterbi path]).  info[0] == 0: the machine has no such structure (result is meaningless)."""
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
    lw = np.ascontiguousarray(log_weight, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.uint8)
    res = ctypes.c_double(0)
    info = np.zeros(12, dtype=np.int32)
    buf = ctypes.create_string_buffer(1 << 16) if compile_log else None
    ids = np.zeros(4 * (len(y) + 1) + 4 * int(n_states), dtype=np.int32) if path else None
    n_ids = ctypes.c_int64(0)
    _check(lib().mb_col_emulate(int(n_states), int(n_in), int(n_out), int(lw.shape[0]), *[_ptr(a) for a in arrs], _ptr(lw),
                                _ptr(y), len(y), int(op), ctypes.byref(res), info.ctypes.data, buf, len(buf) if compile_log else 0,
                                ids.ctypes.data if path else None, len(ids) if path else 0, ctypes.byref(n_ids) if path else None))
    out = (res.value, info)
    if compile_log:
        out += (buf.value.decode(),)
    if path:
        assert n_ids.value <= len(ids)
        out += (ids[: n_ids.value].copy(),)
    return out


def _ptr(a):
    return a.ctypes.data if a is not None and a.size else None


class Machine:
    """Handle on a flattened EvaluatedMachine (src/eval.h:78-98) living on the device."""

    def __init__(self, n_states, n_in, n_out, src, dst, tin, tout, log_weight):
        self.n_states, self.n_in, self.n_out = int(n_states), int(n_in), int(n_out)
        arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
        lw = np.ascontiguousarray(log_weight, dtype=np.float64)
        self.n_trans = int(lw.shape[0])
        self.h = ctypes.c_void_p()
        _check(lib().mb_machine_create(ctypes.byref(self.h), self.n_states, self.n_in, self.n_out, self.n_trans,
                                       *[_ptr(a) for a in arrs], _ptr(lw)))

    @property
    def engine(self) -> int:
        e = ctypes.c_int32(0)
        _check(lib().mb_machine_info(self.h, None, None, ctypes.byref(e)))
        return e.value

    def set_option(self, name: str, value) -> None:
        _check(lib().mb_machine_set_option(self.h, name.encode(), OPTION_UNSET if value is None else int(value)))

    def update_weights(self, log_weight) -> None:
        lw = np.ascontiguousarray(log_weight, dtype=np.float64)
        assert lw.shape[0] == self.n_trans
        _check(lib().mb_machine_update_weights(self.h, _ptr(lw)))

    def close(self):
        if self.h:
            lib().mb_machine_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """Handle on a tokenised SeqPairList (src/seqpair.h:115-121) living on the device."""

    def __init__(self, pairs=None, *, x=None, x_off=None, y=None, y_off=None):
        if pairs is not None:
            xs = [np.asarray(p[0], dtype=np.uint8) for p in pairs]
            ys = [np.asarray(p[1], dtype=np.uint8) for p in pairs]
            x = np.concatenate(xs) if xs else np.zeros(0, np.uint8)
            y = np.concatenate(ys) if ys else np.zeros(0, np.uint8)
            x_off = np.concatenate([[0], np.cumsum([len(a) for a in xs])]).astype(np.int64)
            y_off = np.concatenate([[0], np.cumsum([len(a) for a in ys])]).astype(np.int64)
        self.x = np.ascontiguousarray(x, dtype=np.uint8)
        self.y = np.ascontiguousarray(y, dtype=np.uint8)
        self.x_off = np.ascontiguousarray(x_off, dtype=np.int64)
        self.y_off = np.ascontiguousarray(y_off, dtype=np.int64)
        self.n_pairs = int(self.x_off.shape[0]) - 1
        self.h = ctypes.c_void_p()
        _check(lib().mb_batch_create(ctypes.byref(self.h), self.n_pairs, _ptr(self.x), _ptr(self.x_off),
                                     _ptr(self.y), _ptr(self.y_off)))

    def set_envelopes(self, envs) -> None:
        """envs: per pair None (full matrix) or a list of [inStart, inEnd) per output row (Lo+1 rows);
        envs=None removes all envelopes (Envelope, src/seqpair.h:75-113)."""
        if envs is None:
            _check(lib().mb_batch_set_envelopes(self.h, None, None, None))
            return
        assert len(envs) == self.n_pairs
        rows = [np.asarray(e, dtype=np.int64).reshape(-1, 2) if e is not None else np.zeros((0, 2), np.int64) for e in envs]
        off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
        allr = np.concatenate(rows) if rows else np.zeros((0, 2), np.int64)
        st = np.ascontiguousarray(allr[:, 0]) if len(allr) else np.zeros(1, np.int64)
        en = np.ascontiguousarray(allr[:, 1]) if len(allr) else np.zeros(1, np.int64)
        _check(lib().mb_batch_set_envelopes(self.h, off.ctypes.data, st.ctypes.data, en.ctypes.data))

    def cell_states(self, n_states: int) -> float:
        li = np.diff(self.x_off).astype(np.float64)
        lo = np.diff(self.y_off).astype(np.float64)
        return float(((li + 1) * (lo + 1)).sum() * n_states)

    def last_redo(self) -> int:
        n = ctypes.c_int64(0)
        _check(lib().mb_last_redo(self.h, ctypes.byref(n)))
        return n.value

    def trim(self):
        _check(lib().mb_batch_trim(self.h))

    def wait(self):
        _check(lib().mb_batch_wait(self.h))

    def last_kernel_ms(self):
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        _check(lib().mb_last_kernel_ms(self.h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    def close(self):
        if self.h:
            lib().mb_batch_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def forward(m: Machine, b: Batch) -> np.ndarray:
    out = np.empty(b.n_pairs, dtype=np.float64)
    _check(lib().mb_forward(m.h, b.h, _ptr(out)))
    return out


def backward(m: Machine, b: Batch) -> np.ndarray:
    out = np.empty(b.n_pairs, dtype=np.float64)
    _check(lib().mb_backward(m.h, b.h, _ptr(out)))
    return out


def viterbi_lengths(m: Machine, b: Batch):
    """Viterbi scores + traceback on the device; returns (score, path lengths), paths stay on the device."""
    score = np.empty(b.n_pairs, dtype=np.float64)
    plen = np.zeros(b.n_pairs, dtype=np.int64)
    _check(lib().mb_viterbi(m.h, b.h, _ptr(score), _ptr(plen)))
    return score, plen


def viterbi(m: Machine, b: Batch, paths: bool = True, packed: bool = False):
    """ViterbiMatrix::logLike (+ ::path).  paths: list of int32 arrays of global transition ids,
    or with packed=True the pair (all ids concatenated, offsets[nPairs+1])."""
    if not paths:
        score = np.empty(b.n_pairs, dtype=np.float64)
        _check(lib().mb_viterbi(m.h, b.h, _ptr(score), None))
        return score
    score, plen = viterbi_lengths(m, b)
    trans, off = viterbi_paths(b, plen)
    if packed:
        return score, (trans, off)
    return score, [trans[off[k]:off[k + 1]] for k in range(b.n_pairs)]


def viterbi_paths(b: Batch, plen: np.ndarray):
    """The paths of the batch's last Viterbi call (path lengths `plen`), copied from the device: (all ids
    concatenated as int32, offsets[nPairs+1])."""
    off = np.concatenate([[0], np.cumsum(plen)]).astype(np.int64)
    trans = np.empty(int(off[-1]), dtype=np.int32)
    if off[-1]:
        _check(lib().mb_viterbi_paths(b.h, _ptr(trans), _ptr(off)))
    return trans, off


def forward_into(m: Machine, b: Batch, out: np.ndarray) -> None:
    """mb_forward into a caller-owned float64 array (e.g. a view of pinned memory)."""
    assert out.dtype == np.float64 and out.size >= b.n_pairs and out.flags["C_CONTIGUOUS"]
    _check(lib().mb_forward(m.h, b.h, _ptr(out)))


def viterbi_into(m: Machine, b: Batch, score: np.ndarray, plen: np.ndarray, off: np.ndarray, trans: np.ndarray) -> int:
    """mb_viterbi + mb_viterbi_paths into caller-owned arrays; returns the total path length.

    score float64[nPairs], plen int64[nPairs], off int64[nPairs+1] (filled here), trans int32 / uint16 / uint8 [capacity]."""
    _check(lib().mb_viterbi(m.h, b.h, _ptr(score), _ptr(plen)))
    off[0] = 0
    np.cumsum(plen[: b.n_pairs], out=off[1: b.n_pairs + 1])
    total = int(off[b.n_pairs])
    if total > trans.size:
        raise MachineBossError("viterbi_into: path buffer too small (%d > %d)" % (total, trans.size))
    if total:
        if trans.dtype == np.int32:
            _check(lib().mb_viterbi_paths(b.h, _ptr(trans), _ptr(off)))
        else:      # uint8 / uint16 ids (machines with at most 256 / 65 536 transitions)
            assert trans.dtype in (np.uint8, np.uint16)
            _check(lib().mb_viterbi_paths_narrow(b.h, _ptr(trans), trans.dtype.itemsize, _ptr(off)))
    return total


def viterbi_start(m: Machine, b: Batch, score: np.ndarray, plen: np.ndarray, off: np.ndarray, trans: np.ndarray) -> int:
    """viterbi_into without waiting for the paths: they are on their way into `trans` (page-locked memory) when this
    returns, other calls on the batch may follow, and b.wait() returns once they have arrived."""
    _check(lib().mb_viterbi(m.h, b.h, _ptr(score), _ptr(plen)))
    off[0] = 0
    np.cumsum(plen[: b.n_pairs], out=off[1: b.n_pairs + 1])
    total = int(off[b.n_pairs])
    if total > trans.size:
        raise MachineBossError("viterbi_start: path buffer too small (%d > %d)" % (total, trans.size))
    if total:
        _check(lib().mb_viterbi_paths_start(b.h, _ptr(trans), trans.dtype.itemsize, _ptr(off)))
    return total


def matrix(m: Machine, b: Batch, pair: int, kind: int = 0) -> np.ndarray:
    """DPMatrix cells of one pair, shape (outLen+1, inLen+1, nStates); kind 0 Forward, 1 Backward, 2 Viterbi."""
    li = int(b.x_off[pair + 1] - b.x_off[pair])
    lo = int(b.y_off[pair + 1] - b.y_off[pair])
    out = np.empty((lo + 1, li + 1, m.n_states), dtype=np.float64)
    _check(lib().mb_matrix(m.h, b.h, int(pair), int(kind), _ptr(out)))
    return out


def counts(m: Machine, b: Batch):
    c = np.zeros(m.n_trans, dtype=np.float64)
    ll = np.empty(b.n_pairs, dtype=np.float64)
    _check(lib().mb_counts(m.h, b.h, _ptr(c), _ptr(ll)))
    return c, ll


# ---------------------------------------------------------------------------------------------
# several GPUs of one box (mb_group_*): the list dealt to the devices, one host thread per device
# ---------------------------------------------------------------------------------------------
def shard_pairs(x_off, y_off, n_shards: int) -> np.ndarray:
    """Shard (0 .. n_shards-1) of every pair under the library's longest-processing-time-first deal by cell count."""
    x_off = np.ascontiguousarray(x_off, dtype=np.int64)
    y_off = np.ascontiguousarray(y_off, dtype=np.int64)
    n = int(x_off.shape[0]) - 1
    out = np.zeros(max(n, 1), dtype=np.int32)
    _check(lib().mb_shard_pairs(n, _ptr(x_off), _ptr(y_off), int(n_shards), out.ctypes.data))
    return out[:n]


class Group:
    def __init__(self, devices=None):
        self.h = ctypes.c_void_p()
        if devices is None:
            _check(lib().mb_group_create(ctypes.byref(self.h), None, 0))
        else:
            d = np.ascontiguousarray(devices, dtype=np.int32)
            _check(lib().mb_group_create(ctypes.byref(self.h), d.ctypes.data, int(d.shape[0])))
        n, nccl = ctypes.c_int32(0), ctypes.c_int32(0)
        _check(lib().mb_group_info(self.h, ctypes.byref(n), None, ctypes.byref(nccl)))
        self.n_devices, self.uses_nccl = n.value, bool(nccl.value)

    def close(self):
        if self.h:
            lib().mb_group_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GroupMachine:
    def __init__(self, group: Group, n_states, n_in, n_out, src, dst, tin, tout, log_weight):
        self.group = group
        self.n_states, self.n_in, self.n_out = int(n_states), int(n_in), int(n_out)
        arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (src, dst, tin, tout)]
        lw = np.ascontiguousarray(log_weight, dtype=np.float64)
        self.n_trans = int(lw.shape[0])
        self.h = ctypes.c_void_p()
        _check(lib().mb_group_machine_create(group.h, ctypes.byref(self.h), self.n_states, self.n_in, self.n_out, self.n_trans,
                                             *[_ptr(a) for a in arrs], _ptr(lw)))

    def update_weights(self, log_weight) -> None:
        lw = np.ascontiguousarray(log_weight, dtype=np.float64)
        _check(lib().mb_group_machine_update_weights(self.h, _ptr(lw)))

    def last_loglike(self) -> float:
        v = ctypes.c_double(0)
        _check(lib().mb_group_last_loglike(self.h, ctypes.byref(v)))
        return v.value

    def close(self):
        if self.h:
            lib().mb_group_machine_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GroupBatch:
    def __init__(self, group: Group, pairs=None, *, x=None, x_off=None, y=None, y_off=None):
        self.group = group
        if pairs is not None:
            xs = [np.asarray(p[0], dtype=np.uint8) for p in pairs]
            ys = [np.asarray(p[1], dtype=np.uint8) for p in pairs]
            x = np.concatenate(xs) if xs else np.zeros(0, np.uint8)
            y = np.concatenate(ys) if ys else np.zeros(0, np.uint8)
            x_off = np.concatenate([[0], np.cumsum([len(a) for a in xs])]).astype(np.int64)
            y_off = np.concatenate([[0], np.cumsum([len(a) for a in ys])]).astype(np.int64)
        self.x = np.ascontiguousarray(x, dtype=np.uint8)
        self.y = np.ascontiguousarray(y, dtype=np.uint8)
        self.x_off = np.ascontiguousarray(x_off, dtype=np.int64)
        self.y_off = np.ascontiguousarray(y_off, dtype=np.int64)
        self.n_pairs = int(self.x_off.shape[0]) - 1
        self.h = ctypes.c_void_p()
        _check(lib().mb_group_batch_create(group.h, ctypes.byref(self.h), self.n_pairs, _ptr(self.x), _ptr(self.x_off), _ptr(self.y), _ptr(self.y_off)))

    def shard(self):
        dev = np.zeros(max(self.n_pairs, 1), dtype=np.int32)
        cells = np.zeros(self.group.n_devices, dtype=np.float64)
        _check(lib().mb_group_batch_shard(self.h, dev.ctypes.data, cells.ctypes.data))
        return dev[: self.n_pairs], cells

    def last_kernel_ms(self):
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        _check(lib().mb_group_last_kernel_ms(self.h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    def close(self):
        if self.h:
            lib().mb_group_batch_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def group_forward(m: GroupMachine, b: GroupBatch) -> np.ndarray:
    out = np.empty(max(b.n_pairs, 1), dtype=np.float64)
    _check(lib().mb_group_forward(m.h, b.h, out.ctypes.data))
    return out[: b.n_pairs]


def group_viterbi(m: GroupMachine, b: GroupBatch):
    score = np.empty(max(b.n_pairs, 1), dtype=np.float64)
    plen = np.zeros(max(b.n_pairs, 1), dtype=np.int64)
    _check(lib().mb_group_viterbi(m.h, b.h, score.ctypes.data, plen.ctypes.data))
    off = np.concatenate([[0], np.cumsum(plen[: b.n_pairs])]).astype(np.int64)
    trans = np.empty(max(int(off[-1]), 1), dtype=np.int32)
    if off[-1]:
        _check(lib().mb_group_viterbi_paths(b.h, trans.ctypes.data, off.ctypes.data))
    return score[: b.n_pairs], [trans[off[k]:off[k + 1]] for k in range(b.n_pairs)]


def group_counts(m: GroupMachine, b: GroupBatch):
    c = np.zeros(max(m.n_trans, 1), dtype=np.float64)
    ll = np.empty(max(b.n_pairs, 1), dtype=np.float64)
    _check(lib().mb_group_counts(m.h, b.h, c.ctypes.data, ll.ctypes.data))
    return c[: m.n_trans], ll[: b.n_pairs]
