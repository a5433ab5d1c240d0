"""Host-side mirror of the reference interface, over the C ABI (``include/sdpa_b200.h``).

The reference is a C program whose whole operator API is one function,
``attention(Q, K, V, result, m, n, dk, dv, mpi_rank, mpi_size)``
(``attention-mpi.c:191-192``), plus the helpers it is built from.  This module binds
the shared library with ``ctypes`` and mirrors those names and argument meanings so the
parity tests read like calls into the reference:

* :func:`attention` -- the drop-in entry point on NumPy fp64 arrays;
* :func:`owner_count` / :func:`owner_disp` -- ``attention-mpi.c:19-27``;
* :func:`cvt_d2f` / :func:`cvt_f2d` -- ``attention-mpi.c:31-101`` (device casts);
* :func:`online_softmax_partials` -- the contract of ``online_softmax_attention``
  (``attention-mpi.c:168-189``) over a batch of rows;
* :class:`Context` -- resident K/V shards + the ping-pong Q-batch loop
  (``attention-mpi.c:268-399``), one process per GPU or one process for several.

There is no CPU fallback: if ``libsdpa_b200.so`` is missing the import of the library
fails loudly, and every compute call fails without a CUDA device.
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libsdpa_b200.so"

PREC_AUTO, PREC_F32, PREC_BF16, PREC_BF16X3 = 0, 1, 2, 3
MERGE_NCCL, MERGE_PEER, MERGE_NCCL2 = 0, 1, 2
_MERGE = {"nccl": MERGE_NCCL2, "nccl2": MERGE_NCCL2, "nccl3": MERGE_NCCL, "peer": MERGE_PEER}
DIST_KV, DIST_Q, DIST_AUTO = 0, 1, 2
DTYPE_F64, DTYPE_F32, DTYPE_BF16 = 0, 1, 2
_DTYPE = {"f64": DTYPE_F64, "fp64": DTYPE_F64, "float64": DTYPE_F64, "f32": DTYPE_F32, "fp32": DTYPE_F32, "float32": DTYPE_F32,
          "bf16": DTYPE_BF16, "bfloat16": DTYPE_BF16}
_DIST = {"kv": DIST_KV, "q": DIST_Q, "auto": DIST_AUTO}
_PREC = {"auto": PREC_AUTO, "f32": PREC_F32, "fp32": PREC_F32, "bf16": PREC_BF16, "bf16x3": PREC_BF16X3, "f32x3": PREC_BF16X3}

_dp = ctypes.POINTER(ctypes.c_double)
_fp = ctypes.POINTER(ctypes.c_float)
_ip = ctypes.POINTER(ctypes.c_int)
_dpp = ctypes.POINTER(ctypes.c_void_p)


class SdpaError(RuntimeError):
    pass


class Config(ctypes.Structure):
    _fields_ = [
        ("precision", ctypes.c_int),
        ("q_batch", ctypes.c_int),
        ("kv_splits", ctypes.c_int),
        ("merge", ctypes.c_int),
        ("num_local", ctypes.c_int),
        ("first_device", ctypes.c_int),
        ("world_size", ctypes.c_int),
        ("rank_base", ctypes.c_int),
        ("distribution", ctypes.c_int),
        ("reserved", ctypes.c_int * 7),
    ]


# every symbol include/sdpa_b200.h declares: name -> (restype, argtypes)
_V = ctypes.c_void_p
ABI = {
    "attention": (None, [_V, _V, _V, _V] + [ctypes.c_int] * 6),
    "sdpa_runtime_init": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "sdpa_runtime_shutdown": (None, []),
    "sdpa_runtime_max": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double)]),
    "sdpa_owner_count": (ctypes.c_int, [ctypes.c_int] * 3),
    "sdpa_owner_disp": (ctypes.c_int, [ctypes.c_int] * 3),
    "sdpa_precision_supported": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_int)]),
    "sdpa_precision_supported_for": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_int)]),
    "sdpa_config_init": (None, [ctypes.POINTER(Config)]),
    "sdpa_ctx_create": (ctypes.c_int, [ctypes.POINTER(_V), ctypes.POINTER(Config), _V]),
    "sdpa_ctx_destroy": (ctypes.c_int, [_V]),
    "sdpa_get_unique_id": (ctypes.c_int, [_V]),
    "sdpa_set_bootstrap_id": (ctypes.c_int, [_V]),
    "sdpa_load_kv_host": (ctypes.c_int, [_V, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int]),
    "sdpa_load_kv_device": (ctypes.c_int, [_V, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int]),
    "sdpa_load_kv_host_full": (ctypes.c_int, [_V, _V, _V, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "sdpa_attention_host": (ctypes.c_int, [_V, _V, _V, ctypes.c_int]),
    "sdpa_attention_device": (ctypes.c_int, [_V, _dpp, _V, ctypes.c_int]),
    "sdpa_attention_device_full": (ctypes.c_int, [_V, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int, _dpp, _V, ctypes.c_int]),
    "sdpa_host_alloc": (ctypes.c_void_p, [ctypes.c_size_t]),
    "sdpa_host_free": (None, [_V]),
    "sdpa_host_copy": (ctypes.c_int, [_V, _V, ctypes.c_size_t]),
    "sdpa_enqueue_device_full": (ctypes.c_int, [_V, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int, _dpp, _V, ctypes.c_int]),
    "sdpa_synchronize": (ctypes.c_int, [_V]),
    "sdpa_attention_device_typed": (ctypes.c_int, [_V, ctypes.c_int, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int, _dpp, _V, ctypes.c_int]),
    "sdpa_enqueue_device_typed": (ctypes.c_int, [_V, ctypes.c_int, _dpp, _dpp, _ip, ctypes.c_int, ctypes.c_int, _dpp, _V, ctypes.c_int]),
    "sdpa_scatter_attention": (ctypes.c_int, [_V, _V, _V, _V, _V] + [ctypes.c_int] * 4),
    "sdpa_online_softmax_partials": (ctypes.c_int, [_V, ctypes.c_int, _V, ctypes.c_int, _V, _V, _V]),
    "sdpa_last_timings": (ctypes.c_int, [_V, _fp]),
    "sdpa_accumulated_timings": (ctypes.c_int, [_V, ctypes.POINTER(ctypes.c_double), ctypes.c_int]),
    "sdpa_last_kernel": (ctypes.c_char_p, [_V]),
    "sdpa_cvt_d2f": (ctypes.c_int, [_V, _V, ctypes.c_size_t, _V]),
    "sdpa_cvt_f2d": (ctypes.c_int, [_V, _V, ctypes.c_size_t, _V]),
    "sdpa_cvt_d2bf16": (ctypes.c_int, [_V, _V, ctypes.c_size_t, _V]),
    "sdpa_cvt_d2bf16x2": (ctypes.c_int, [_V, _V, _V, ctypes.c_size_t, _V]),
    "sdpa_last_error": (ctypes.c_char_p, []),
    "sdpa_version": (ctypes.c_char_p, []),
    "sdpa_device_count": (ctypes.c_int, []),
    "sdpa_launch_count": (ctypes.c_ulonglong, []),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load ``libsdpa_b200.so`` (raises if it has not been built -- no fallback)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise SdpaError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the attention path)")
        L = ctypes.CDLL(str(LIB_PATH), mode=ctypes.RTLD_GLOBAL)
        for name, (res, args) in ABI.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().sdpa_last_error().decode(errors="replace")
        raise SdpaError(f"{what} failed (status {status}): {msg}")


def device_count() -> int:
    return int(lib().sdpa_device_count())


def launch_count() -> int:
    return int(lib().sdpa_launch_count())


def version() -> str:
    return lib().sdpa_version().decode()


# ---------------------------------------------------------------------------
# shard map (attention-mpi.c:19-27)
# ---------------------------------------------------------------------------
def owner_count(n: int, size: int, rank: int) -> int:
    return int(lib().sdpa_owner_count(n, size, rank))


def owner_disp(n: int, size: int, rank: int) -> int:
    return int(lib().sdpa_owner_disp(n, size, rank))


def _as_f64(a, name: str) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.ndim != 2:
        raise ValueError(f"{name} must be a 2-D array")
    return a


# ---------------------------------------------------------------------------
# the reference entry point (attention-mpi.c:191-192)
# ---------------------------------------------------------------------------
def attention(Q, K, V, result=None, m=None, n=None, dk=None, dv=None, mpi_rank: int = 0, mpi_size: int = 1):
    """``attention(Q, K, V, result, m, n, dk, dv, mpi_rank, mpi_size)``.

    Q [m,dk], K [n,dk], V [n,dv] fp64 row-major; returns (and fills) result [m,dv] fp64.
    With ``mpi_size > 1`` only rank 0 passes arrays (others pass ``None`` and get ``None``),
    exactly like the reference (attention-mpi.c:508-517).  Precision / GPUs come from the
    environment (``SDPA_PRECISION``, ``SDPA_NGPUS``) as documented in ``include/sdpa_b200.h``.
    Fatal errors terminate the process, as the reference harness does.
    """
    L = lib()
    if mpi_rank == 0:
        Q, K, V = _as_f64(Q, "Q"), _as_f64(K, "K"), _as_f64(V, "V")
        m = Q.shape[0] if m is None else m
        dk = Q.shape[1] if dk is None else dk
        n = K.shape[0] if n is None else n
        dv = V.shape[1] if dv is None else dv
        if K.shape[1] != dk or V.shape[0] != n:
            raise ValueError("inconsistent Q/K/V shapes")
        if result is None:
            result = np.empty((m, dv), dtype=np.float64)
        if result.dtype != np.float64 or not result.flags.c_contiguous or result.size != m * dv:
            raise ValueError("result must be a C-contiguous fp64 array of m*dv elements")
        L.attention(Q.ctypes.data, K.ctypes.data, V.ctypes.data, result.ctypes.data, m, n, dk, dv, mpi_rank, mpi_size)
        return result
    L.attention(None, None, None, None, 0, 0, 0, 0, mpi_rank, mpi_size)
    return None


def precision_supported(precision, dk: int, dv: int):
    """(supported, resolved precision name) -- which kernel family a (precision, dk, dv) request lands on."""
    res = ctypes.c_int(-1)
    ok = lib().sdpa_precision_supported(_PREC[precision] if isinstance(precision, str) else int(precision), dk, dv, ctypes.byref(res))
    names = {PREC_F32: "f32", PREC_BF16: "bf16", PREC_BF16X3: "bf16x3"}
    return bool(ok), names.get(res.value)


def _dtype(dtype) -> int:
    """An sdpa_dtype from a name ("bf16", "fp32", ...), a torch / NumPy dtype, or the integer itself."""
    if isinstance(dtype, int):
        return dtype
    return _DTYPE[str(dtype).rsplit(".", 1)[-1]]


def precision_supported_for(dtype, precision, dk: int, dv: int):
    """:func:`precision_supported` for operands of element type ``dtype``: bf16 operands resolve AUTO to the bf16 kernel
    (where it takes the shape), fp64 / fp32 operands follow the fp64 rule."""
    res = ctypes.c_int(-1)
    ok = lib().sdpa_precision_supported_for(_dtype(dtype), _PREC[precision] if isinstance(precision, str) else int(precision), dk, dv,
                                             ctypes.byref(res))
    names = {PREC_F32: "f32", PREC_BF16: "bf16", PREC_BF16X3: "bf16x3"}
    return bool(ok), names.get(res.value)


def runtime_init(mpi_rank: int = 0, mpi_size: int = 1) -> None:
    _check(lib().sdpa_runtime_init(mpi_rank, mpi_size), "sdpa_runtime_init")


def runtime_shutdown() -> None:
    lib().sdpa_runtime_shutdown()


def get_unique_id() -> bytes:
    buf = ctypes.create_string_buffer(128)
    _check(lib().sdpa_get_unique_id(buf), "sdpa_get_unique_id")
    return buf.raw


def set_bootstrap_id(uid: bytes | None) -> None:
    if uid is None:
        lib().sdpa_set_bootstrap_id(None)
        return
    if len(uid) != 128:
        raise ValueError("ncclUniqueId must be 128 bytes")
    _check(lib().sdpa_set_bootstrap_id(ctypes.create_string_buffer(uid, 128)), "sdpa_set_bootstrap_id")


# ---------------------------------------------------------------------------
# context: resident K/V shards + ping-pong Q batches
# ---------------------------------------------------------------------------
class Context:
    """One process' share of the K/V shards (``num_local`` GPUs out of ``world_size``)."""

    def __init__(self, precision: str | int = "auto", q_batch: int = 0, kv_splits: int = 0, merge: str = "nccl2",
                 num_local: int = 1, first_device: int = 0, world_size: int = 0, rank_base: int = 0,
                 nccl_id: bytes | None = None, distribution: str = "kv"):
        L = lib()
        cfg = Config()
        L.sdpa_config_init(ctypes.byref(cfg))
        cfg.precision = _PREC[precision] if isinstance(precision, str) else int(precision)
        cfg.q_batch, cfg.kv_splits = int(q_batch), int(kv_splits)
        cfg.merge = _MERGE[merge]
        cfg.num_local, cfg.first_device = int(num_local), int(first_device)
        cfg.world_size, cfg.rank_base = int(world_size), int(rank_base)
        cfg.distribution = _DIST[distribution]
        self.num_local = int(num_local)
        self.world_size = int(world_size) if world_size else int(num_local)
        self.rank_base = int(rank_base)
        self._h = ctypes.c_void_p()
        idbuf = ctypes.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
        _check(L.sdpa_ctx_create(ctypes.byref(self._h), ctypes.byref(cfg), idbuf), "sdpa_ctx_create")
        self.dk = self.dv = 0

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            lib().sdpa_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _ptr_array(ptrs):
        arr = (ctypes.c_void_p * len(ptrs))(*[ctypes.c_void_p(int(p) if p else 0) for p in ptrs])
        return arr

    def load_kv_host(self, K_shards, V_shards) -> None:
        """One (n_local_i x dk, n_local_i x dv) fp64 NumPy pair per local GPU (host memory)."""
        Ks = [_as_f64(k, "K shard") for k in K_shards]
        Vs = [_as_f64(v, "V shard") for v in V_shards]
        if len(Ks) != self.num_local or len(Vs) != self.num_local:
            raise ValueError("need one K and one V shard per local GPU")
        dk, dv = Ks[0].shape[1], Vs[0].shape[1]
        counts = (ctypes.c_int * self.num_local)(*[k.shape[0] for k in Ks])
        self._keep = (Ks, Vs)
        _check(lib().sdpa_load_kv_host(self._h, self._ptr_array([k.ctypes.data for k in Ks]),
                                       self._ptr_array([v.ctypes.data for v in Vs]), counts, dk, dv), "sdpa_load_kv_host")
        self.dk, self.dv = dk, dv

    def load_kv_host_ptrs(self, K_ptrs, V_ptrs, n_local, dk: int, dv: int) -> None:
        """Raw host pointers (e.g. pinned torch tensors' ``data_ptr()``)."""
        counts = (ctypes.c_int * self.num_local)(*[int(c) for c in n_local])
        _check(lib().sdpa_load_kv_host(self._h, self._ptr_array(K_ptrs), self._ptr_array(V_ptrs), counts, dk, dv),
               "sdpa_load_kv_host")
        self.dk, self.dv = dk, dv

    def load_kv_device_ptrs(self, K_ptrs, V_ptrs, n_local, dk: int, dv: int) -> None:
        """fp64 device pointers, one per local GPU (e.g. torch CUDA tensors' ``data_ptr()``)."""
        counts = (ctypes.c_int * self.num_local)(*[int(c) for c in n_local])
        _check(lib().sdpa_load_kv_device(self._h, self._ptr_array(K_ptrs), self._ptr_array(V_ptrs), counts, dk, dv),
               "sdpa_load_kv_device")
        self.dk, self.dv = dk, dv

    def load_kv_host_full(self, K, V) -> None:
        K, V = _as_f64(K, "K"), _as_f64(V, "V")
        self._keep = (K, V)
        _check(lib().sdpa_load_kv_host_full(self._h, K.ctypes.data, V.ctypes.data, K.shape[0], K.shape[1], V.shape[1]),
               "sdpa_load_kv_host_full")
        self.dk, self.dv = K.shape[1], V.shape[1]

    def attention_host(self, Q, result=None):
        Q = _as_f64(Q, "Q")
        m = Q.shape[0]
        if self.rank_base == 0 and result is None:
            result = np.empty((m, self.dv), dtype=np.float64)
        rp = result.ctypes.data if result is not None else None
        _check(lib().sdpa_attention_host(self._h, Q.ctypes.data, rp, m), "sdpa_attention_host")
        return result

    def attention_host_ptr(self, Q_ptr: int, result_ptr: int | None, m: int) -> None:
        _check(lib().sdpa_attention_host(self._h, ctypes.c_void_p(Q_ptr), ctypes.c_void_p(result_ptr or 0), m),
               "sdpa_attention_host")

    def attention_device_ptrs(self, Q_ptrs, result_ptr: int | None, m: int) -> None:
        _check(lib().sdpa_attention_device(self._h, self._ptr_array(Q_ptrs), ctypes.c_void_p(result_ptr or 0), m),
               "sdpa_attention_device")

    def attention_device_full(self, K_ptrs, V_ptrs, n_local, dk: int, dv: int, Q_ptrs, result_ptr: int | None, m: int,
                              blocking: bool = True) -> None:
        """The whole path on device-resident fp64 arrays in one C call (K/V cast, Q batches, merge).
        ``blocking=False`` only enqueues the pass (``synchronize()`` waits for all queued passes)."""
        key = (tuple(K_ptrs), tuple(V_ptrs), tuple(n_local), tuple(Q_ptrs))
        if getattr(self, "_full_key", None) != key:   # marshal the pointer arrays once per distinct argument set
            counts = (ctypes.c_int * self.num_local)(*[int(c) for c in n_local])
            self._full_args = (self._ptr_array(K_ptrs), self._ptr_array(V_ptrs), counts, self._ptr_array(Q_ptrs))
            self._full_key = key
        ka, va, counts, qa = self._full_args
        fn = lib().sdpa_attention_device_full if blocking else lib().sdpa_enqueue_device_full
        _check(fn(self._h, ka, va, counts, dk, dv, qa, ctypes.c_void_p(result_ptr or 0), m),
               "sdpa_attention_device_full" if blocking else "sdpa_enqueue_device_full")
        self.dk, self.dv = dk, dv

    def attention_device_typed(self, dtype, K_ptrs, V_ptrs, n_local, dk: int, dv: int, Q_ptrs, result_ptr: int | None, m: int,
                               blocking: bool = True) -> None:
        """:meth:`attention_device_full` on device arrays of element type ``dtype`` ("f64", "f32", "bf16", a torch dtype or
        ``DTYPE_*``); the result has the same type.  bf16 operands at the bf16 kernel and fp32 operands at the fp32 kernel are
        read in place (no cast kernel runs)."""
        counts = (ctypes.c_int * self.num_local)(*[int(c) for c in n_local])
        fn = lib().sdpa_attention_device_typed if blocking else lib().sdpa_enqueue_device_typed
        _check(fn(self._h, _dtype(dtype), self._ptr_array(K_ptrs), self._ptr_array(V_ptrs), counts, dk, dv, self._ptr_array(Q_ptrs),
                  ctypes.c_void_p(result_ptr or 0), m),
               "sdpa_attention_device_typed" if blocking else "sdpa_enqueue_device_typed")
        self.dk, self.dv = dk, dv

    def synchronize(self) -> None:
        _check(lib().sdpa_synchronize(self._h), "sdpa_synchronize")

    def scatter_attention(self, Q=None, K=None, V=None, result=None):
        """Reference calling convention across processes: data on the shard-0 process only."""
        if self.rank_base == 0:
            Q, K, V = _as_f64(Q, "Q"), _as_f64(K, "K"), _as_f64(V, "V")
            m, dk = Q.shape
            n, dv = V.shape
            if result is None:
                result = np.empty((m, dv), dtype=np.float64)
            _check(lib().sdpa_scatter_attention(self._h, Q.ctypes.data, K.ctypes.data, V.ctypes.data, result.ctypes.data,
                                                m, n, dk, dv), "sdpa_scatter_attention")
            return result
        _check(lib().sdpa_scatter_attention(self._h, None, None, None, None, 0, 0, 0, 0), "sdpa_scatter_attention")
        return None

    def online_softmax_partials(self, Qf_dev_ptr: int, m: int, contrib_ptr: int, lmax_ptr: int, lsum_ptr: int,
                                local: int = 0) -> None:
        _check(lib().sdpa_online_softmax_partials(self._h, local, ctypes.c_void_p(Qf_dev_ptr), m, ctypes.c_void_p(contrib_ptr),
                                                  ctypes.c_void_p(lmax_ptr), ctypes.c_void_p(lsum_ptr)),
               "sdpa_online_softmax_partials")

    def last_timings(self) -> dict:
        out = (ctypes.c_float * 6)()
        _check(lib().sdpa_last_timings(self._h, out), "sdpa_last_timings")
        keys = ("total_ms", "cast_ms", "fused_ms", "merge_ms", "fused_launches", "launches")
        return dict(zip(keys, [float(x) for x in out]))

    def accumulated_timings(self, reset: bool = False) -> dict:
        """Stage times summed over all attention calls since the last reset (queried now, not inside the calls)."""
        out = (ctypes.c_double * 6)()
        _check(lib().sdpa_accumulated_timings(self._h, out, 1 if reset else 0), "sdpa_accumulated_timings")
        keys = ("total_ms", "cast_ms", "fused_ms", "merge_ms", "fused_launches", "calls")
        return dict(zip(keys, [float(x) for x in out]))

    def last_kernel(self) -> str:
        return lib().sdpa_last_kernel(self._h).decode()


# ---------------------------------------------------------------------------
# device casts (attention-mpi.c:31-101) on raw device pointers
# ---------------------------------------------------------------------------
def cvt_d2f(dst_ptr: int, src_ptr: int, count: int, stream: int = 0) -> None:
    _check(lib().sdpa_cvt_d2f(ctypes.c_void_p(dst_ptr), ctypes.c_void_p(src_ptr), count, ctypes.c_void_p(stream)), "sdpa_cvt_d2f")


def cvt_f2d(dst_ptr: int, src_ptr: int, count: int, stream: int = 0) -> None:
    _check(lib().sdpa_cvt_f2d(ctypes.c_void_p(dst_ptr), ctypes.c_void_p(src_ptr), count, ctypes.c_void_p(stream)), "sdpa_cvt_f2d")


def cvt_d2bf16x2(hi_ptr: int, lo_ptr: int, src_ptr: int, count: int, stream: int = 0) -> None:
    """The operand split of the bf16x3 precision: hi = bf16(fp32(x)), lo = bf16(fp32(x) - hi)."""
    _check(lib().sdpa_cvt_d2bf16x2(ctypes.c_void_p(hi_ptr), ctypes.c_void_p(lo_ptr), ctypes.c_void_p(src_ptr), count,
                                   ctypes.c_void_p(stream)), "sdpa_cvt_d2bf16x2")


def cvt_d2bf16(dst_ptr: int, src_ptr: int, count: int, stream: int = 0) -> None:
    _check(lib().sdpa_cvt_d2bf16(ctypes.c_void_p(dst_ptr), ctypes.c_void_p(src_ptr), count, ctypes.c_void_p(stream)),
           "sdpa_cvt_d2bf16")
