"""CPU oracle for the attention hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this module; the
engine never does.  It offers

* a NumPy fp64 restatement of the serial definition (``attention.c:20-75``),
* ctypes bindings to ``oracle/sdpa_oracle.c`` (the C restatement of both the
  serial fp64 program and the sharded fp32 online-softmax program,
  ``attention-mpi.c:19-27,168-189,340-380``),
* the reference's binary data-file format (``attention-mpi.c:425-454`` for the
  inputs, ``:472-481`` for the answer block) -- writer and reader with 64-bit
  offsets,
* runners for the reference binaries compiled unmodified into ``oracle/_ref``.

Parity pin: the reference ships no golden vectors; this oracle is pinned
against the compiled reference itself (``tests/test_oracle.py`` and the
fixtures under ``tests/golden/`` produced by ``tests/golden/make_golden.py``).
"""
from __future__ import annotations

import ctypes
import os
import re
import struct
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
BUILD_DIR = HERE / "_build"
REF_DIR = HERE / "_ref"
LIB_PATH = BUILD_DIR / "liboracle.so"
REF_SERIAL = REF_DIR / "attention_serial"
REF_MPI = REF_DIR / "attention_mpi"

_c_double_p = ctypes.POINTER(ctypes.c_double)
_c_float_p = ctypes.POINTER(ctypes.c_float)


def build(reference: str | os.PathLike | None = None, quiet: bool = True) -> None:
    """Compile the C restatement and, if the reference sources are present, oracle/_ref.  reference=None: the
    Makefile's default (REFERENCE from the environment, else the checkout next to this repository)."""
    args = ["make", "-C", str(HERE), "all"]
    if reference is not None:
        args.append(f"REFERENCE={reference}")
    subprocess.run(args, check=True, stdout=subprocess.DEVNULL if quiet else None)


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            subprocess.run(["make", "-C", str(HERE), "oracle"], check=True, stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(str(LIB_PATH))
        L.oracle_owner_count.argtypes = [ctypes.c_int] * 3
        L.oracle_owner_count.restype = ctypes.c_int
        L.oracle_owner_disp.argtypes = [ctypes.c_int] * 3
        L.oracle_owner_disp.restype = ctypes.c_int
        L.oracle_attention_f64_rows.argtypes = [_c_double_p] * 4 + [ctypes.c_int] * 6
        L.oracle_attention_f64_rows.restype = None
        L.oracle_sharded_attention_f32.argtypes = [_c_double_p] * 4 + [ctypes.c_int] * 5
        L.oracle_sharded_attention_f32.restype = ctypes.c_int
        L.oracle_online_softmax_partials_f32.argtypes = [_c_float_p] * 6 + [ctypes.c_int] * 4
        L.oracle_online_softmax_partials_f32.restype = None
        L.oracle_merge_partials_f32.argtypes = [_c_float_p] * 4 + [ctypes.c_int] * 3
        L.oracle_merge_partials_f32.restype = None
        L.oracle_cvt_d2f.argtypes = [_c_float_p, _c_double_p, ctypes.c_size_t]
        L.oracle_cvt_d2f.restype = None
        L.oracle_cvt_f2d.argtypes = [_c_double_p, _c_float_p, ctypes.c_size_t]
        L.oracle_cvt_f2d.restype = None
        L.oracle_num_threads.argtypes = []
        L.oracle_num_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def _dp(a: np.ndarray):
    return a.ctypes.data_as(_c_double_p)


def _fp(a: np.ndarray):
    return a.ctypes.data_as(_c_float_p)


def _c64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _c32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


# --------------------------------------------------------------------------
# shard map (attention-mpi.c:19-27)
# --------------------------------------------------------------------------
def owner_count(n: int, size: int, rank: int) -> int:
    return n // size + (1 if rank < n % size else 0)


def owner_disp(n: int, size: int, rank: int) -> int:
    return rank * (n // size) + min(rank, n % size)


# --------------------------------------------------------------------------
# fp64 definition (attention.c:20-75)
# --------------------------------------------------------------------------
def attention_f64_numpy(Q, K, V, rows: slice | None = None) -> np.ndarray:
    """Vectorised NumPy fp64 softmax(QK^T/sqrt(dk))V.  BLAS summation order differs
    from the reference's left-to-right loops by fp64 rounding only (~1e-15)."""
    Q, K, V = _c64(Q), _c64(K), _c64(V)
    if rows is not None:
        Q = Q[rows]
    dk = Q.shape[1]
    out = np.empty((Q.shape[0], V.shape[1]), dtype=np.float64)
    step = max(1, (1 << 24) // max(1, K.shape[0]))
    for i in range(0, Q.shape[0], step):
        s = (Q[i:i + step] @ K.T) * (1.0 / np.sqrt(float(dk)))
        s -= s.max(axis=1, keepdims=True)
        np.exp(s, out=s)
        s /= s.sum(axis=1, keepdims=True)
        out[i:i + step] = s @ V
    return out


def attention_f64_streamed(Q, kv_shards) -> np.ndarray:
    """The same fp64 definition with K/V arriving shard by shard (`kv_shards` yields (K_r, V_r) in row order): per-shard
    (max, sum, weighted V) states in fp64, combined with the identity of attention-mpi.c:342-380 -- never more than one
    shard in host memory (c5: 2 x 1 GiB of fp64 K/V).  Equal to attention_f64_numpy up to fp64 rounding."""
    Q = _c64(Q)
    scale = 1.0 / np.sqrt(float(Q.shape[1]))
    gmax = np.full((Q.shape[0], 1), -np.inf)
    gsum = np.zeros((Q.shape[0], 1))
    acc = None
    for K, V in kv_shards:
        K, V = _c64(K), _c64(V)
        if acc is None:
            acc = np.zeros((Q.shape[0], V.shape[1]))
        if K.shape[0] == 0:
            continue
        s = (Q @ K.T) * scale
        new_max = np.maximum(gmax, s.max(axis=1, keepdims=True))
        keep = np.where(np.isneginf(gmax), 0.0, np.exp(gmax - new_max))
        np.exp(s - new_max, out=s)
        gsum = gsum * keep + s.sum(axis=1, keepdims=True)
        acc = acc * keep + s @ V
        gmax = new_max
    return acc / gsum


def attention_f64(Q, K, V, row_begin: int = 0, row_end: int | None = None) -> np.ndarray:
    """C restatement with the reference's exact operation order (bit-identical to
    the compiled attention.c).  Rows outside [row_begin,row_end) are left zero."""
    Q, K, V = _c64(Q), _c64(K), _c64(V)
    m, dk = Q.shape
    n, dv = V.shape
    row_end = m if row_end is None else row_end
    out = np.zeros((m, dv), dtype=np.float64)
    lib().oracle_attention_f64_rows(_dp(Q), _dp(K), _dp(V), _dp(out), m, n, dk, dv, row_begin, row_end)
    return out


# --------------------------------------------------------------------------
# sharded fp32 online softmax (attention-mpi.c:168-189, 340-380)
# --------------------------------------------------------------------------
def online_softmax_partials_f32(Qf, K_local, V_local):
    Qf, K_local, V_local = _c32(Qf), _c32(K_local), _c32(V_local)
    rows, dk = Qf.shape
    n_local = K_local.shape[0]
    dv = V_local.shape[1] if V_local.ndim == 2 and V_local.shape[0] else (V_local.shape[1] if V_local.ndim == 2 else 0)
    contrib = np.zeros((rows, dv), dtype=np.float32)
    lmax = np.zeros(rows, dtype=np.float32)
    lsum = np.zeros(rows, dtype=np.float32)
    lib().oracle_online_softmax_partials_f32(_fp(contrib), _fp(lmax), _fp(lsum), _fp(Qf), _fp(K_local),
                                             _fp(V_local), rows, n_local, dk, dv)
    return contrib, lmax, lsum


def merge_partials_f32(contrib, lmax, lsum) -> np.ndarray:
    """contrib [shards, rows, dv]; lmax, lsum [shards, rows] -> [rows, dv]."""
    contrib, lmax, lsum = _c32(contrib), _c32(lmax), _c32(lsum)
    shards, rows, dv = contrib.shape
    out = np.zeros((rows, dv), dtype=np.float32)
    lib().oracle_merge_partials_f32(_fp(out), _fp(contrib), _fp(lmax), _fp(lsum), shards, rows, dv)
    return out


def sharded_attention_f32(Q, K, V, shards: int = 1) -> np.ndarray:
    Q, K, V = _c64(Q), _c64(K), _c64(V)
    m, dk = Q.shape
    n, dv = V.shape
    out = np.zeros((m, dv), dtype=np.float64)
    rc = lib().oracle_sharded_attention_f32(_dp(Q), _dp(K), _dp(V), _dp(out), m, n, dk, dv, shards)
    if rc != 0:
        raise MemoryError("oracle_sharded_attention_f32 failed")
    return out


def cvt_d2f(x) -> np.ndarray:
    x = _c64(x)
    out = np.empty(x.shape, dtype=np.float32)
    lib().oracle_cvt_d2f(_fp(out), _dp(x), x.size)
    return out


def cvt_f2d(x) -> np.ndarray:
    x = _c32(x)
    out = np.empty(x.shape, dtype=np.float64)
    lib().oracle_cvt_f2d(_dp(out), _fp(x), x.size)
    return out


def bf16_round(x) -> np.ndarray:
    """fp64/fp32 -> bf16 (round to nearest even, via fp32 like the device cast) -> fp32."""
    f = np.ascontiguousarray(x, dtype=np.float32)
    u = f.view(np.uint32).astype(np.uint64)
    rounded = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return rounded.astype(np.uint32).view(np.float32).reshape(f.shape)


# --------------------------------------------------------------------------
# synthetic inputs (SURVEY 8d): i.i.d. N(0,1) fp64, fixed seed per config
# --------------------------------------------------------------------------
def make_inputs(m: int, n: int, dk: int, dv: int, seed: int = 0, score_gain: float = 1.0):
    rng = np.random.default_rng(seed)
    Q = rng.standard_normal((m, dk))
    K = rng.standard_normal((n, dk))
    V = rng.standard_normal((n, dv))
    if score_gain != 1.0:
        Q *= score_gain
    return Q, K, V


# --------------------------------------------------------------------------
# data-file format: int32 m,n,dk,dv ; Q ; K ; V ; expected   (all fp64 row-major)
# --------------------------------------------------------------------------
def write_data_file(path, Q, K, V, expected) -> None:
    Q, K, V, expected = _c64(Q), _c64(K), _c64(V), _c64(expected)
    m, dk = Q.shape
    n, dv = V.shape
    assert K.shape == (n, dk) and expected.shape == (m, dv)
    with open(path, "wb") as f:
        f.write(struct.pack("<4i", m, n, dk, dv))
        for a in (Q, K, V, expected):
            a.tofile(f)


def read_data_file(path, with_answers: bool = True):
    with open(path, "rb") as f:
        m, n, dk, dv = struct.unpack("<4i", f.read(16))
        Q = np.fromfile(f, dtype=np.float64, count=m * dk).reshape(m, dk)
        K = np.fromfile(f, dtype=np.float64, count=n * dk).reshape(n, dk)
        V = np.fromfile(f, dtype=np.float64, count=n * dv).reshape(n, dv)
        exp = np.fromfile(f, dtype=np.float64, count=m * dv).reshape(m, dv) if with_answers else None
    return Q, K, V, exp


def verify_rule(result, expected, threshold: float = 0.02) -> bool:
    """The reference's acceptance rule (attention-mpi.c:476,483): every element within
    an absolute 0.02 of the expected value, and no NaN."""
    result = np.asarray(result)
    return bool(np.all(np.isfinite(result)) and np.max(np.abs(result - expected), initial=0.0) <= threshold)


# --------------------------------------------------------------------------
# compiled reference runners (oracle/_ref, built by oracle/Makefile)
# --------------------------------------------------------------------------
_ELAPSED = re.compile(r"Elapsed time:\s*([0-9.]+)\s*us")


def host_has_avx512() -> bool:
    try:
        return "avx512f" in Path("/proc/cpuinfo").read_text()
    except OSError:
        return False


def ref_available(kind: str = "mpi") -> bool:
    p = REF_MPI if kind == "mpi" else REF_SERIAL
    return p.exists() and os.access(p, os.X_OK) and (kind != "mpi" or host_has_avx512())


def run_reference(data_file, kind: str = "mpi", ranks: int = 1, timeout: float = 600.0, pin_cpus=None):
    """Run a compiled reference binary on a data file.  Returns (correct, elapsed_us, stdout).
    pin_cpus: list of logical CPUs; shim rank r is pinned to pin_cpus[r % len] (the `mpirun --bind-to core` analogue)."""
    exe = REF_MPI if kind == "mpi" else REF_SERIAL
    env = dict(os.environ)
    env["MPI_SHIM_NP"] = str(int(ranks))
    if pin_cpus:
        env["MPI_SHIM_CPUS"] = ",".join(str(int(c)) for c in pin_cpus)
    proc = subprocess.run([str(exe), str(data_file)], capture_output=True, text=True, env=env, timeout=timeout)
    out = proc.stdout
    mt = _ELAPSED.search(out)
    return ("Correct!" in out), (float(mt.group(1)) if mt else None), out


def _ref_lib(kind: str) -> ctypes.CDLL:
    path = REF_DIR / ("libattention_mpi.so" if kind == "mpi" else "libattention_serial.so")
    return ctypes.CDLL(str(path))


def reference_attention(Q, K, V, kind: str = "serial") -> np.ndarray:
    """Call the reference's own attention() (compiled unmodified into oracle/_ref with
    -Dmain=...).  kind="serial": attention.c:20-21 (fp64).  kind="mpi": attention-mpi.c:191-192
    with mpi_rank=0, mpi_size=1 on the single-rank shim (fp32 AVX-512 path)."""
    Q, K, V = _c64(Q), _c64(K), _c64(V)
    m, dk = Q.shape
    n, dv = V.shape
    out = np.zeros((m, dv), dtype=np.float64)
    L = _ref_lib(kind)
    if kind == "mpi":
        L.attention.argtypes = [_c_double_p] * 4 + [ctypes.c_int] * 6
        L.attention.restype = None
        L.attention(_dp(Q), _dp(K), _dp(V), _dp(out), m, n, dk, dv, 0, 1)
    else:
        L.attention.argtypes = [_c_double_p] * 4 + [ctypes.c_int] * 4
        L.attention.restype = None
        L.attention(_dp(Q), _dp(K), _dp(V), _dp(out), m, n, dk, dv)
    return out
