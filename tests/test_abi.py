"""The C-ABI library loads without a GPU and exports every symbol include/sdpa_b200.h declares."""
import ctypes
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _declared_symbols():
    text = (ROOT / "include" / "sdpa_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", text)
    keep = [n for n in names if n == "attention" or n.startswith("sdpa_")]
    return sorted(set(keep))


def test_header_symbols_are_exported_and_bound(sdpa):
    declared = _declared_symbols()
    assert "attention" in declared and len(declared) >= 20
    L = sdpa.lib()
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/sdpa_b200.h but not exported"
    assert sorted(sdpa.ABI) == declared, "host.py ABI table and the header disagree"


def test_config_struct_layout(sdpa):
    assert ctypes.sizeof(sdpa.Config) == 16 * 4
    cfg = sdpa.Config()
    sdpa.lib().sdpa_config_init(ctypes.byref(cfg))
    assert cfg.precision == sdpa.PREC_AUTO and cfg.num_local == 1 and cfg.merge == sdpa.MERGE_NCCL2
    assert cfg.distribution == sdpa.DIST_KV                       # the reference's K/V sharding is the default
    assert sdpa.Config.distribution.offset == 8 * 4               # right behind rank_base; the struct size did not move


def test_owner_map_matches_reference_formula(sdpa, oracle):
    for n in (0, 1, 5, 13, 4096, 65536, 1048576):
        for size in (1, 2, 3, 4, 8):
            for r in range(size):
                assert sdpa.owner_count(n, size, r) == oracle.owner_count(n, size, r)
                assert sdpa.owner_disp(n, size, r) == oracle.owner_disp(n, size, r)


def test_no_cpu_fallback(sdpa):
    """Without a CUDA device the engine refuses to create a context (and says why).  Where a GPU is present, a child
    process with every device hidden makes the same attempt."""
    if sdpa.device_count() == 0:
        with pytest.raises(sdpa.SdpaError, match="no CPU fallback"):
            sdpa.Context()
        return
    code = ("import sdpa_b200\ntry:\n    sdpa_b200.Context()\nexcept sdpa_b200.SdpaError as e:\n    print('refused:', e)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(ROOT),
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode == 0 and "refused:" in r.stdout and "no CPU fallback" in r.stdout, r


def test_version_string(sdpa):
    assert "sm_100a" in sdpa.version()


def test_staging_pool_copy_is_exact(sdpa):
    """The multi-threaded memcpy that feeds the pinned staging ring (csrc/host_staging.cu): every size class,
    odd offsets, repeated use of the pool."""
    import numpy as np
    rng = np.random.default_rng(11)
    L = sdpa.lib()
    for nbytes in (0, 1, 4095, 1 << 20, (1 << 20) + 1, 3 * (1 << 20) + 12345, 8 << 20, (8 << 20) + 4097):
        src = rng.integers(0, 256, nbytes + 64, dtype=np.uint8)
        dst = np.zeros(nbytes + 64, dtype=np.uint8)
        for off in (0, 3):
            dst[:] = 0
            lanes = L.sdpa_host_copy(dst.ctypes.data + off, src.ctypes.data + off, nbytes)
            assert lanes >= 2
            assert np.array_equal(dst[off:off + nbytes], src[off:off + nbytes])
            assert not dst[:off].any() and not dst[off + nbytes:].any()


def test_precision_resolution_rules(sdpa):
    """AUTO keeps the reference's fp32 accuracy class: the split-precision tensor-core kernel where the shape fits the SM's
    shared memory, else the fp32 CUDA-core kernel; plain bf16 only on request.  (Host-side rule, no GPU needed.)"""
    ps = sdpa.precision_supported
    assert ps("auto", 128, 128) == (True, "bf16x3") and ps("auto", 64, 64) == (True, "bf16x3") and ps("auto", 80, 48) == (True, "bf16x3")
    assert ps("auto", 64, 256) == (True, "bf16x3")              # narrow dk leaves room for a 256-wide V
    assert ps("auto", 128, 256) == (True, "f32") and ps("auto", 200, 64) == (True, "f32")
    assert ps("auto", 100, 100) == (True, "f32") and ps("auto", 1, 1) == (True, "f32")   # not multiples of 8
    assert ps("auto", 300, 64) == (False, "f32")                 # beyond every kernel (dk, dv <= 256)
    assert ps("bf16", 256, 256) == (True, "bf16") and ps("bf16", 8, 8) == (True, "bf16") and ps("bf16", 200, 136) == (True, "bf16")
    assert ps("bf16", 100, 128)[0] is False and ps("bf16", 264, 128)[0] is False
    assert ps("bf16x3", 128, 128)[0] and not ps("bf16x3", 128, 256)[0] and not ps("bf16x3", 192, 64)[0]
    assert ps("f32", 256, 256) == (True, "f32") and ps("f32", 257, 8)[0] is False
