"""sdpa_b200 -- B200-native scaled-dot-product-attention engine (host-side Python mirror).

The product is the CUDA library ``libsdpa_b200.so`` behind the C ABI in
``include/sdpa_b200.h``; this package only binds it (``host.py``) and builds it
(``build.py``).  Import name: ``sdpa_b200`` (see ``sdpa_b200.py`` at the repo root, which
loads this directory -- its on-disk name contains hyphens).
"""
from . import build as build_mod  # noqa: F401
from .host import (  # noqa: F401
    ABI, Config, Context, SdpaError, attention, cvt_d2bf16, cvt_d2bf16x2, cvt_d2f, cvt_f2d, device_count, get_unique_id, launch_count, lib,
    owner_count, owner_disp, precision_supported, precision_supported_for, runtime_init, runtime_shutdown, set_bootstrap_id, version,
    PREC_AUTO, PREC_BF16, PREC_BF16X3, PREC_F32, MERGE_NCCL, MERGE_NCCL2, MERGE_PEER, DIST_KV, DIST_Q, DIST_AUTO, DTYPE_F64, DTYPE_F32, DTYPE_BF16, LIB_PATH,
)
from .parallel import bootstrap_context, max_over_ranks  # noqa: F401
