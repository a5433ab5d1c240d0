"""Typed device passes (sdpa_attention_device_typed / sdpa_enqueue_device_typed) on fp32 and bf16 arrays.

The central check is bit-exactness: the kernels see the same operand bits as the fp64 path does on the same values, so the
typed result must equal the fp64 result of the same (resolved) precision, rounded once into the dtype (fp64 -> fp32 -> bf16,
round to nearest even, like the library's result cast).  Every result is also checked against the fp64 oracle on the
dtype-rounded operands: the stated kernel tolerances (f32 / bf16x3 1e-5, bf16 2e-3) plus the rounding of the result."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]

KERNEL_ATOL = {"f32": 1e-5, "bf16x3": 1e-5, "bf16": 2e-3}


def _torch_dtype(name):
    import torch
    return {"f32": torch.float32, "bf16": torch.bfloat16}[name]


def _dev(arrays, dtype):
    """NumPy fp64 arrays -> CUDA tensors of `dtype` (rounded to nearest even)."""
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda().to(dtype) for a in arrays]


def _run_typed(ctx, dtype, K, V, Q, blocking=True, result=None):
    import torch
    m, dv = Q.shape[0], V.shape[1]
    out = result if result is not None else torch.zeros(m, dv, dtype=Q.dtype, device="cuda")
    ctx.attention_device_typed(dtype, [K.data_ptr()], [V.data_ptr()], [K.shape[0]], K.shape[1], dv, [Q.data_ptr()], out.data_ptr(), m,
                               blocking=blocking)
    return out


def _run_f64(prec, K, V, Q, **cfg):
    """The fp64 path at precision `prec` on the same (rounded) values; the result rounded like a typed result.

    The tensor-core kernels work on 256-row blocks of Q.  A typed pass reads a batch's Q through a map of exactly its rows
    (TMA zero-fills the rest of the block); the fp64 path reads its Q slot, whose rows past the batch hold what the slot held
    before, and the overflow guard looks at every row of the block -- stale rows can hand the launch to the exact variant
    (right, but other bits).  So the reference pass gets Q padded with zero rows to whole blocks: the same kernel
    configuration (row blocks, splits, pieces) and the same operand bits as the typed pass."""
    import torch
    import sdpa_b200
    m = Q.shape[0]
    m_run = -(-m // 256) * 256 if prec in ("bf16", "bf16x3") and m > 0 else m
    Kd, Vd = (t.double().contiguous() for t in (K, V))
    Qd = torch.zeros(m_run, Q.shape[1], dtype=torch.float64, device="cuda")
    Qd[:m] = Q.double()
    out = torch.zeros(m_run, V.shape[1], dtype=torch.float64, device="cuda")
    with sdpa_b200.Context(precision=prec, **cfg) as ctx:
        ctx.attention_device_full([Kd.data_ptr()], [Vd.data_ptr()], [K.shape[0]], K.shape[1], V.shape[1], [Qd.data_ptr()],
                                  out.data_ptr(), m_run)
    return out[:m].float().to(Q.dtype)


def _tol(kernel_prec, dtype_name, ref):
    return KERNEL_ATOL[kernel_prec] + (np.abs(ref).max() * 2.0 ** -8 if dtype_name == "bf16" else 1e-6)


def _oracle_ref(oracle, K, V, Q):
    return oracle.attention_f64_numpy(*(t.double().cpu().numpy() for t in (Q, K, V)))


SHAPES = [(600, 16384, 128, 128), (300, 1500, 64, 64), (100, 200, 80, 48), (77, 130, 100, 36)]


@pytest.mark.parametrize("m,n,dk,dv", SHAPES)
@pytest.mark.parametrize("prec", ["auto", "f32", "bf16", "bf16x3"])
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_typed_pass_is_the_fp64_pass_rounded(sdpa, oracle, dtype, prec, m, n, dk, dv):
    ok, resolved = sdpa.precision_supported_for(dtype, prec, dk, dv)
    if not ok:
        pytest.skip(f"{prec} has no kernel for dk={dk} dv={dv}")
    Q, K, V = oracle.make_inputs(m, n, dk, dv, seed=m + n + dk)
    Kt, Vt, Qt = _dev((K, V, Q), _torch_dtype(dtype))
    expect = _run_f64(resolved, Kt, Vt, Qt)
    ref = _oracle_ref(oracle, Kt, Vt, Qt)
    for blocking in (True, False):
        with sdpa.Context(precision=prec) as ctx:
            got = _run_typed(ctx, dtype, Kt, Vt, Qt, blocking=blocking)
            if not blocking:
                ctx.synchronize()
            if resolved == "bf16" and dk == dv == 128:
                assert ctx.last_kernel() == "bf16_umma_v8"
        assert got.dtype == Qt.dtype
        assert np.array_equal(got.float().cpu().numpy(), expect.float().cpu().numpy()), (blocking, resolved)
        np.testing.assert_allclose(got.double().cpu().numpy(), ref, rtol=0, atol=_tol(resolved, dtype, ref))


@pytest.mark.parametrize("dtype,prec", [("bf16", "auto"), ("f32", "auto"), ("f32", "f32"), ("bf16", "bf16x3")])
def test_several_q_batches(sdpa, oracle, dtype, prec):
    m, n, d = 1000, 3000, 128
    Q, K, V = oracle.make_inputs(m, n, d, d, seed=21)
    Kt, Vt, Qt = _dev((K, V, Q), _torch_dtype(dtype))
    resolved = sdpa.precision_supported_for(dtype, prec, d, d)[1]
    expect = _run_f64(resolved, Kt, Vt, Qt, q_batch=384)
    with sdpa.Context(precision=prec, q_batch=384) as ctx:
        got = _run_typed(ctx, dtype, Kt, Vt, Qt)
        assert ctx.last_timings()["fused_launches"] == 3
        queued = _run_typed(ctx, dtype, Kt, Vt, Qt, blocking=False)
        ctx.synchronize()
    for g in (got, queued):
        assert np.array_equal(g.float().cpu().numpy(), expect.float().cpu().numpy())


def test_bf16_d128_pass_runs_no_cast(sdpa, oracle):
    """bf16 operands at d = 128: the fused kernel reads K, V and Q through tensor maps bound to the caller's arrays -- no cast
    kernel, zero cast-stage time; one fused launch and its split merge, then the result cast."""
    m, n, d = 600, 16384, 128
    Q, K, V = oracle.make_inputs(m, n, d, d, seed=5)
    Kt, Vt, Qt = _dev((K, V, Q), _torch_dtype("bf16"))
    with sdpa.Context() as ctx:
        _run_typed(ctx, "bf16", Kt, Vt, Qt)
        t = ctx.last_timings()
        assert ctx.last_kernel() == "bf16_umma_v8"
    assert t["cast_ms"] == 0.0 and t["fused_ms"] > 0.0
    assert t["fused_launches"] == 1


def test_misaligned_operand_is_refused(sdpa, oracle):
    import torch
    m, n, d = 64, 256, 128
    Q, K, V = oracle.make_inputs(m, n, d, d, seed=2)
    Kt, Vt, Qt = _dev((K, V, Q), torch.bfloat16)
    buf = torch.zeros(n * d + 8, dtype=torch.bfloat16, device="cuda")
    Kmis = buf[1:1 + n * d].view(n, d)
    Kmis.copy_(Kt)
    out = torch.zeros(m, d, dtype=torch.bfloat16, device="cuda")
    with sdpa.Context() as ctx:
        with pytest.raises(sdpa.SdpaError, match="aligned") as e:
            _run_typed(ctx, "bf16", Kmis, Vt, Qt, result=out)
        assert "status 1" in str(e.value)   # SDPA_ERR_INVALID
        with pytest.raises(sdpa.SdpaError, match="aligned"):
            _run_typed(ctx, "bf16", Kt, Vt, Qt.view(-1)[1:1 + (m - 1) * d].view(m - 1, d))
        # the cast path (fp32 kernel) takes the same misaligned array
        with sdpa.Context(precision="f32") as ctx2:
            got = _run_typed(ctx2, "bf16", Kmis, Vt, Qt)
        assert np.array_equal(got.float().cpu().numpy(), _run_f64("f32", Kt, Vt, Qt).float().cpu().numpy())


def test_typed_passes_interleaved_with_fp64_cast_ahead_passes(sdpa, oracle):
    """One queue: fp64 passes that cast ahead (persistent kernel, side-stream casts) between typed passes that run no cast
    (bf16) or cast in the compute stream (fp32).  Every typed result equals its own pass run alone, bit for bit."""
    import torch
    m, d = 600, 128
    shapes = (16384, 20000, 1500, 16384 + 136, 16384)
    kinds = ("f64", "bf16", "f64", "f32", "f64")
    cases = [oracle.make_inputs(m, n, d, d, seed=60 + k) for k, n in enumerate(shapes)]
    dev, expect = [], []
    for kind, (Q, K, V) in zip(kinds, cases):
        if kind == "f64":
            t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (K, V, Q)]
            out = torch.zeros(m, d, dtype=torch.float64, device="cuda")
            with sdpa.Context(precision="bf16") as ctx:
                ctx.attention_device_full([t[0].data_ptr()], [t[1].data_ptr()], [t[0].shape[0]], d, d, [t[2].data_ptr()], out.data_ptr(), m)
            expect.append(out.cpu().numpy())
        else:   # the context's precision is bf16: the bf16 pass reads its operands in place, the fp32 pass casts them
            t = _dev((K, V, Q), _torch_dtype(kind))
            expect.append(_run_f64("bf16", *t).float().cpu().numpy())
        dev.append(t)
    with sdpa.Context(precision="bf16") as ctx:
        outs = [torch.zeros(m, d, dtype=t[2].dtype, device="cuda") for t in dev]
        for rep in range(3):
            for kind, (Kd, Vd, Qd), out in zip(kinds, dev, outs):
                if kind == "f64":
                    ctx.attention_device_full([Kd.data_ptr()], [Vd.data_ptr()], [Kd.shape[0]], d, d, [Qd.data_ptr()], out.data_ptr(), m,
                                              blocking=False)
                else:
                    _run_typed(ctx, kind, Kd, Vd, Qd, blocking=False, result=out)
        ctx.synchronize()
    for kind, out, e in zip(kinds, outs, expect):
        if kind == "f64":   # (its Q slot's stale rows may hand a launch to the exact variant: the fp64 path within its tolerance)
            np.testing.assert_allclose(out.cpu().numpy(), e, rtol=0, atol=2e-3)
        else:
            assert np.array_equal(out.float().cpu().numpy(), e), kind


def test_chained_bf16_passes_see_the_previous_result(sdpa, oracle):
    """Queued bf16 passes whose Q is the previous pass's bf16 result: no cast kernel stands between the result cast of one
    pass and the fused kernel of the next, which reads the result in place -- stream order alone must keep them in sequence."""
    import torch
    m, d, n = 600, 128, 16384
    Q, K, V = oracle.make_inputs(m, n, d, d, seed=81)
    V = V * 50.0
    Kt, Vt, Qt = _dev((K, V, Q), torch.bfloat16)
    with sdpa.Context() as ctx:
        r1, r2, r3 = (torch.zeros(m, d, dtype=torch.bfloat16, device="cuda") for _ in range(3))
        _run_typed(ctx, "bf16", Kt, Vt, Qt, blocking=False, result=r1)
        _run_typed(ctx, "bf16", Kt, Vt, r1, blocking=False, result=r2)
        _run_typed(ctx, "bf16", Kt, Vt, r2, blocking=False, result=r3)
        ctx.synchronize()
    e1 = _run_f64("bf16", Kt, Vt, Qt)
    e2 = _run_f64("bf16", Kt, Vt, e1)
    e3 = _run_f64("bf16", Kt, Vt, e2)
    for got, e in ((r1, e1), (r2, e2), (r3, e3)):
        assert np.array_equal(got.float().cpu().numpy(), e.float().cpu().numpy())
    assert (r2.float() - Vt.float().mean(dim=0)).abs().max().item() > 0.5   # the chain mattered


@pytest.mark.parametrize("dtype,prec,d", [("bf16", "auto", 128), ("bf16", "auto", 64), ("f32", "bf16x3", 128)])
def test_queued_typed_pass_repairs_a_fired_guard_at_synchronize(sdpa, oracle, dtype, prec, d):
    """The data of the fp64 repair test: three queued passes, the middle one overflows the fast kernel's exponent guard and is
    re-run (exact variant, same dtype) at sdpa_synchronize."""
    import torch
    m = 300
    good = oracle.make_inputs(m, 1500, d, d, seed=3)
    bad = oracle.make_inputs(m, 1500, d, d, seed=11)
    bad = (bad[0] * 3.0, np.concatenate([bad[1][:128] * 0.01, bad[1][128:] * 30.0]), bad[2])
    cases = [good, bad, good]
    tdt = _torch_dtype(dtype)
    dev = [_dev((K, V, Q), tdt) for (Q, K, V) in cases]
    resolved = sdpa.precision_supported_for(dtype, prec, d, d)[1]
    with sdpa.Context(precision=prec) as ctx:
        outs = [torch.zeros(m, d, dtype=tdt, device="cuda") for _ in cases]
        for rep in range(2):
            for (Kd, Vd, Qd), out in zip(dev, outs):
                _run_typed(ctx, dtype, Kd, Vd, Qd, blocking=False, result=out)
        ctx.synchronize()
    for k, ((Kd, Vd, Qd), out) in enumerate(zip(dev, outs)):
        got = out.double().cpu().numpy()
        assert np.isfinite(got).all()
        ref = _oracle_ref(oracle, Kd, Vd, Qd)
        tol = 2e-2 if k == 1 else _tol(resolved, dtype, ref)
        np.testing.assert_allclose(got, ref, rtol=0, atol=tol + (np.abs(ref).max() * 2.0 ** -8 if k == 1 and dtype == "bf16" else 0))


def test_no_keys_and_no_rows(sdpa, oracle):
    """A pass over an empty K/V shard equals the fp64 pass on it; a pass of zero rows writes nothing."""
    import torch
    m, d = 50, 64
    Q = oracle.make_inputs(m, 1, d, d, seed=4)[0]
    for dtype in ("bf16", "f32"):
        tdt = _torch_dtype(dtype)
        Qt = _dev((Q,), tdt)[0]
        K0 = torch.zeros(0, d, dtype=tdt, device="cuda")
        out = torch.full((m, d), 7.0, dtype=tdt, device="cuda")
        with sdpa.Context() as ctx:
            _run_typed(ctx, dtype, K0, K0, Qt, result=out)
            assert torch.equal(out, _run_f64(sdpa.precision_supported_for(dtype, "auto", d, d)[1], K0, K0, Qt))
            out.fill_(7.0)
            ctx.attention_device_typed(dtype, [K0.data_ptr()], [K0.data_ptr()], [0], d, d, [Qt.data_ptr()], out.data_ptr(), 0)
            torch.cuda.synchronize()
            assert (out == 7.0).all()


def _need_gpus(sdpa, n):
    if sdpa.device_count() < n:
        pytest.skip(f"needs {n} GPUs, {sdpa.device_count()} visible")


@pytest.mark.parametrize("merge", ["nccl2", "peer"])
@pytest.mark.parametrize("dtype,prec,m,n,d", [("bf16", "auto", 700, 5000, 128), ("f32", "auto", 300, 1001, 80), ("f32", "f32", 129, 3, 64),
                                              ("bf16", "auto", 900, 4100, 128), ("bf16", "f32", 50, 1, 32)])
def test_two_local_gpus(sdpa, oracle, merge, dtype, prec, m, n, d):
    """K/V rows sharded over two GPUs of one process (n = 3: ragged; n = 1: GPU 1 owns no key), queued and blocking, against
    the oracle on the dtype-rounded operands."""
    _need_gpus(sdpa, 2)
    import torch
    Q, K, V = oracle.make_inputs(m, n, d, d, seed=m + n)
    tdt = _torch_dtype(dtype)
    resolved = sdpa.precision_supported_for(dtype, prec, d, d)[1]
    ref = oracle.attention_f64_numpy(*(oracle.bf16_round(a).astype(np.float64) if dtype == "bf16" else a.astype(np.float32).astype(np.float64)
                                       for a in (Q, K, V)))
    Qh = torch.from_numpy(Q).to(tdt)
    parts = []
    for g in range(2):
        first, count = sdpa.owner_disp(n, 2, g), sdpa.owner_count(n, 2, g)
        with torch.cuda.device(g):
            parts.append((torch.from_numpy(np.ascontiguousarray(K[first:first + count])).to(tdt).cuda(),
                          torch.from_numpy(np.ascontiguousarray(V[first:first + count])).to(tdt).cuda(), Qh.cuda(), count))
    with sdpa.Context(precision=prec, num_local=2, merge=merge) as ctx:
        for blocking in (True, False):
            out = torch.zeros(m, d, dtype=tdt, device="cuda:0")
            ctx.attention_device_typed(dtype, [p[0].data_ptr() for p in parts], [p[1].data_ptr() for p in parts], [p[3] for p in parts],
                                       d, d, [p[2].data_ptr() for p in parts], out.data_ptr(), m, blocking=blocking)
            if not blocking:
                ctx.synchronize()
            np.testing.assert_allclose(out.double().cpu().numpy(), ref, rtol=0, atol=_tol(resolved, dtype, ref))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from sdpa_b200 import parallel
    from oracle import oracle as o

    m, n, d = 1500, 6001, 128
    Q, K, V = o.make_inputs(m, n, d, d, seed=77)
    first, count = parallel.shard_rows(n, world, rank)
    for dtype, prec, merge, q_batch in (("bf16", "auto", "peer", 512), ("bf16", "auto", "peer", 0), ("f32", "auto", "peer", 512),
                                        ("f32", "f32", "nccl2", 512), ("bf16", "auto", "nccl2", 0)):
        tdt = {"f32": torch.float32, "bf16": torch.bfloat16}[dtype]
        Kd, Vd, Qd = (torch.from_numpy(np.ascontiguousarray(a)).cuda().to(tdt) for a in (K[first:first + count], V[first:first + count], Q))
        ctx = parallel.bootstrap_context(precision=prec, q_batch=q_batch, local_rank=rank, merge=merge)
        outs = [torch.zeros(m, d, dtype=tdt, device="cuda") if rank == 0 else None for _ in range(2)]
        ptr = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
        ctx.attention_device_typed(dtype, [Kd.data_ptr()], [Vd.data_ptr()], [count], d, d, [Qd.data_ptr()], ptr(outs[0]), m)
        for _ in range(3):   # queued passes back to back (the exchange of one overlaps the next), one wait
            ctx.attention_device_typed(dtype, [Kd.data_ptr()], [Vd.data_ptr()], [count], d, d, [Qd.data_ptr()], ptr(outs[1]), m,
                                       blocking=False)
        ctx.synchronize()
        if rank == 0:
            rnd = (lambda a: o.bf16_round(a).astype(np.float64)) if dtype == "bf16" else (lambda a: a.astype(np.float32).astype(np.float64))
            ref = o.attention_f64_numpy(rnd(Q), rnd(K), rnd(V))
            tol = (2e-3 if dtype == "bf16" else 1e-5) + (np.abs(ref).max() * 2.0 ** -8 if dtype == "bf16" else 1e-6)
            for out in outs:
                np.testing.assert_allclose(out.double().cpu().numpy(), ref, rtol=0, atol=tol)
        ctx.close()
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_one_process_per_gpu(sdpa, oracle, tmp_path):
    _need_gpus(sdpa, 2)
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_rank_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))
