"""Step time of queued device-resident passes on one GPU by operand type: what a caller that holds bf16 / fp32 arrays gains
over widening them to fp64.

    python tools/typed_step.py [--rounds 8] [--steps 20] [--sets 6] [--out profiles/r03/typed_step_c3.json]

Configurations, alternated round by round in one process (c3: m = 8192, n = 65536, dk = dv = 128):
    f64_bf16   fp64 operands, precision bf16   (the pass bench.py times)
    bf16_auto  bf16 operands, precision AUTO   (-> bf16: the fused kernel reads the caller's arrays, no cast kernel)
    f64_auto   fp64 operands, precision AUTO   (-> bf16x3)
    f32_auto   fp32 operands, precision AUTO   (-> bf16x3: fp32 -> bf16 hi/lo cast)
Every step takes the next of `--sets` K/V/Q sets, so the working set exceeds the 126 MB L2 (6 bf16 sets: 6 x 34 MB).
Timing: CUDA events around `--steps` queued passes and the closing sdpa_synchronize, per round; the stage split (casts, fused
kernel, merge) from the library's own stage events.  Afterwards the typed results are compared bit for bit with the fp64 pass
at the resolved precision on the same values, rounded into the dtype.  Prints one JSON document (and writes it to --out)."""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

M, N, D = 8192, 65536, 128
CONFIGS = (("f64_bf16", "f64", "bf16"), ("bf16_auto", "bf16", "auto"), ("f64_auto", "f64", "auto"), ("f32_auto", "f32", "auto"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the name from the runtime at least
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sets", type=int, default=6)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    import sdpa_b200
    if sdpa_b200.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("typed_step.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    gen = torch.Generator(device="cuda").manual_seed(1234)
    base = [[torch.randn(r, D, dtype=torch.float64, device="cuda", generator=gen) for r in (N, N, M)] for _ in range(args.sets)]
    tdt = {"f64": torch.float64, "f32": torch.float32, "bf16": torch.bfloat16}
    ops = {dt: [[t.to(tdt[dt]) for t in s] for s in base] for dt in ("f64", "f32", "bf16")}
    outs = {name: [torch.zeros(M, D, dtype=tdt[dt], device="cuda") for _ in range(args.sets)] for name, dt, _ in CONFIGS}
    ctxs = {name: sdpa_b200.Context(precision=prec) for name, _, prec in CONFIGS}

    def step(name, dt, k):
        Kd, Vd, Qd = ops[dt][k]
        fn = ctxs[name].attention_device_full if dt == "f64" else \
            (lambda *a, **kw: ctxs[name].attention_device_typed(dt, *a, **kw))
        fn([Kd.data_ptr()], [Vd.data_ptr()], [N], D, D, [Qd.data_ptr()], outs[name][k].data_ptr(), M, blocking=False)

    def timed(name, dt, steps, first):
        ctx = ctxs[name]
        ctx.accumulated_timings(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for j in range(steps):
            step(name, dt, (first + j) % args.sets)
        ctx.synchronize()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), ctx.accumulated_timings(reset=True)

    for name, dt, _ in CONFIGS:   # warm every shape, kernel and set
        timed(name, dt, max(args.warmup, args.sets), 0)
    per_round = {name: [] for name, _, _ in CONFIGS}
    stages = {name: {"cast_ms": 0.0, "fused_ms": 0.0, "merge_ms": 0.0, "calls": 0.0} for name, _, _ in CONFIGS}
    for r in range(args.rounds):
        for name, dt, _ in (CONFIGS if r % 2 == 0 else CONFIGS[::-1]):   # alternate the order too
            ms, st = timed(name, dt, args.steps, r * args.steps)
            per_round[name].append(1e3 * ms / args.steps)
            for key in stages[name]:
                stages[name][key] += st[key]
    flop = 2.0 * M * N * (D + D)
    result = {"tool": "typed_step", "card": card(), "m": M, "n": N, "dk": D, "dv": D, "sets": args.sets, "rounds": args.rounds,
              "steps_per_round": args.steps, "timing": "CUDA events around each round's queued passes + sdpa_synchronize", "configs": {}}
    for name, dt, prec in CONFIGS:
        us = per_round[name]
        med = statistics.median(us)
        calls = max(1.0, stages[name]["calls"])
        result["configs"][name] = {
            "operands": dt, "precision": prec, "resolved": sdpa_b200.precision_supported_for(dt, prec, D, D)[1],
            "kernel": ctxs[name].last_kernel(), "us_per_step_median": med, "us_per_step_min": min(us), "us_per_step_max": max(us),
            "spread_pct": 100.0 * (max(us) - min(us)) / med, "us_per_round": us, "tflops_median": flop / (med * 1e-6) / 1e12,
            "stage_us_per_pass": {k: 1e3 * stages[name][k] / calls for k in ("cast_ms", "fused_ms", "merge_ms")}}

    # bit-exactness: a typed result == the fp64 pass at the resolved precision on the same (rounded) values, rounded into the dtype
    exact = {}
    for name, dt, prec in CONFIGS:
        if dt == "f64":
            continue
        resolved = result["configs"][name]["resolved"]
        Kd, Vd, Qd = ops[dt][0]
        K64, V64, Q64 = (t.double().contiguous() for t in (Kd, Vd, Qd))
        r64 = torch.zeros(M, D, dtype=torch.float64, device="cuda")
        with sdpa_b200.Context(precision=resolved) as ctx:
            ctx.attention_device_full([K64.data_ptr()], [V64.data_ptr()], [N], D, D, [Q64.data_ptr()], r64.data_ptr(), M)
        typed = torch.zeros(M, D, dtype=tdt[dt], device="cuda")
        ctxs[name].attention_device_typed(dt, [Kd.data_ptr()], [Vd.data_ptr()], [N], D, D, [Qd.data_ptr()], typed.data_ptr(), M)
        ref = r64.float().to(tdt[dt])
        exact[name] = {"bit_exact": bool(torch.equal(typed, ref)), "elements_differing": int((typed != ref).sum().item()),
                       "vs_fp64_unrounded_operands_max_abs": float((typed.double() - outs[
                           "f64_bf16" if resolved == "bf16" else "f64_auto"][0]).abs().max().item())}
    result["bit_exact"] = exact
    for c in ctxs.values():
        c.close()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
