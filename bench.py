#!/usr/bin/env python
"""bench.py -- throughput of the attention hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus N --steps K --warmup W      # the reference's CPU path

Workload (BASELINE.json): the tensor-core configuration c3 -- m=8192 query rows, d_k=d_v=128,
K/V rows sharded over the GPUs with 65536 rows per GPU (n = 65536*N; N=1 is exactly c3, and
c4's per-GPU shard).  Weak scaling: per-GPU K/V shard fixed, Q replicated, so whole-job
FLOPs = 2*m*n*(dk+dv) grow with N.  `--config c2` runs the fp32 configuration instead.

A step is one full pass of the path on fp64 inputs: cast K/V shard, cast Q batches, fused
QK^T->softmax->.V kernel, split/shard merge (NCCL MAX/SUM/SUM for N>1), fp64 result on rank 0.
  value : inputs resident in HBM as fp64 (the contract's input type) when the timed region starts
  e2e   : the same through the C ABI with pinned HOST buffers (H2D of K/V shard + Q, D2H of result)
Timing: CUDA events around exactly K steps, barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DK = DV = 128
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return d, "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock, power and clock-event reasons of this rank's GPU while the timed region runs.

    NVML is read in-process (pynvml, the source nvidia-smi prints) from a thread every 10 ms; `start()` does
    the NVML attach BEFORE the warm-up so that no driver initialisation overlaps the timed steps (eight
    `nvidia-smi` processes attaching to an 8-GPU box during the timed region stretched the steps 3x).  A 20-step
    region lasts a few milliseconds, so bench.py keeps the same load running under the sampler for about a
    second more and says so in `clocks.window`.  Falls back to one `nvidia-smi -lms 100` on rank 0."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, uuid: str | None = None, allow_subprocess: bool = True):
        self.gpu = gpu_index
        self.uuid = uuid
        self.allow_subprocess = allow_subprocess
        self.rows = []          # (sm_mhz, max_mhz, power_w, [reason names])
        self.proc = None
        self._thr = None
        self._stop = threading.Event()
        self._active = threading.Event()
        self._nvml = None
        self._handle = None
        self.source = "none"

    # -- setup (untimed) ----------------------------------------------------------------------
    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                for cand in (self.uuid, "GPU-" + self.uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            self._nvml, self._handle, self.source = pynvml, h, "nvml"
            self._thr = threading.Thread(target=self._poll_nvml, daemon=True)
            self._thr.start()
            return self
        except Exception:
            self._nvml = None
        exe = shutil.which("nvidia-smi")
        if exe and self.allow_subprocess:
            try:
                self.proc = subprocess.Popen([exe, f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                              "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.source = "nvidia-smi"
                self._thr = threading.Thread(target=self._read_smi, daemon=True)
                self._thr.start()
                t0 = time.time()
                while not self.rows and time.time() - t0 < 15.0:   # wait for the attach to finish
                    time.sleep(0.05)
            except Exception:
                self.proc = None
        return self

    def _poll_nvml(self):
        nv, h = self._nvml, self._handle
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = 0.0
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    clk = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    self.rows.append((clk, mx, pw, [n for n, bit in names if mask & bit]))
                except Exception:
                    pass
            self._stop.wait(0.010)

    def _read_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.strip().split(",")]
            if len(parts) >= 7:
                try:
                    row = (float(parts[0]), float(parts[1]), float(parts[2]),
                           [n for n, v in zip(names, parts[3:7]) if v.lower().startswith("active")])
                except Exception:
                    continue
                if self._active.is_set() or not self.rows:
                    self.rows.append(row)

    # -- the sampled window -------------------------------------------------------------------
    def __enter__(self):
        if self._thr is None:
            self.start()
        self.rows = self.rows[:0] if self.source == "nvml" else self.rows[-1:]
        self._active.set()
        return self

    def __exit__(self, *exc):
        self._active.clear()

    def close(self):
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self._thr:
            self._thr.join(timeout=5)
        if self._nvml is not None:
            try:
                self._nvml.nvmlShutdown()
            except Exception:
                pass

    def summary(self):
        sm, mx, power, reasons = [], 0, [], set()
        for clk, cmax, pw, why in self.rows:
            mx = max(mx, cmax)
            if pw < 300.0:      # idle sample (before the first launch / after the last): not "under load"
                continue
            sm.append(clk)
            power.append(pw)
            reasons.update(why)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None, "source": self.source,
                "window": "timed region + ~1 s of the same steps (samples with power draw >= 300 W)"}


# --------------------------------------------------------------------------- workloads (BASELINE.json configs)
# c3 is the headline (weak scaling: 65536 keys per GPU, Q replicated, n = 65536*N; N=1 is exactly c3).  c2 / c4 / c5 are
# run at their BASELINE shapes behind the headline when the GPU count matches (c2 at N=1, c4 at N=4, c5 at N=8) and are
# reported under "configs".  c1 (serial fp64, m=n=512, d=64) is the CPU correctness reference: a parity-test case.
CONFIGS = {
    "c3": {"m": 8192, "n_per_gpu": 65536, "prec": "bf16", "tol": 1e-2, "gpus": None,
           "desc": "c3: m=8192 n=65536/GPU dk=dv=128 bf16->fp32 tensor-core path"},
    "c2": {"m": 4096, "n_total": 4096, "prec": "auto", "tol": 1e-5, "gpus": 1,
           "desc": "c2: m=4096 n=4096 dk=dv=128 fp32, no sharding (default precision: fp32-accurate bf16x3 split on tcgen05)"},
    "c4": {"m": 16384, "n_total": 262144, "prec": "bf16", "tol": 1e-2, "gpus": 4,
           "desc": "c4: m=16384 n=262144 dk=dv=128, K/V sharded over 4 GPUs, Q ping-pong batches + exchange per batch"},
    "c5": {"m": 32768, "n_total": 1048576, "prec": "bf16", "tol": 1e-2, "gpus": 8,
           "desc": "c5: m=32768 n=1048576 dk=dv=128, K/V sharded over 8 GPUs, Q ping-pong batches + exchange per batch"},
}
EXTRAS_BY_GPUS = {1: ["c2"], 4: ["c4"], 8: ["c5"]}
Q_SEED, SHARD_SEED0, PARITY_SEED, PARITY_ROWS = 1234, 1000, 777, 64


def owner_count(n: int, size: int, rank: int) -> int:      # attention-mpi.c:19-22
    return n // size + (1 if rank < n % size else 0)


def config_shape(name: str, world: int, m_override: int = 0, n_per_gpu_override: int = 0):
    """(m, [keys of every rank's shard]) of a configuration on `world` GPUs."""
    c = CONFIGS[name]
    m = m_override or c["m"]
    if "n_per_gpu" in c or n_per_gpu_override:
        per = n_per_gpu_override or c["n_per_gpu"]
        return m, [per] * world
    return m, [owner_count(c["n_total"], world, r) for r in range(world)]


def make_q(m: int):
    import torch
    g = torch.Generator().manual_seed(Q_SEED)
    return torch.randn(m, DK, dtype=torch.float64, generator=g)


def make_shard(rank: int, rows: int):
    """The K/V rows of shard `rank`: seeded by the shard index only, so rank 0 can regenerate every shard for the oracle check."""
    import torch
    g = torch.Generator().manual_seed(SHARD_SEED0 + rank)
    K = torch.randn(rows, DK, dtype=torch.float64, generator=g)
    V = torch.randn(rows, DV, dtype=torch.float64, generator=g)
    return K, V


def parity_rows(m: int):
    import numpy as np
    rng = np.random.default_rng(PARITY_SEED)
    return np.sort(rng.choice(m, size=min(PARITY_ROWS, m), replace=False))


DUMP_BYTES_MAX, DUMP_SEED = 64 * 10**6, 4321


def dump_outputs(out_dir, result) -> None:
    """--dump-outputs: the fp64 result [m, dv] that rank 0's caller received from the last timed step, as result.npy.  Above
    DUMP_BYTES_MAX it is a fixed seeded sample of rows (sorted) instead, their indices in result_rows.npy (float64, exact)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    row_bytes = result.shape[1] * result.itemsize
    if result.nbytes > DUMP_BYTES_MAX:
        keep = (DUMP_BYTES_MAX - 4096) // (row_bytes + 8)     # 4096: room for the two .npy headers
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(result.shape[0], size=keep, replace=False))
        np.save(os.path.join(out_dir, "result_rows.npy"), rows.astype(np.float64))
        result = result[rows]
    np.save(os.path.join(out_dir, "result.npy"), np.ascontiguousarray(result, dtype=np.float64))


def oracle_rows(m: int, shard_rows, rows):
    """fp64 oracle (oracle.attention_f64_numpy = attention.c:20-75) of the selected Q rows against the FULL K/V,
    every shard regenerated from its seed.  Checker only: runs outside every timed region, on rank 0."""
    import numpy as np
    from oracle import oracle
    Q = make_q(m).numpy()[rows]

    def shards():   # one shard in host memory at a time (c5: 1M keys = 2 GiB of fp64 K/V)
        for r, cnt in enumerate(shard_rows):
            K, V = make_shard(r, cnt)
            yield K.numpy(), V.numpy()
    return oracle.attention_f64_streamed(Q, shards())


# --------------------------------------------------------------------------- reference / CPU baseline
def cpu_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def physical_core_cpus():
    """One logical CPU per physical core among the CPUs this process may run on (the reference's authors ran one MPI
    rank per core, README.md:137-141); the shim pins rank r to the r-th entry so ranks never share or migrate."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except Exception:
        allowed = list(range(os.cpu_count() or 1))
    try:
        seen, cpus = set(), []
        cpu = phys = core = None
        for line in Path("/proc/cpuinfo").read_text().splitlines() + [""]:
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip() and cpu is not None:
                if cpu in allowed and (phys, core) not in seen:
                    seen.add((phys, core))
                    cpus.append(cpu)
                cpu = phys = core = None
        return cpus or allowed
    except Exception:
        return allowed


def physical_cores() -> int:
    return max(1, len(physical_core_cpus()))


REF_ROWS = 2048      # Q rows of the CPU arm's sample: the SAME for every GPU count (the K/V side is always complete)


class ReferenceSample:
    """A bounded sample of the workload for the CPU arm: `rows` Q rows against the FULL K/V of the configuration,
    written in the reference's file format with a correct answer block (its harness prints the elapsed time only when
    its own verify() passes, attention-mpi.c:526-532).  A second, one-row file times what the reference spends before
    its batch loop -- dims broadcast, root-side cvt_d2f of K and V, Bcast/Scatterv (attention-mpi.c:193-266) -- which is
    inside its `Elapsed time` and does not shrink with the row sample."""

    def __init__(self, n: int, rows: int = REF_ROWS):
        from oracle import oracle
        import numpy as np
        self.oracle = oracle
        self.n = n
        self.rows = int(rows)
        Q, K, V = oracle.make_inputs(self.rows, n, DK, DV, seed=4242)
        ans = oracle.attention_f64_numpy(Q, K, V)
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        self.dir = tempfile.mkdtemp(prefix="sdpa_ref_", dir=base)
        self.path = os.path.join(self.dir, "sample.bin")
        oracle.write_data_file(self.path, Q, K, V, ans)
        self.path1 = os.path.join(self.dir, "one_row.bin")
        oracle.write_data_file(self.path1, Q[:1], K, V, ans[:1])
        self.Q, self.K, self.V, self.ans = Q, K, V, ans
        self.np = np
        self.cpus = physical_core_cpus()

    def close(self):
        shutil.rmtree(self.dir, ignore_errors=True)

    def kind_and_cores(self):
        if self.oracle.ref_available("mpi"):
            return "reference", len(self.cpus)
        return "port", int(self.oracle.lib().oracle_num_threads())

    def _run_file(self, path) -> float:
        ok, us, out = self.oracle.run_reference(path, "mpi", ranks=len(self.cpus), timeout=1800, pin_cpus=self.cpus)
        if not ok or us is None:
            raise RuntimeError(f"reference binary did not verify: {out[-400:]}")
        return us * 1e-6

    def run_once(self) -> float:
        """Seconds for one pass over the sample (the program's own Elapsed time for kind=reference)."""
        kind, _ = self.kind_and_cores()
        if kind == "reference":
            return self._run_file(self.path)
        t0 = time.perf_counter()
        got = self.oracle.sharded_attention_f32(self.Q, self.K, self.V, shards=1)
        dt = time.perf_counter() - t0
        if not self.oracle.verify_rule(got, self.ans):
            raise RuntimeError("oracle port failed its own check")
        return dt

    def distribution_seconds(self):
        """The reference's K/V cast + distribution time (one-row run), or None for the port."""
        kind, _ = self.kind_and_cores()
        if kind != "reference":
            return None
        return min(self._run_file(self.path1) for _ in range(2))

    def describe(self):
        return (f"{self.rows} Q rows x full K/V (n={self.n}, dk=dv={DK}), program's own timer, "
                f"one rank pinned per physical core")


def tflops_from_rows_per_s(rows_per_s: float, n: int) -> float:
    return rows_per_s * 2.0 * n * (DK + DV) / 1e12


def shared_config(name: str, world: int, m: int, n: int, n_local: int) -> dict:
    """The `config` object: identical in both arms (the driver compares them)."""
    return {"workload": CONFIGS[name]["desc"], "m": m, "n": n, "n_per_gpu": n_local, "dk": DK, "dv": DV,
            "sharding": f"kv-rows/{world} (owner_count/owner_disp), Q replicated",
            "l2": "inputs_larger_than_l2 (fp64 Q+K+V per GPU = %d MiB)" % ((n_local * (DK + DV) + m * DK) * 8 >> 20)}


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, shard_rows = config_shape(args.config, args.gpus, args.m, args.n_per_gpu)
    n = sum(shard_rows)
    sample = ReferenceSample(n, rows=min(REF_ROWS, m))
    try:
        kind, cores = sample.kind_and_cores()
        for _ in range(max(0, args.warmup)):
            sample.run_once()
        times = [sample.run_once() for _ in range(max(1, args.steps))]
        dist_s = sample.distribution_seconds()
    finally:
        sample.close()
    total = sum(times)
    rows_per_s = sample.rows * len(times) / total
    value = tflops_from_rows_per_s(rows_per_s, n)
    step_s = total / len(times)
    cb = {"value": value, "unit": "TFLOP/s", "cores": cores, "kind": kind, "sample": sample.describe(),
          "q_rows_per_s": rows_per_s, "rows": sample.rows, "seconds_per_pass": step_s,
          "kv_cast_and_distribution_s": dist_s,
          "batch_loop_s": (step_s - dist_s) if dist_s is not None else None,
          "note": "value = sample rows / program's Elapsed time, which includes the root's K/V cast + distribution "
                  "(attention-mpi.c:213-266); that part grows with n and does not shrink with the row sample"}
    line = {
        "impl": "reference", "metric": "attention_tflops", "value": value, "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * step_s, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic N(0,1), seeded",
        "q_rows_per_s": rows_per_s,
        "config": shared_config(args.config, args.gpus, m, n, shard_rows[0]),
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- our arm
class Workload:
    """One configuration resident on this rank: pinned host arrays, fp64 device arrays, the two step functions."""

    def __init__(self, torch, ctx, name, rank, world, m, shard_rows):
        self.torch, self.ctx, self.name, self.rank, self.world = torch, ctx, name, rank, world
        self.m, self.shard_rows = m, shard_rows
        self.n_local = shard_rows[rank]
        self.n = sum(shard_rows)
        self.Qh = make_q(m).pin_memory()
        K, V = make_shard(rank, self.n_local)
        self.Kh, self.Vh = K.pin_memory(), V.pin_memory()
        self.Rh = torch.zeros(m, DV, dtype=torch.float64).pin_memory() if rank == 0 else None
        self.Qd, self.Kd, self.Vd = self.Qh.cuda(), self.Kh.cuda(), self.Vh.cuda()
        self.Rd = torch.zeros(m, DV, dtype=torch.float64, device="cuda") if rank == 0 else None
        self._kd, self._vd, self._qd = [self.Kd.data_ptr()], [self.Vd.data_ptr()], [self.Qd.data_ptr()]
        self._rd = self.Rd.data_ptr() if self.Rd is not None else None
        self.flops_step = 2.0 * m * self.n * (DK + DV)

    def step_device(self):
        # queued pass (sdpa_enqueue_device_full): K steps run back to back in stream order, one wait at the end
        self.ctx.attention_device_full(self._kd, self._vd, [self.n_local], DK, DV, self._qd, self._rd, self.m, blocking=False)

    def step_host(self):
        self.ctx.load_kv_host_ptrs([self.Kh.data_ptr()], [self.Vh.data_ptr()], [self.n_local], DK, DV)
        self.ctx.attention_host_ptr(self.Qh.data_ptr(), self.Rh.data_ptr() if self.Rh is not None else None, self.m)

    def h2d_bytes(self):
        return (self.n * (DK + DV) + self.world * self.m * DK) * 8     # every rank uploads its shard and the replicated Q

    def d2h_bytes(self):
        return self.m * DV * 8

    def parity_check(self, tol):
        """Rank 0: a seeded row subset of BOTH results (device-resident pass, host pass) against the fp64 oracle on the
        full K/V (all shards regenerated).  The reference's own acceptance rule (0.02, attention-mpi.c:476) is checked too."""
        import numpy as np
        rows = parity_rows(self.m)
        ref = oracle_rows(self.m, self.shard_rows, rows)
        idx = self.torch.from_numpy(rows)
        dev = self.Rd.cpu()[idx].numpy()
        host = self.Rh[idx].numpy()
        e_dev = float(np.abs(dev - ref).max()) if np.isfinite(dev).all() else float("inf")
        e_host = float(np.abs(host - ref).max()) if np.isfinite(host).all() else float("inf")
        err = max(e_dev, e_host)
        return {"rows": int(len(rows)), "against": "oracle.attention_f64_numpy (attention.c:20-75) on the full K/V, all shards regenerated from their seeds",
                "max_abs_err": err, "max_abs_err_device_path": e_dev, "max_abs_err_host_path": e_host, "tol": tol,
                "reference_gate_0.02": bool(err <= 0.02), "ok": bool(err <= tol)}

    def free(self):
        for a in ("Qd", "Kd", "Vd", "Rd", "Qh", "Kh", "Vh", "Rh"):
            setattr(self, a, None)
        self.torch.cuda.empty_cache()


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    os.environ["SDPA_STAGE_TIMING_EVERY"] = str(max(1, args.stage_timing_every))   # read by the library at context creation
    import sdpa_b200
    from sdpa_b200 import parallel

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_ctx(prec):
        if world > 1:
            return parallel.bootstrap_context(precision=prec, q_batch=args.q_batch, kv_splits=args.kv_splits,
                                              local_rank=local_rank, merge=args.merge)
        return sdpa_b200.Context(precision=prec, q_batch=args.q_batch, kv_splits=args.kv_splits, first_device=local_rank)

    host_enqueue_us = [0.0]

    def timed(ctx, fn, steps, collect=None):
        if collect is not None:
            ctx.accumulated_timings(reset=True)   # stage events are queried once, after the loop
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # Nothing rank-local between the barrier and the first step: a rank that starts late makes the others wait inside the
        # timed region (seen once: 5.8 ms of one 4-GPU run's first exchange step, profiles/r02/visit19_*), and the elapsed time
        # is the MAX over ranks.
        barrier()
        e0.record()
        h0 = time.perf_counter()
        for _ in range(steps):
            fn()
        host_enqueue_us[0] = (time.perf_counter() - h0) * 1e6 / max(1, steps)   # host time to ISSUE one step (not a device time)
        ctx.synchronize()   # the library runs on its own streams: wait for them before the closing event
        e1.record()
        barrier()
        if collect is not None:
            collect(ctx.accumulated_timings(reset=True))
        return parallel.max_over_ranks(e0.elapsed_time(e1))  # ms, max over ranks

    def measure(name, W, K, sampler=None, m_override=0, n_per_gpu_override=0, prec_override=None, parity=True, keep_result=False):
        """Warm-up, K timed device-resident steps, K timed host (e2e) steps, oracle parity check.  Collective over ranks.
        keep_result: rank 0 also returns (as "result") the fp64 output its last timed device-resident step wrote."""
        cfg = CONFIGS[name]
        prec = prec_override or cfg["prec"]
        m, shard_rows = config_shape(name, world, m_override, n_per_gpu_override)
        ctx = make_ctx(prec)
        wl = Workload(torch, ctx, name, rank, world, m, shard_rows)
        for _ in range(W):
            wl.step_device()
        ctx.synchronize()
        stage = {"ms": 0.0, "launches": 0.0, "cast_ms": 0.0, "merge_ms": 0.0, "total_ms": 0.0, "calls": 0.0}
        result = []

        def timed_device():
            ms = timed(ctx, wl.step_device, K, collect)
            if keep_result and wl.Rd is not None:   # copied before any later step writes the buffer again
                result.append(wl.Rd.cpu().numpy())
            return ms

        def collect(t):
            stage["ms"] += t["fused_ms"]
            stage["launches"] += t["fused_launches"]
            stage["cast_ms"] += t["cast_ms"]
            stage["merge_ms"] += t["merge_ms"]
            stage["total_ms"] += t["total_ms"]
            stage["calls"] += t["calls"]      # passes of the timed region that carried stage marks (every --stage-timing-every-th)

        clocks = None
        launches0 = sdpa_b200.launch_count()
        if sampler is not None:
            with sampler as clk:
                ms_dev = timed_device()
                launches = sdpa_b200.launch_count() - launches0   # kernels launched inside the timed region only
                # The timed region is a few milliseconds: keep the identical load running so the sampler sees it.
                # Every step is collective across ranks, so the extra steps are a COUNT derived from the
                # max-reduced time (identical on all ranks), never a per-rank wall-clock loop.
                extra = int(min(20000, max(1, 1000.0 / max(ms_dev / K, 1e-3))))
                for _ in range(extra):
                    wl.step_device()
                ctx.synchronize()
                barrier()
            clocks = clk.summary()
        else:
            ms_dev = timed_device()
            launches = sdpa_b200.launch_count() - launches0
        kernel_name = ctx.last_kernel()
        issue_us = host_enqueue_us[0]
        # e2e: pinned host buffers through the C ABI (blocking calls, the reference's semantics)
        ms_host = float("nan")
        if parity:
            for _ in range(2):
                wl.step_host()
            ms_host = timed(ctx, wl.step_host, K)
        parity = wl.parity_check(cfg["tol"] if prec == "bf16" else min(cfg["tol"], 1e-5)) if (rank == 0 and parity) else None
        res = {
            "name": name, "m": m, "n": wl.n, "n_local": wl.n_local, "prec": prec, "kernel": kernel_name, "steps": K, "warmup": W,
            "ms_dev": ms_dev, "ms_host": ms_host, "flops_step": wl.flops_step, "launches": int(launches),
            "value": wl.flops_step * K / (ms_dev * 1e-3) / 1e12, "e2e_value": wl.flops_step * K / (ms_host * 1e-3) / 1e12,
            "h2d": wl.h2d_bytes(), "d2h": wl.d2h_bytes(), "stage": stage, "clocks": clocks, "parity": parity, "host_issue_us": issue_us,
            "q_batches": -(-m // (args.q_batch or 8192)), "result": result[0] if result else None,
        }
        wl.free()
        ctx.close()
        return res

    # NVML attach happens here, before the warm-up: nothing driver-side may start inside the timed region
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    sampler = ClockSampler(local_rank, gpu_uuid, allow_subprocess=(rank == 0)).start()
    barrier()

    W, K = max(3, args.warmup), args.steps
    head = measure(args.config, W, K, sampler, args.m, args.n_per_gpu, args.precision, keep_result=bool(args.dump_outputs))
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, head["result"])
    clocks = head["clocks"]
    sampler.close()
    if world > 1:   # every rank sampled its own GPU: report the slowest median clock and the union of the reasons
        per_rank = [None] * world
        dist.all_gather_object(per_rank, clocks)
        meds = [c["sm_mhz"] for c in per_rank if c and c["sm_mhz"]]
        clocks = dict(per_rank[0])
        clocks["sm_mhz"] = min(meds) if meds else None
        clocks["reasons"] = sorted({r for c in per_rank if c for r in c["reasons"]})
        clocks["samples"] = sum(c["samples"] for c in per_rank if c)
        pw = [c["power_w_max"] for c in per_rank if c and c["power_w_max"]]
        clocks["power_w_max"] = max(pw) if pw else None
        clocks["per_rank_sm_mhz"] = [c["sm_mhz"] if c else None for c in per_rank]

    # ---- the other BASELINE configurations that fit this GPU count, at their stated shapes -----------------
    extras = {}
    extra_names = [x for x in (args.extra.split(",") if args.extra else EXTRAS_BY_GPUS.get(world, [])) if x and x != "none"]
    if args.m or args.n_per_gpu or args.config != "c3":
        extra_names = [x for x in extra_names if args.extra]   # shape overrides / other headline: only what was asked for
    extra_errors = {}
    for name in extra_names:
        try:
            r = measure(name, 3, K)
        except Exception as exc:   # an extra configuration must not cost the headline line; the failure is reported in it
            extra_errors[name] = repr(exc)
            print("bench: extra configuration %s failed: %r" % (name, exc), file=sys.stderr)
            continue
        if rank == 0:
            extras[name] = {
                "workload": CONFIGS[name]["desc"], "m": r["m"], "n": r["n"], "n_per_gpu": r["n_local"], "kernel": r["kernel"],
                "value": r["value"], "unit": "TFLOP/s", "ms_per_step": r["ms_dev"] / r["steps"], "steps": r["steps"],
                "q_rows_per_s": r["m"] * r["steps"] / (r["ms_dev"] * 1e-3), "q_batches_per_step": r["q_batches"],
                "e2e": {"value": r["e2e_value"], "unit": "TFLOP/s", "ms_per_step": r["ms_host"] / r["steps"],
                        "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
                "stage_ms_per_step": {"cast": r["stage"]["cast_ms"] / max(1.0, r["stage"]["calls"]), "fused": r["stage"]["ms"] / max(1.0, r["stage"]["calls"]),
                                      "merge": r["stage"]["merge_ms"] / max(1.0, r["stage"]["calls"]), "passes_timed": r["stage"]["calls"]},
                "gpu_launches": r["launches"], "parity_check": r["parity"],
            }

    # ---- the fused kernel with the SMs to itself ----------------------------------------------------------
    # Queued passes cast K/V/Q of pass i+1 on a side stream BESIDE the fused kernel of pass i (cast-ahead): the fused stage of
    # the timed region above is the kernel sharing its SMs with an HBM-bound kernel.  The same loop with the casts back in the
    # compute stream (SDPA_CAST_AHEAD=0) times the kernel alone -- reported next to the in-step figure, never instead of it.
    alone = None
    cast_ahead_on = os.environ.get("SDPA_CAST_AHEAD", "1") != "0"
    if world == 1 and head["kernel"] == "bf16_umma_v8" and cast_ahead_on and not args.no_alone:
        was = os.environ.get("SDPA_CAST_AHEAD")
        os.environ["SDPA_CAST_AHEAD"] = "0"
        r = None
        try:
            r = measure(args.config, 3, K, None, args.m, args.n_per_gpu, args.precision, parity=False)
        except Exception as exc:   # the extra leg must never cost the headline line
            print("bench: the `alone` leg failed: %r" % (exc,), file=sys.stderr)
        finally:
            if was is None:
                del os.environ["SDPA_CAST_AHEAD"]
            else:
                os.environ["SDPA_CAST_AHEAD"] = was
        calls_a = max(1.0, r["stage"]["calls"]) if r else 1.0
        alone = None if r is None else {"fused_ms": r["stage"]["ms"] / max(1.0, r["stage"]["launches"]), "cast_ms": r["stage"]["cast_ms"] / calls_a,
                 "merge_ms": r["stage"]["merge_ms"] / calls_a, "ms_per_step": r["ms_dev"] / r["steps"], "value": r["value"], "steps": r["steps"],
                 "flops_per_launch": 2.0 * r["m"] * r["n_local"] * (DK + DV) * calls_a / max(1.0, r["stage"]["launches"])}

    # ---- roofline of the dominant kernel (the fused attention kernel), this rank ---------------
    peaks, peaks_src = load_peaks()
    st = head["stage"]
    m, n, n_local = head["m"], head["n"], head["n_local"]
    kernel_name = head["kernel"]
    calls = max(1.0, st["calls"])
    flops_per_launch = 2.0 * m * n_local * (DK + DV) * calls / max(1.0, st["launches"])   # launches counted over the same marked passes
    avg_ms = st["ms"] / max(1.0, st["launches"])
    achieved = flops_per_launch / (avg_ms * 1e-3) / 1e12 if avg_ms > 0 else 0.0
    peak = float(peaks.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"]))
    bound_note = {"bf16_umma": "tcgen05 bf16 dense; peak = cuBLAS bf16 burst", "bf16_umma_v8": "tcgen05 bf16 dense (persistent kernel); peak = cuBLAS bf16 burst",
                  "f32_simt": "fp32 CUDA-core kernel reported against the bf16 tensor peak (its own FFMA ceiling is ~72 TFLOP/s)"}.get(
                      kernel_name, "tcgen05, bf16 operands; peak = cuBLAS bf16 burst (split-precision kernels execute 3 MMAs per algorithmic MMA)")
    traffic, traffic_src = None, None
    prof = ROOT / "profiles" / "fused_kernel_traffic.json"
    if prof.exists():
        try:
            ent = json.loads(prof.read_text()).get(kernel_name, {})
            traffic = ent.get("dram_bytes_per_launch")
            traffic_src = "static: %s" % ent.get("source", "ncu --set full capture under profiles/")
        except Exception:
            traffic = None
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel_name, "avg_launch_ms": avg_ms, "launches": st["launches"],
                "flops_per_launch": flops_per_launch, "peak_source": peaks_src, "note": bound_note,
                "frac_of_sustained": achieved / float(peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"]))}
    if alone is not None and alone["fused_ms"] > 0:
        a = alone["flops_per_launch"] / (alone["fused_ms"] * 1e-3) / 1e12
        roofline["timed_with"] = "the background cast of the next queued pass on the same SMs (cast-ahead); `alone` = same loop, SDPA_CAST_AHEAD=0"
        roofline["alone"] = {"achieved": a, "frac": a / peak if peak else None, "avg_launch_ms": alone["fused_ms"],
                             "step_ms": alone["ms_per_step"], "step_value": alone["value"],
                             "stage_ms_per_step": {"cast": alone["cast_ms"], "fused": alone["fused_ms"], "merge": alone["merge_ms"]}}

    line = None
    failed = False
    if rank == 0:
        ms_dev, ms_host = head["ms_dev"], head["ms_host"]
        line = {
            "metric": "attention_tflops", "value": head["value"], "unit": "TFLOP/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"f32_simt": "f32", "bf16x3_umma": "bf16x3 (fp32 operands as bf16 hi+lo, fp32 accumulate)"}.get(kernel_name, "bf16"),
            "data": "synthetic N(0,1), seeded",
            "q_rows_per_s": m * K / (ms_dev * 1e-3),
            "config": shared_config(args.config, world, m, n, n_local),
            "impl_detail": {
                "precision": head["prec"], "kernel": kernel_name,
                "merge": "none" if world == 1 else {"peer": "device-side exchange (CUDA IPC, epoch flags): %s" % {
                                                        "instream": "ONE merge kernel on the root's compute stream takes its own pieces and the other shards' states (read over NVLink)",
                                                        "overlap": "root merge kernel on the comm stream reads every shard's state over NVLink",
                                                        "push": "shards push their states into the root's inbox, background merge kernel on the root",
                                                        "pushsync": "shards push their states into the root's inbox, final merge on the root's compute stream",
                                                                                                            "auto": "single-batch passes: 2 GPUs = one merge kernel on the root's compute stream (own pieces + the other "
                                                                "shard's state over NVLink), more GPUs = shards push their states into the root's inbox, final merge on the "
                                                                "root's compute stream; passes of several Q batches: root merge on the comm stream reads the states over NVLink",
                                                    }.get(os.environ.get("SDPA_ROOT_MERGE", "auto"), "root merge"),
                                                    "nccl2": "nccl allreduce(MAX) + reduce(SUM over [contrib|lsum])",
                                                    "nccl3": "nccl allreduce(MAX), allreduce(SUM), reduce(SUM)"}[args.merge],
                "submission": "K passes queued back to back (sdpa_enqueue_device_full), one wait after the last; e2e uses the blocking host call",
                "stages": "cast = K/V/Q fp64 -> compute precision (queued passes on the persistent kernel: a background kernel on a side "
                          "stream beside the PREVIOUS pass's fused kernel -- it overlaps, the stages do not add up to the step); fused = the "
                          "fused attention kernel; merge = its guard twin (exact variant, exits at once unless the overflow guard fired) + "
                          "split merge (+ cross-GPU exchange)",
                "stage_timing": "CUDA-event stage marks (cast | fused | merge) on every %d-th queued pass of the timed region: "
                                "a timestamp event costs ~2 us of stream time, 4 of them per pass were 3.6 %% of the c3 step "
                                "(profiles/r02/visit6_g1_nomarks.json)" % args.stage_timing_every},
            "e2e": {"value": head["e2e_value"], "unit": "TFLOP/s", "h2d_bytes_per_step": head["h2d"], "d2h_bytes_per_step": head["d2h"],
                    "ms_per_step": ms_host / K, "q_rows_per_s": m * K / (ms_host * 1e-3)},
            "gpu_launches": head["launches"],
            "host_issue_us_per_step": head["host_issue_us"],   # host time to enqueue one queued pass (must stay below the device step)
            "clocks": clocks,
            "roofline": roofline,
            "stage_ms_per_step": {"cast": st["cast_ms"] / calls, "fused": st["ms"] / calls, "merge": st["merge_ms"] / calls,
                                  "library_total": st["total_ms"] / calls, "passes_timed": st["calls"]},
            "parity_check": head["parity"],
            "configs": extras,
        }
        failed = not head["parity"]["ok"] or any(not e["parity_check"]["ok"] for e in extras.values()) or bool(extra_errors)
        if extra_errors:
            line["config_errors"] = extra_errors
    # ---- CPU baseline beside it (rank 0, N=1 only) --------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            sample = ReferenceSample(n, rows=min(REF_ROWS, m))
            try:
                kind, cores = sample.kind_and_cores()
                dt = sample.run_once()
                dist_s = sample.distribution_seconds()
            finally:
                sample.close()
            rps = sample.rows / dt
            line["cpu_baseline"] = {"value": tflops_from_rows_per_s(rps, n), "unit": "TFLOP/s", "cores": cores, "kind": kind,
                                    "sample": sample.describe(), "q_rows_per_s": rps, "seconds": dt, "rows": sample.rows,
                                    "kv_cast_and_distribution_s": dist_s,
                                    "batch_loop_s": (dt - dist_s) if dist_s is not None else None}
        except Exception as exc:  # the baseline must not sink the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "TFLOP/s", "cores": 0, "kind": "unavailable", "sample": str(exc)[:200]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        flag = torch.tensor([1 if failed else 0], device="cuda")
        dist.broadcast(flag, src=0)
        failed = bool(flag.item())
        dist.destroy_process_group()
    if failed:
        if rank == 0:
            print("bench.py: parity_check FAILED against the oracle", file=sys.stderr)
        sys.exit(3)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c3")
    ap.add_argument("--precision", choices=["auto", "f32", "bf16", "bf16x3"], default=None)
    ap.add_argument("--m", type=int, default=0)
    ap.add_argument("--n-per-gpu", type=int, default=0)
    ap.add_argument("--q-batch", type=int, default=0)
    ap.add_argument("--kv-splits", type=int, default=0)
    ap.add_argument("--merge", choices=["peer", "nccl2", "nccl3"], default="peer",
                    help="cross-GPU merge: peer = device-side exchange over CUDA-IPC peer memory (default); nccl2/nccl3 = NCCL collectives")
    ap.add_argument("--extra", default="",
                    help="comma list of further BASELINE configs to run behind the headline (default: c2 at 1 GPU, c4 at 4, c5 at 8; 'none' = skip)")
    ap.add_argument("--no-alone", action="store_true", help="skip the extra loop that times the fused kernel without the cast beside it")
    ap.add_argument("--stage-timing-every", type=int, default=4,
                    help="stage marks (CUDA events around cast / fused kernel / merge) on every k-th queued pass (1 = every pass)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the output of the headline's last timed step to DIR/result.npy (fp64; inputs are "
                         "seeded, so runs with the same arguments compare output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's output: it needs --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
