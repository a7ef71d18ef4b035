#!/usr/bin/env python
"""bench.py -- candidates/sec scored (qLogEI, 1M x 20D discrete space), BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W              # our arm (CUDA, sm_100a), BASELINE config 2
    python bench.py --config 4|5 --gpus N ...                  # the other single-path configs (extra lines)
    python bench.py --impl reference --steps K --warmup W      # reference arm (CPU restatement)
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs, DIR/*.npy

A "step" is one pass of the hot path over one batch: posterior + qLogEI + global arg-max over the rank's
candidate shard (config 2: 1,000,000 x 20 rows, n=256 training points, Matern-5/2 ARD, S=512 Sobol base
samples, q=1), ending with the arg-max key on the host.  With N>1 every rank scores its own shard (weak scaling:
the candidate set is row-sharded, SURVEY.md 8e) and the global winner comes out of ``bb_allreduce_best``: one warp
per rank folding the packed (score, index) key into every peer's slot over NVLink (no host-issued collective).
The same run also reports STRONG scaling (the 1M set split N ways).  The only place this file touches
``oracle/`` is the CPU-baseline leg and the ``--impl reference`` arm.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_PER_GPU = 1_000_000
D = 20
N_TRAIN = 256
S = 512
SOBOL_SEED = 1234
METRIC = "candidates/sec scored (qLogEI, 1M x 20D discrete space)"
UNIT = "candidates/s"
# identical in both arms (the driver compares the arms' `config`); arm-specific remarks live in `notes`
CONFIG2 = {
    "workload": "BASELINE config 2: 1M x 20D grid candidates per GPU (row-sharded), n=256, Matern-5/2 ARD "
                "prior-mode hyper-parameters, qLogEI S=512 Sobol, q=1",
    "candidates_per_gpu": N_PER_GPU, "d": D, "n_train": N_TRAIN, "mc_samples": S, "q": 1,
    "step_ends": "global arg-max (packed key) on the host",
}


def _workload(n_rows: int, shard: int = 0):
    """Config-2 shard: the training set (and so the model) is identical on every rank -- it is
    drawn from the seed-0 candidate set; the candidate rows of shard r > 0 come from seed 1000+r."""
    from baybe_b200.synthetic import numeric_grid_workload

    base = numeric_grid_workload(N=N_PER_GPU, d=D, n=N_TRAIN, seed=0)
    if shard == 0:
        return base, base.candidates[:n_rows]
    other = numeric_grid_workload(N=n_rows, d=D, n=N_TRAIN, seed=1000 + shard)
    return base, other.candidates


def _ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the headline kernel from the committed ncu
    --set full capture (profiles/, one launch at this exact workload): the newest k_fused_ts summary."""
    names = sorted(p.name for p in (ROOT / "profiles").glob("r0*_k_fused_ts*_ncu_full_summary.txt"))[::-1]
    for name in names + ["r01_k_fused_tc_ncu_full_summary.txt"]:
        f = ROOT / "profiles" / name
        if not f.exists():
            continue
        tot, found = 0.0, 0
        for line in f.read_text().splitlines():
            parts = line.split()
            if parts and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                mult = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(parts[2], 1.0)
                tot += float(parts[1]) * mult
                found += 1
        if found == 2:
            return tot, name
    return None, None


def _peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": d["bf16_tflops"], "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self._nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self) -> dict:
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def _cpu_reference(steps: int, warmup: int, full_steps: int, n_sample: int = 50_000):
    """Time the CPU restatement of the reference path (oracle, torch float64, host threads, 2048-row chunks like
    optimize_acqf_discrete).  The first `full_steps` timed steps score ALL 1,000,000 config-2 candidates, the
    remaining timed steps (and the warm-up) a `n_sample`-row sample of them -- the per-candidate cost of the
    chunked path does not depend on the row count, and the whole run stays within a few minutes."""
    import torch

    import oracle
    from tests.helpers import oracle_model

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    w, cand_full = _workload(N_PER_GPU)
    cand = cand_full[:n_sample]
    om = oracle_model(w)
    acq = oracle.AcqSpec("qLogEI")
    acq.best_f = oracle.best_f_from_training(om, w.train_x, acq)
    z = oracle.sobol_normal_samples(S, 1, SOBOL_SEED)[:, 0]
    # "all the host threads it can use": the 2048-row chunks of the reference path stop scaling
    # (and then collapse) well before 100+ threads, so pick the fastest thread count <= available
    best_t, cores = None, 1
    for t in sorted({c for c in (4, 8, 16, 32, 64, avail) if c <= avail}):
        torch.set_num_threads(t)
        oracle.acq_values(om, acq, cand[:4096], z, chunk=2048)
        t0 = time.perf_counter()
        oracle.acq_values(om, acq, cand[:8192], z, chunk=2048)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, cores = dt, t
    torch.set_num_threads(cores)
    times, rows = [], []
    for i in range(warmup + steps):
        x = cand_full if (i >= warmup and i - warmup < full_steps) else cand
        t0 = time.perf_counter()
        vals = oracle.acq_values(om, acq, x, z, chunk=2048)
        int(torch.argmax(vals))
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            rows.append(len(x))
    total = sum(times)
    # SURVEY.md 8(d) also asks for the best-effort single-pass form (no 2048-row chunking): two passes, best one
    single = None
    for _ in range(2):
        t0 = time.perf_counter()
        vals = oracle.acq_values(om, acq, cand, z, chunk=len(cand))
        int(torch.argmax(vals))
        dt = time.perf_counter() - t0
        single = dt if single is None else min(single, dt)
    full_rate = [r / t for r, t in zip(rows, times) if r == N_PER_GPU]
    return {"value": sum(rows) / total, "ms_per_step_1m": 1e3 * N_PER_GPU * total / sum(rows), "cores": cores,
            "single_pass_value": n_sample / single, "full_steps": min(full_steps, steps), "n_sample": n_sample,
            "full_step_value": (sum(full_rate) / len(full_rate)) if full_rate else None}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = _cpu_reference(args.steps, args.warmup, full_steps=2)
    sample = (f"{r['full_steps']} timed steps over all 1,000,000 config-2 candidates, the other timed steps over "
              f"{r['n_sample']} of them; 2048-row chunks, torch float64, {r['cores']} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step_1m"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": CONFIG2,
        "notes": "reference arm = CPU restatement of the reference's BoTorch/GPyTorch path (oracle port); "
                 "botorch/gpytorch are not installable offline; ms_per_step is normalised to a 1,000,000-row step",
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample,
                         "single_pass_value": r["single_pass_value"], "full_step_value": r["full_step_value"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


class _Timer:
    """K timed steps, per-step CUDA events on the launching stream, L2 flushed (untimed) before every step,
    barrier + synchronize on both sides, MAX over ranks of the summed step times."""

    def __init__(self, dev, world):
        import torch

        self.torch, self.dev, self.world = torch, dev, world
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def __call__(self, fn, k, w_, idle_start=False):
        """idle_start: synchronise after the (untimed) L2 flush, so that the timed call starts on an idle device and
        its host-side launch path is inside the measurement -- used for the end-to-end lines, which time what a user's
        call costs.  Without it the host enqueues the step while the flush is still running (launch latency hidden),
        and the host->device pass was bimodal from run to run (DESIGN.md section 6)."""
        torch = self.torch
        import torch.distributed as dist

        for _ in range(w_):
            fn()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total = 0.0
        for _ in range(k):
            self.flush.fill_(1)  # evict the candidate shard from L2 (untimed)
            if idle_start:
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            t = torch.tensor([total], device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total = float(t.item())
        return total


def _setup_dist():
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the baybe_b200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local_rank, dev


def run_b200(args):
    import torch
    import torch.distributed as dist

    from baybe_b200 import AcqConfig, DeviceGP, sobol_normal_samples
    from baybe_b200.bits import encode_levels
    from baybe_b200.engine import unpack_best

    world, rank, local_rank, dev = _setup_dist()
    steps, warmup = args.steps, max(args.warmup, 3)
    peer = None
    if world > 1:
        from baybe_b200.peers import get_peer_reduce

        peer = get_peer_reduce(dev)

    w, cand = _workload(N_PER_GPU, shard=rank)
    gp = DeviceGP(device=dev, **w.gp_kwargs())
    acq0 = AcqConfig(kind="qLogEI")
    acq = AcqConfig(kind="qLogEI", best_f=gp.best_f(acq0))
    z = sobol_normal_samples(S, 1, SOBOL_SEED)[:, 0].to(dev, torch.float32)
    x_host = torch.from_numpy(cand).to(torch.float32).pin_memory()
    x_dev = x_host.to(dev)
    codes_np, table_np, bits = encode_levels(cand)  # the discrete space in its compact exact form (done once)
    codes_host = torch.from_numpy(codes_np).pin_memory()
    table = torch.from_numpy(table_np).to(dev)  # 880 bytes, resident
    offset = rank * N_PER_GPU
    key_host = torch.empty(1, dtype=torch.int64).pin_memory()
    timed = _Timer(dev, world)

    def finish(key):
        if peer is not None:
            key = peer.allreduce_best(key)  # one warp per rank, NVLink peer atomics; no host-issued collective
        key_host.copy_(key, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # arg-max key is on the host: step ends
        return key_host

    def step_device():
        _, key = gp.score(acq, x_dev, z, index_offset=offset, want_scores=False)
        return finish(key)

    def step_e2e():
        # public API call with the HOST candidate set in its level-coded form (4-bit codes + value table): the fused
        # kernel is launched once and consumes row tiles as the copy stream delivers them; all bytes cross PCIe
        # inside the step
        _, key = gp.score_coded(acq, codes_host, table, bits, z, index_offset=offset, want_scores=False)
        return finish(key)

    def step_e2e_f32():
        # same with the float32 host matrix (80 B per candidate): PCIe-bound
        _, key = gp.score(acq, x_host, z, index_offset=offset, want_scores=False)
        return finish(key)

    if world > 1:
        dist.barrier()  # the ranks finish their set-up seconds apart; the peer reduction waits ~11 s at most
    with ClockSampler(local_rank) as clocks:
        total_ms = timed(step_device, steps, warmup)
    best_val, best_idx = unpack_best(int(key_host.item()))
    e2e_ms = timed(step_e2e, steps, warmup, idle_start=True)
    key_coded = int(key_host.item())
    e2e32_ms = timed(step_e2e_f32, steps, 2, idle_start=True) / steps
    key_f32 = int(key_host.item())
    gp.check_host_pass()
    if peer is not None:
        peer.check()

    # dominant kernel alone (events on the launching stream), for the roofline
    def kernel_only():
        gp.score(acq, x_dev, z, index_offset=offset, want_scores=False)

    kern_ms = timed(kernel_only, steps, 1) / steps
    ms_per_step = total_ms / steps
    value = world * N_PER_GPU / (ms_per_step * 1e-3)
    e2e_value = world * N_PER_GPU / (e2e_ms / steps * 1e-3)

    # strong scaling: the SAME 1,000,000-row set (seed 0) split over the ranks
    strong = None
    if world > 1:
        _, all_rows = _workload(N_PER_GPU, shard=0)
        per = -(-N_PER_GPU // world)
        lo, hi = min(rank * per, N_PER_GPU), min((rank + 1) * per, N_PER_GPU)
        xs = torch.from_numpy(all_rows[lo:hi]).to(dev, torch.float32)

        def step_strong():
            _, key = gp.score(acq, xs, z, index_offset=lo, want_scores=False)
            return finish(key)

        s_ms = timed(step_strong, steps, warmup) / steps
        strong = {"value": N_PER_GPU / (s_ms * 1e-3), "unit": UNIT, "ms_per_step": s_ms,
                  "candidates_total": N_PER_GPU, "rows_per_gpu": per,
                  "best": dict(zip(("value", "index"), unpack_best(int(key_host.item()))))}

    if rank == 0:
        peaks = _peaks()
        flops = N_PER_GPU * (2.0 * N_TRAIN * N_TRAIN + 2.0 * N_TRAIN * D)  # SURVEY 8d: 2n^2 + 2nd per candidate
        achieved = flops / (kern_ms * 1e-3) / 1e12
        traffic, traffic_src = _ncu_traffic_bytes()
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            r = _cpu_reference(6, 1, full_steps=1)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                   "sample": f"1 pass over all 1,000,000 config-2 candidates + 5 passes over {r['n_sample']} of them, "
                             "2048-row chunks, torch float64",
                   "single_pass_value": r["single_pass_value"],
                   "single_pass_note": "50,000-row sample scored in one unchunked pass (best of 2), same thread count"}
        launches = (3 + (1 if world > 1 else 0)) * steps  # key init + qLogEI table + fused kernel (+ one-warp peer reduction)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": CONFIG2,
            "notes": {
                "layout": "fp32 row-major, resident in HBM",
                "l2": "flushed between timed steps (256 MiB write, untimed)",
                "reduction": ("single GPU" if world == 1 else
                              "bb_allreduce_best: one warp per rank, atomicMax.sys into every peer's slot over NVLink "
                              "(CUDA IPC mapped), no host-issued collective" if peer.kind == "peer" else
                              "BB_PEER_REDUCE=0: host-issued ncclAllReduce(MAX, int64) per step"),
                "precision": "distance GEMM (fp16 hi/mid/lo split, 2^-33) and K* L^-T (fp16 hi/lo split, A operand "
                             "in tensor memory) on tcgen05, fp32 TMEM accumulate; packed-fp32 Matern epilogue and MC",
                "best": {"value": best_val, "index": best_idx},
                "e2e_coded_matches_resident": key_coded == int(key_host.item()) if world == 1 else None,
            },
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(codes_host.numel() + table.numel() * 4), "d2h_bytes_per_step": 8,
                    "timing": "per step: L2 flush (untimed), device synchronised, then events around the public call "
                              "incl. its host-side launch path, H2D of all bytes and the D2H of the key",
                    "api": f"DeviceGP.score_coded(pinned host {bits}-bit level codes + value table) -> bb_score_fused_overlapped "
                           "-> host arg-max key; ONE kernel launch that consumes row tiles as the copy stream publishes "
                           "them (growing H2D blocks + cuStreamWriteValue32), codes expanded in the kernel's staging step; "
                           "scores bit-identical to the float32 matrix",
                    "fp32_matrix": {"value": world * N_PER_GPU / (e2e32_ms * 1e-3), "h2d_bytes_per_step": x_host.numel() * 4,
                                    "api": "DeviceGP.score(pinned host fp32 matrix)"}},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "roofline": {
                "bound": "tensor", "kernel": "k_fused_ts<matern52>", "achieved": achieved,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
                "traffic": traffic, "traffic_unit": "bytes per launch (ncu --set full, profiles/)",
                "traffic_source": traffic_src,
                "algorithmic_bytes": N_PER_GPU * (4 * D + 4), "kernel_ms": kern_ms, "peak_source": peaks["source"],
                "note": "algorithmic flops = N*(2n^2 + 2nd) (SURVEY 8d); the tensor pipe executes 3 split products "
                        "over 8.5/16 of the n^2 (triangular skip at 16-column granularity) plus 6 split products of "
                        "the distance GEMM over K = 32; see DESIGN.md",
            },
            "cpu_baseline": cpu,
        }
        if strong is not None:
            line["strong_scaling"] = strong
        if args.dump_outputs:
            outs = {"best_value": best_val, "best_index": best_idx}
            outs["e2e_best_value"], outs["e2e_best_index"] = unpack_best(key_coded)
            outs["e2e_f32_best_value"], outs["e2e_f32_best_index"] = unpack_best(key_f32)
            if strong is not None:
                outs["strong_best_value"], outs["strong_best_index"] = strong["best"]["value"], strong["best"]["index"]
            _dump_outputs(args.dump_outputs, outs)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_other(args):
    """BASELINE configs 4 and 5 (extra lines, not the driver's headline): same JSON shape."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from baybe_b200 import AcqConfig, DeviceGP, sobol_normal_samples
    from baybe_b200.engine import unpack_best
    from baybe_b200.synthetic import fingerprint_workload, task_workload

    world, rank, local_rank, dev = _setup_dist()
    steps, warmup = args.steps, max(args.warmup, 3)
    peer = None
    if world > 1:
        from baybe_b200.peers import get_peer_reduce

        peer = get_peer_reduce(dev)
    z = sobol_normal_samples(S, 1, SOBOL_SEED)[:, 0].to(dev, torch.float32)
    timed = _Timer(dev, world)
    key_host = torch.empty(1, dtype=torch.int64).pin_memory()
    peaks = _peaks()
    if args.config == 4:
        # 10M x 2048-bit fingerprints (Bernoulli 0.05), n = 512, ScaleKernel(RBF); STRONG: 10M split over the ranks
        total_rows = 10_000_000
        per = -(-total_rows // world)
        lo, hi = min(rank * per, total_rows), min((rank + 1) * per, total_rows)
        w = fingerprint_workload(N=4096, d=2048, n=512, seed=1)
        gp = DeviceGP(device=dev, **w.gp_kwargs())
        g = torch.Generator(device=dev).manual_seed(1000 + rank)
        x = torch.empty((hi - lo, 256), dtype=torch.uint8, device=dev)
        for a in range(0, hi - lo, 500_000):  # generate in blocks: the boolean staging tensor is 8x the packed size
            b = min(a + 500_000, hi - lo)
            bits = torch.rand((b - a, 256, 8), device=dev, generator=g) < 0.05
            x[a:b] = (bits.to(torch.uint8) << torch.arange(8, device=dev, dtype=torch.uint8)).sum(dim=2).to(torch.uint8)
        del bits
        n_tr, d_feat = 512, 2048
        name = "BASELINE config 4: 10M x 2048-bit Morgan-like fingerprints (bit-packed), n=512, ScaleKernel(RBF), qLogEI S=512"
        scaling, metric = "strong", "candidates/sec scored (qLogEI, 10M x 2048-bit fingerprint space)"
        kern_rows = min(hi - lo, 262_144)
        kernel_fn = lambda: gp.kernel_matrix(x[:kern_rows])  # noqa: E731  (k_kmat_tc alone: the dominant kernel)
        kern_flops = kern_rows * 2.0 * n_tr * d_feat
        kern_name = "k_kmat_tc<rbf,bits> (distance GEMM of one 262,144-row block)"
        rl_note = ("algorithmic flops = rows*2*n*d; the bit-linear form issues 2 fp16 split products, so the tensor "
                   "pipe executes 2x this")
        total = total_rows
    else:
        # 4 tasks x 250k rows (config-2 grid + task column), ICM kernel, n = 512; rows sharded regardless of task
        total_rows = 1_000_000
        w = task_workload(N_per_task=250_000, n_tasks=4, d_num=20, n_per_task=128, seed=0)
        per = -(-total_rows // world)
        lo, hi = min(rank * per, total_rows), min((rank + 1) * per, total_rows)
        perm = np.random.default_rng(0).permutation(total_rows)  # shards see all tasks
        gp = DeviceGP(device=dev, **w.gp_kwargs())
        x = torch.from_numpy(w.candidates[perm[lo:hi]]).to(dev, torch.float32)
        n_tr, d_feat = 512, 21
        name = "BASELINE config 5: 4 tasks x 250k candidates (20 numeric + task column), ICM kernel, n=512, qLogEI S=512"
        scaling, metric = "strong", "candidates/sec scored (qLogEI, 4 x 250k transfer-learning space)"
        kernel_fn = lambda: gp.score(acq, x, z, want_scores=False)  # noqa: E731
        kern_flops = (hi - lo) * (2.0 * n_tr * n_tr + 2.0 * n_tr * d_feat)
        kern_name = "k_fused<matern52> (FFMA2 distances, tcgen05 V contraction, n_pad=512)"
        rl_note = "algorithmic flops = rows*(2n^2 + 2nd)"
        total = total_rows
    acq = AcqConfig(kind="qLogEI", best_f=gp.best_f(AcqConfig(kind="qLogEI")))

    def step():
        _, key = gp.score(acq, x, z, index_offset=lo, want_scores=False)
        if peer is not None:
            key = peer.allreduce_best(key)
        key_host.copy_(key, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    if world > 1:
        dist.barrier()  # data generation differs per rank by seconds; the peer reduction waits ~11 s at most
    with ClockSampler(local_rank) as clocks:
        total_ms = timed(step, steps, warmup)
    best_val, best_idx = unpack_best(int(key_host.item()))
    kern_ms = timed(kernel_fn, steps, 2) / steps
    topk = None
    if args.config == 5:
        # "NCCL top-k argmax": per-rank bb_topk + one all-gather of k (value, index) pairs
        from baybe_b200.recommenders import distributed_topk

        scores, _ = gp.score(acq, x, z, index_offset=lo)
        v, i = distributed_topk(scores, None, 8, offset=lo)
        topk = {"values": v.tolist(), "positions_in_shard_order": i.tolist()}
    if peer is not None:
        peer.check()
    if rank == 0:
        ms = total_ms / steps
        achieved = kern_flops / (kern_ms * 1e-3) / 1e12
        line = {
            "metric": metric, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": name, "candidates_total": total, "rows_per_gpu": per},
            "e2e": None, "gpu_launches": None, "clocks": clocks.summary(),
            "roofline": {"bound": "tensor", "kernel": kern_name, "achieved": achieved, "peak": peaks["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": None,
                         "kernel_ms": kern_ms, "peak_source": peaks["source"], "note": rl_note},
            "cpu_baseline": None,
            "notes": {"best": {"value": best_val, "index": best_idx}, "topk": topk},
        }
        if args.dump_outputs:
            _dump_outputs(args.dump_outputs, {"best_value": best_val, "best_index": best_idx})
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def _dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write what the timed path returned in its last step as ``out_dir/<name>.npy`` (float64: every value here,
    indices included, is exact in it).  The inputs are seeded, so two builds run with the same arguments can be
    compared output for output."""
    import numpy as np

    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.asarray(a, dtype=np.float64))


def _emit(line: dict) -> None:
    """Write the ONE JSON line to the real stdout (fd saved before libraries could print to it)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def run_hybrid(args):
    """BASELINE config 3 (extra line, single GPU): hybrid space of 8 discrete x 4 continuous parameters, qNEI with 512
    MC samples, one batch recommendation q = 16 per step through baybe_b200.hybrid.recommend_hybrid (search by
    scoring).  The unit stays candidates/s: rows swept by the qNEI scorer per second."""
    import numpy as np
    import torch

    from baybe_b200 import AcqConfig, DeviceGP
    from baybe_b200 import hybrid as hy

    world, rank, local_rank, dev = _setup_dist()
    if world > 1:
        raise SystemExit("bench.py --config 3 is a single-GPU line")
    rng = np.random.default_rng(0)
    levels = [3, 3, 3, 3, 2, 2, 2, 2]  # 8 discrete parameters: 1296 configurations
    grids = np.meshgrid(*[np.linspace(0.0, 1.0, k) for k in levels], indexing="ij")
    disc = np.stack([g.reshape(-1) for g in grids], axis=1)
    d_disc, d_cont, n = disc.shape[1], 4, 64
    train_x = np.hstack([disc[rng.integers(0, len(disc), n)], rng.random((n, d_cont))])
    f = train_x @ rng.normal(0, 1, d_disc + d_cont) + np.sin(3 * train_x[:, -1]) * (1 + train_x[:, 0])
    train_y = f + 0.05 * rng.standard_normal(n)
    bounds = np.array([[0.0] * (d_disc + d_cont), [1.0] * (d_disc + d_cont)])
    gp = DeviceGP(train_x, train_y, bounds, "matern52", np.full(d_disc + d_cont, 0.8), 1e-2, 0.0, device=dev)
    acq = AcqConfig(kind="qNEI")
    search = hy.HybridSearch(n_sobol=1024, n_seeds=64, n_local=128, n_rounds=6)
    rows_per_step = 16 * (len(disc) * min(search.n_sobol, search.max_rows // len(disc))
                          + search.n_rounds * search.n_seeds * search.n_local)
    cb = np.array([[0.0] * d_cont, [1.0] * d_cont])
    steps, warmup = args.steps, 1
    last = {}

    def step():
        last["out"] = hy.recommend_hybrid(gp, acq, disc, cb, 16, None, S, 3, search)

    timed = _Timer(dev, world)
    with ClockSampler(local_rank) as clocks:
        ms = timed(step, steps, warmup) / steps
    pts, idx, value = last["out"]
    if args.dump_outputs:
        _dump_outputs(args.dump_outputs, {"points": pts, "configuration_index": idx, "joint_qnei": value})
    _emit({
        "metric": "candidates/sec scored (qNEI S=512, hybrid 8 discrete x 4 continuous, q=16 batch)",
        "value": rows_per_step / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "BASELINE config 3: 1296 discrete configurations x 4 continuous parameters, n=64, "
                               "qNEI (512 MC samples, baseline = training inputs), q=16 sequential greedy, "
                               "search by scoring (1024 Sobol points per configuration + 6 refinement sweeps)",
                   "rows_scored_per_recommendation": rows_per_step},
        "e2e": None, "gpu_launches": None, "clocks": clocks.summary(), "roofline": None, "cpu_baseline": None,
        "notes": {"joint_qnei_of_batch": value, "first_point": pts[0].tolist(),
                  "pipeline": "bb_kernel_matrix + bb_posterior(+cross) + cuBLAS GEMM (library) + bb_nei_reduce"},
    })


def main():
    global _REAL_STDOUT
    # NCCL / torch may print banners to stdout; keep stdout clean for the single JSON line
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", type=int, choices=[2, 3, 4, 5], default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA arm")
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 2:
        run_b200(args)
    elif args.config == 3:
        run_hybrid(args)
    else:
        run_other(args)


if __name__ == "__main__":
    main()
