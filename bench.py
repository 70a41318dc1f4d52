#!/usr/bin/env python
"""Headline benchmark: `Flow.log_prob` samples/s on the MNIST-shape USFlow stack (BASELINE.json
configs[1]: D=784 NonUSFlow, K=8 coupling blocks, conditioner MLP 784-256-256-1568, LU + Householder
affine conjugation, Normal base), synthetic data, batch-sharded over N GPUs (weak scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.  `--dump-outputs DIR` also writes the
log_prob vector the last timed step returned as DIR/log_prob.npy (float32; one file per rank under torchrun); inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.  Compare within the
tier's tolerance: packing the weights is not bit-reproducible in fp32, and in the bf16 tier that moves a few bf16
roundings, so one build's log_prob varies from run to run by up to about 3e-3 relative (bf16x2: 5e-6, fp32: 1e-6;
measured on a B200 at its 1000 W power limit).
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# ---- workload: BASELINE.json configs[1] / SURVEY.md section 8(d) "C2 MNIST" --------------------------------
D, K_BLOCKS, HIDDEN = 784, 8, [256, 256]
ROWS_PER_GPU = 65536
ALG_FLOP_PER_SAMPLE = 26.84e6      # mask-pruned, conditioner counted once (SURVEY 8d / BASELINE.md section 4)
ALG_BYTES_PER_SAMPLE = 4 * D + 4
LAST_LAYER_GAIN = 0.25             # trained-flow-like activations (see DESIGN.md "Synthetic weights")
CPU_ROWS = 65536                   # BASELINE.md section 3: the CPU arm scores B = 65536 (and B = 32) like the GPU arm
CPU_SMALL_ROWS = 32
TRAIN_SMALL_ROWS = 64              # SURVEY 8(d): training B per GPU = 64 (the reference's regime) and 4096
# DRAM bytes per launch at 65536 rows from the committed ncu capture (profiles/): {kind: bytes}; filled from
# profiles/r2/ncu_dram_bytes.json when present (written by scripts/ncu_summary.py), else the round-1 capture
NCU_DRAM_BYTES = {"affine_gemm": 174.4e6, "conditioner+coupling": 120.3e6, "final_gemm+base": 174.4e6}

# Every BASELINE.json config shape (SURVEY.md 8d "Config -> concrete stack"): name -> (flow kind, D, K, conditioner,
# base, last-layer gain, constructor kwargs, algorithmic MFLOP/sample (pruned, SURVEY 8d / BASELINE.md section 4),
# roofline that bounds it).  `--config NAME` benches one of them; the default run adds a short resident-input line for
# each under "configs" (at whatever GPU count it was launched with -> 1 / 2 / 4 / 8 through the driver's scaling run).
CONFIGS = {
    "C1-gmm-D2": ("USFlow", 2, 10, ("densenn1", [128, 128]), "usnormal", 0.5, dict(affine_conjugation=True, householder=0, prior_scale=1.0), 0.333, "hbm"),
    "C1-gmm-D128": ("USFlow", 128, 10, ("densenn1", [128, 128]), "usnormal", 0.5, dict(affine_conjugation=True, householder=0, prior_scale=1.0), 1.35, "tensor"),
    "C2-mnist-D784": ("NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0), 26.84, "tensor"),
    "C3-fashion-D784": ("NonUSFlow", 784, 11, ("mlp", [200, 200, 200]), "laplace", 0.25, dict(affine_conjugation=True, householder=0), 35.24, "tensor"),
    "C4-adbench-D6": ("NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0), 0.001, "hbm"),
    "C4-adbench-D64": ("NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0), 0.10, "hbm"),
    "C4-adbench-D500-K3": ("NonUSFlow", 500, 3, ("mlp", [128]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0), 4.10, "tensor"),
    "C4-adbench-D500-K8": ("NonUSFlow", 500, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True), 12.67, "tensor"),
    "C5-mvtec-D128": ("USFlow", 128, 10, ("densenn1", [512, 256]), "normal", 0.5, dict(affine_conjugation=True, householder=0), 4.30, "tensor"),
    "C5-mvtec-D256": ("NonUSFlow", 256, 10, ("mlp", [512, 256]), "normal", 0.25, dict(affine_conjugation=True), 8.00, "tensor"),
}
DEFAULT_CONFIG = "C2-mnist-D784"


def build_config_flow(ns, name, device):
    from _cases import build_flow as _bf, tame
    kind, d, k, cond, base, gain, kw, _, _ = CONFIGS[name]
    torch.manual_seed(0)
    flow = _bf(ns, kind, d, k, cond, base=base, **kw)
    tame(flow, gain)
    return flow.to(device).eval()


def build_flow(ns, device, dtype=torch.float32):
    return build_config_flow(ns, DEFAULT_CONFIG, device)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index, self.err = [], None, index, ""
        self.sm = self.rows

    def _cmd(self, loop):
        cmd = ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"]
        return cmd + (["-lms", "50"] if loop else [])

    def start(self):
        try:
            self.proc = subprocess.Popen(self._cmd(True), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:
            self.proc, self.err = None, repr(e)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def sample_once(self):
        """One synchronous sample (taken while kernels are in flight) in case the loop produced none."""
        try:
            r = subprocess.run(self._cmd(False), capture_output=True, text=True, timeout=20)
            if r.stdout.strip():
                self.rows.append(r.stdout.strip().splitlines()[0])
            else:
                self.err = (r.stderr or "").strip()[:200]
        except Exception as e:
            self.err = repr(e)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable: " + self.err]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.err = self.err or (self.proc.stderr.read() or "").strip()[:200]
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if not sm and self.err:
            out["error"] = self.err
        return out


class NvmlSampler:
    """In-process NVML sampling thread (same counters as the nvidia-smi query above: SM clock, max SM
    clock, clock-event reasons).  Preferred over spawning `nvidia-smi -lms`, which was measured to stall
    kernel launches on this box (a 2 ms step became 12 ms while it polled).  NVML queries and CUDA launches share
    a driver lock: with three queries every 50 ms some runs lost 30-50 % of the timed region to stalled graph
    launches (host enqueue 1.2-2.6 ms per step instead of 0.04), so the thread asks for two values every 100 ms."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index, period_s=0.1):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        self.period, self.sm, self.mask, self.stop_flag, self.rows = period_s, [], 0, False, []
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))

    def _one(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _loop(self):
        while not self.stop_flag:
            try:
                self._one()
            except Exception as e:          # keep the bench alive; report below
                self.err = repr(e)
                return
            time.sleep(self.period)

    def start(self):
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def sample_once(self):
        try:
            self._one()
        except Exception as e:
            self.err = repr(e)

    def stop(self):
        self.stop_flag = True
        if hasattr(self, "t"):
            self.t.join(timeout=2)
        try:        # one power reading, AFTER the timed region: every NVML query takes the driver lock the launches need
            self.rows.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
        except Exception:
            pass
        sm = sorted(self.sm)
        pw = sorted(self.rows)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in self.REASONS.items() if self.mask & b), "samples": len(sm),
                "power_w": pw[len(pw) // 2] if pw else None, "source": "nvml"}


class NullSampler:
    sm = []

    def start(self):
        pass

    def sample_once(self):
        pass

    def stop(self):
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampling disabled (USF_BENCH_SAMPLER=0)"], "samples": 0}


def make_sampler(index):
    if os.environ.get("USF_BENCH_SAMPLER", "1") == "0":
        return NullSampler()
    try:
        return NvmlSampler(index)
    except Exception:
        return ClockSampler(index)


def measured_peak_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md sustained)"


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_dram_bytes():
    p = os.path.join(ROOT, "profiles", "r2", "ncu_dram_bytes.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return {k: float(v) for k, v in j["bytes_per_launch"].items()}, j.get("source", "profiles/r2/ncu_dram_bytes.json")
        except Exception:
            pass
    return dict(NCU_DRAM_BYTES), "ncu --set full dram__bytes_read+write per launch, profiles/r1b_final/tc_kernels_full_raw.csv (round 1 capture)"


_FLUSH = {}


def timed_steps_with_flush(step, steps, dev, busy=None):
    """K steps timed one by one with CUDA events, a 256 MB write (> the 126 MB L2) between them outside the timed
    intervals: for workloads whose inputs would otherwise sit in L2 from one step to the next.  -> (total ms, last result)"""
    buf = _FLUSH.get(dev)
    if buf is None:
        buf = _FLUSH[dev] = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    out = None
    for a, b in evs:
        buf.fill_(1)
        a.record()
        out = step()
        b.record()
    if busy is not None:
        busy(evs[-1][1])            # e.g. clock sampling while the enqueued steps execute
    torch.cuda.synchronize(dev)
    return sum(a.elapsed_time(b) for a, b in evs), out


DUMP_LIMIT_BYTES = 64 << 20        # --dump-outputs: bytes written in all, over every rank


def dump_outputs(path, arrays, world=1):
    """Writes each `{name: tensor}` as `path/<name>.npy`, float32 (float64 stays float64).  Past this rank's share of
    DUMP_LIMIT_BYTES, every array keeps the same seeded sample of its rows, in order, so that runs stay comparable."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: (v if v.dtype == torch.float64 else v.float()).detach().cpu().numpy() for k, v in arrays.items()}
    limit = DUMP_LIMIT_BYTES // world
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = max(1, a.shape[0] * limit // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_reference_run(steps, warmup, rows, config=DEFAULT_CONFIG):
    """The reference's CPU PyTorch path for the same workload, fp32, eval() + no_grad() exactly as
    `adbench_wrapper.py:422-424`, all host threads: the reference's OWN unmodified `nf4ad.flows.NonUSFlow` +
    `nf4ad.transforms.MaskedAffineCoupling` (snapshot `oracle/_ref`, kind "reference") -- or, if the snapshot is missing,
    the oracle's restatement of them (kind "port") -- on the oracle's `src.usflows` / `pyro` shim (the genuine USFlows /
    pyro packages are not installable: no network, un-vendored, un-pinned).  3 warm-ups, median of >= 10 repeats with
    perf_counter (BASELINE.md section 3).  -> (samples/s from the median, cores, median ms, kind, last step's log_prob)"""
    import oracle
    kind = "reference" if oracle.ref_available() else "port"
    ns = oracle.load_ref() if kind == "reference" else oracle.load()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    flow = build_config_flow(ns, config, "cpu")
    d = CONFIGS[config][1]
    x = torch.randn(rows, d, generator=torch.Generator().manual_seed(42))
    with torch.no_grad():
        for _ in range(warmup):
            flow.log_prob(x)
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            lp = flow.log_prob(x)
            ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2] if len(ts) % 2 else 0.5 * (ts[len(ts) // 2 - 1] + ts[len(ts) // 2])
    return rows / med, cores, med * 1e3, kind, lp


def reference_train_run(device, rows, steps, warmup, config=DEFAULT_CONFIG):
    """BASELINE.md section 3, training baseline: the `ADBenchFlow.fit`-equivalent step of the reference
    (`adbench_wrapper.py:375-392`: zero_grad, loss = -log_prob(batch).mean(), backward, torch.optim.Adam step, the loss
    read back on the host) with the reference's own classes on the oracle's src.usflows / pyro shim, in torch eager --
    on the host cores (`device` "cpu") or on the B200 (ATen + cuBLAS; none of this repo's kernels).  Host wall clock
    around whole steps (each ends with the reference's own host read of the loss, i.e. a device sync), median.
    -> dict, or {"error": ...}."""
    import oracle
    out = {"batch": rows, "steps": steps, "warmup": warmup}
    try:
        ns = oracle.load_ref() if oracle.ref_available() else oracle.load()
        flow = build_config_flow(ns, config, device).train()
        opt = torch.optim.Adam(flow.parameters(), lr=1e-4)
        d = CONFIGS[config][1]
        x = torch.randn(rows, d, generator=torch.Generator().manual_seed(42)).to(device)
        ts, last = [], float("nan")
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            opt.zero_grad()
            loss = -flow.log_prob(x).mean()
            loss.backward()
            opt.step()
            last = float(loss.detach().cpu())
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
        ts.sort()
        med = ts[len(ts) // 2] if len(ts) % 2 else 0.5 * (ts[len(ts) // 2 - 1] + ts[len(ts) // 2])
        out.update({"value": rows / med, "unit": "samples/s", "ms_per_step": med * 1e3, "finite": last == last})
        del flow, opt, x
    except Exception as e:
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    return out


def torch_eager_gpu_run(steps, warmup, rows, dev, config=DEFAULT_CONFIG):
    """SURVEY 8(d): "also record torch-eager ON THE B200 (cuBLAS / ATen) as the existing GPU kernels to beat".  The same
    classes as `cpu_reference_run` (the reference's own NonUSFlow + MaskedAffineCoupling on the oracle's src.usflows / pyro
    shim), moved to the GPU with `.to(device)` and scored exactly as `adbench_wrapper.py:419-424` does: fp32, eval(),
    no_grad(), one call on the whole batch -- every layer an ATen op, the GEMMs cuBLAS SGEMM (torch's default
    `allow_tf32 = False`) and, second, cuBLAS TF32 (`allow_tf32 = True`: the tensor-core form of the stock path).
    None of this repo's kernels run here.  Part of the cpu_baseline leg (a baseline, never the product path).
    -> dict, or {"error": ...} if the shim does not run on this device."""
    import oracle
    out = {"api": "reference NonUSFlow.log_prob on cuda through torch eager (ATen + cuBLAS), fp32, eval()+no_grad()",
           "rows": rows, "steps": steps, "warmup": warmup}
    try:
        kind = "reference" if oracle.ref_available() else "port"
        ns = oracle.load_ref() if kind == "reference" else oracle.load()
        out["kind"] = kind
        flow = build_config_flow(ns, config, dev)
        d = CONFIGS[config][1]
        x = torch.randn(rows, d, generator=torch.Generator().manual_seed(42)).to(dev)
        prev = torch.backends.cuda.matmul.allow_tf32
        try:
            for tag, tf32 in (("fp32", False), ("tf32", True)):
                torch.backends.cuda.matmul.allow_tf32 = tf32
                with torch.no_grad():
                    for _ in range(warmup):
                        flow.log_prob(x)
                    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
                    for a, b in evs:
                        a.record()
                        lp = flow.log_prob(x)
                        b.record()
                torch.cuda.synchronize(dev)
                ts = sorted(a.elapsed_time(b) for a, b in evs)
                med = ts[len(ts) // 2] if len(ts) % 2 else 0.5 * (ts[len(ts) // 2 - 1] + ts[len(ts) // 2])
                out[tag] = {"value": rows / (med * 1e-3), "unit": "samples/s", "ms_per_step": med,
                            "finite": bool(torch.isfinite(lp).all())}
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        del flow, x
        torch.cuda.empty_cache()
    except Exception as e:                      # a baseline must never take the bench line down with it
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x2", "tf32x3", "fp32", "auto"])
    ap.add_argument("--rows", type=int, default=ROWS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--prewarm-s", type=float, default=1.0, help="untimed clock pre-warm (0 for profiler runs)")
    ap.add_argument("--train-steps", type=int, default=10, help="timed training steps (0 disables the leg)")
    ap.add_argument("--train-rows", type=int, default=4096, help="per-GPU training batch")
    ap.add_argument("--config", default=DEFAULT_CONFIG, choices=sorted(CONFIGS), help="BASELINE.json config shape to bench")
    ap.add_argument("--no-configs", dest="configs", action="store_false", help="skip the short per-config lines")
    ap.add_argument("--no-sweep", dest="sweep", action="store_false", help="skip the batch-size sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the log_prob the last timed step returned to DIR/log_prob.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    # a run that stops making progress (a collective waiting for a rank that died, a hung teardown) must not sit on the
    # GPUs: after USF_BENCH_TIMEOUT_S seconds every thread's stack goes to stderr and the process exits non-zero
    import faulthandler
    faulthandler.dump_traceback_later(float(os.environ.get("USF_BENCH_TIMEOUT_S", "1500")), exit=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ckind, cD, cK, ccond, cbase, cgain, ckw, calg, cbound = CONFIGS[args.config]
    config = {"workload": f"{args.config}: {ckind} log_prob scoring, D={cD}, K={cK}, conditioner {ccond[0]} {ccond[1]}, "
                          f"{'LU+Householder' if ckw.get('householder', 1) else 'LU'} conjugation, {cbase} base"
                          + (" (BASELINE.json configs[1], MNIST shape: MLP 784-256-256-1568)" if args.config == DEFAULT_CONFIG else ""),
              "rows_per_gpu": args.rows, "global_rows": args.rows * max(world, 1), "parallelism": f"batch-shard x{world}",
              "l2_policy": f"inputs larger than L2 ({args.rows * cD * 4 / 1e6:.0f} MB fp32 per GPU), no flush needed"
                           if args.rows * cD * 4 > 126e6 else "L2 flushed between timed steps (256 MB write)",
              "weights": f"seeded init (seed 0), last conditioner layer x{cgain}"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        # BASELINE.md section 3: the same workload (B = rows per GPU of our arm) on the host cores.  A step is one
        # log_prob call over the whole batch; if K + W steps of it would not end within a few minutes the step becomes a
        # bounded row sample of it (said in cpu_baseline.sample)
        rows = args.rows
        t_probe = cpu_reference_run(1, 1, min(rows, 4096), args.config)[2] * 1e-3 * rows / min(rows, 4096)
        budget_s = 240.0
        if (args.steps + args.warmup) * t_probe > budget_s:
            rows = max(1024, int(rows * budget_s / ((args.steps + args.warmup) * t_probe)) // 1024 * 1024)
        v, cores, ms, kind, lp = cpu_reference_run(args.steps, args.warmup, rows, args.config)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"log_prob": lp})
        v32, _, ms32, _, _ = cpu_reference_run(max(args.steps, 10), 3, CPU_SMALL_ROWS, args.config)
        line = {"impl": "reference", "metric": "log_prob samples/sec", "value": v, "unit": "samples/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": kind,
                                 "sample": f"{rows} rows per step ({'the full batch' if rows == args.rows else 'bounded sample of the ' + str(args.rows) + '-row batch'}), "
                                           f"median of {args.steps} steps after {args.warmup} warm-ups; the reference's own NonUSFlow + "
                                           "MaskedAffineCoupling (oracle/_ref snapshot) on the oracle's src.usflows/pyro shim "
                                           "(real USFlows/pyro not installable), fp32, eval()+no_grad()",
                                 "small_batch": {"rows": CPU_SMALL_ROWS, "value": v32, "ms_per_step": ms32}},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (B200)
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import nf4ad_b200
    from nf4ad_b200 import _lib
    from nf4ad_b200.parallel import ShardedScorer, bind_to_gpu_numa
    # multi-rank host: pin this rank to its GPU's NUMA node BEFORE the first host buffer exists (parallel.bind_to_gpu_numa)
    numa = bind_to_gpu_numa(local, local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))) if world > 1 else {"bound": False}
    P = nf4ad_b200.namespace()
    flow = build_config_flow(P, args.config, dev)
    flow.precision = args.precision
    B = args.rows
    D = cD
    gen = torch.Generator().manual_seed(42 + rank)
    x_host = torch.randn(B, D, generator=gen).pin_memory()
    x = x_host.to(dev)
    scorer = ShardedScorer(flow)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput: K steps of the fused launch chain -----------------------------------
    with torch.no_grad():
        # pre-warm: a step is only ~2-3 ms, so run the same step for >= 1 s first to bring the GPU out of its
        # idle P-state to steady clocks (untimed), then the W warm-up steps the contract asks for
        # (untimed) until the step time has settled: a fresh process can sit in a slow state for a second or more
        # (idle clocks / power state; steps of 3-13 ms were seen), which must not leak into the timed region.  Batches
        # of 20 steps are timed with events until two consecutive batches agree within 3 %, for at least
        # `prewarm_s` and at most 8 s.
        t_pw = time.perf_counter()
        prev_ms = None
        while args.prewarm_s > 0:
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for _ in range(20):
                lp = scorer.score_local(x)
            p1.record()
            torch.cuda.synchronize()
            cur_ms = p0.elapsed_time(p1)
            elapsed = time.perf_counter() - t_pw
            settled = prev_ms is not None and abs(cur_ms - prev_ms) <= 0.03 * prev_ms
            if (elapsed >= args.prewarm_s and settled) or elapsed > 8.0:
                break
            prev_ms = cur_ms
        for _ in range(args.warmup):
            lp = scorer.score_local(x)
        barrier()
        # Clock / throttle sampling DURING the timed region without touching its launches: the K steps are enqueued first
        # (asynchronous, ~0.04 ms of host time each), then NVML is polled from this thread while the GPU works through
        # them.  (A sampling thread beside the launching loop shares a driver lock with the launches: on some boxes every
        # query stalled the loop for milliseconds -- a run of this file measured 12 ms per step at 0.07 ms kernels.)
        sampler = make_sampler(local)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def sample_while_busy(done_event, limit=40):
            if rank != 0:
                return
            n = 0
            while n < limit and not done_event.query():
                sampler.sample_once()
                n += 1
            if n == 0:
                sampler.sample_once()
        small_input = B * D * 4 <= 126e6          # fits the 126 MB L2: flush it between timed steps (untimed)
        barrier()
        t_host = time.perf_counter()
        if not small_input:
            e0.record()
            for i in range(args.steps):
                lp = scorer.score_local(x)
            host_enqueue_ms = (time.perf_counter() - t_host) * 1e3 / args.steps   # host time to enqueue one step
            e1.record()
            sample_while_busy(e1)              # kernels are in flight: every launch of the region is already enqueued
            barrier()
            ms_total = e0.elapsed_time(e1)
        else:
            ms_total, lp = timed_steps_with_flush(lambda: scorer.score_local(x), args.steps, dev, busy=sample_while_busy)
            host_enqueue_ms = float("nan")
            barrier()
        gstats = (ctypes.c_longlong * 4)()
        gfail = ctypes.create_string_buffer(160)
        _lib.lib().usf_debug_graph_stats(gstats, gfail, 160)
        graph_info = {"replays": int(gstats[0]), "captures": int(gstats[1]), "failed_captures": int(gstats[2]),
                      "eager_runs": int(gstats[3]), "last_failure": gfail.value.decode()}
        clocks = sampler.stop() if rank == 0 else None
        launches_per_step = flow.last_launches
        eff_main, cal_err = flow.effective_precision, flow.bf16_calibration_err      # the tier the timed steps ran at
        fpr_main = flow._stack(True, dev, eff_main).flops_per_row()
        assert launches_per_step > 0, "fused CUDA path did not run"
        assert bool(torch.isfinite(lp).all())
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"log_prob" if world == 1 else f"log_prob_rank{rank}": lp}, world)

        # ---- end to end through the public API: pinned host rows -> H2D -> log_prob -> scores D2H, every step
        # (the call sequence of ADBenchFlow.predict_score, adbench_wrapper.py:419-433) + score gather to rank 0
        for _ in range(12):        # untimed: covers the scorer's trial calls over its fp32-head candidates (parallel.py)
            scorer.predict_score_host(x_host)
        barrier()
        t0 = time.perf_counter()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            scores = scorer.predict_score_host(x_host, gather=True)
        f1.record()
        barrier()
        e2e_ms = max(f0.elapsed_time(f1), (time.perf_counter() - t0) * 1e3 if world == 1 else 0.0)

        # ---- what the link alone allows: the same pinned rows copied to the device, nothing else (all ranks at once).  When
        # this is as slow as the end-to-end call, the call is bound by the host -> device feed (PCIe / host DRAM shared by
        # the ranks of one host), not by the scoring pipeline.
        x_land = torch.empty_like(x)
        for _ in range(2):
            x_land.copy_(x_host, non_blocking=True)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(args.steps):
            x_land.copy_(x_host, non_blocking=True)
        c1.record()
        barrier()
        h2d_only_ms = c0.elapsed_time(c1)
        del x_land

        # ---- the same call as the reference's callers make it: a PAGEABLE numpy array through
        # ADBenchFlow.predict_score (adbench_wrapper.py:406-433: torch.FloatTensor(X).to(device) ... .cpu().numpy());
        # host wall clock around the blocking calls (the result is a host array)
        import numpy as np
        from nf4ad_b200.adbench import ADBenchFlow
        X_np = np.array(x_host.numpy(), copy=True)              # a plain (pageable) copy, as a caller's array is
        wrapper = ADBenchFlow(flow_model=flow, device=str(dev), verbose=False)
        score_np = (lambda: wrapper.predict_score(X_np)) if world == 1 else \
            (lambda: scorer.predict_score_host(torch.from_numpy(X_np)).numpy())
        for _ in range(3):
            score_np()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            s_np = score_np()
        torch.cuda.synchronize()
        pageable_ms = (time.perf_counter() - t0) * 1e3
        pageable_h2d = int(getattr(wrapper, "_scorer", scorer).last_h2d_bytes) if world == 1 else int(scorer.last_h2d_bytes)
        assert s_np.shape == (B,) and bool(np.isfinite(s_np).all())
        barrier()

        # ---- per-launch device time of every kernel of one step (CUDA events on the launching stream)
        n_prof = launches_per_step * 3
        _lib.check(_lib.lib().usf_profile_begin(n_prof + 8))
        for _ in range(3):
            scorer.score_local(x)
        ms = (ctypes.c_float * (n_prof + 8))()
        tags = (ctypes.c_int * (n_prof + 8))()
        n = ctypes.c_int(0)
        _lib.check(_lib.lib().usf_profile_end(ms, tags, ctypes.byref(n)))
        per_tag = {}
        for i in range(n.value):
            per_tag.setdefault(tags[i], []).append(ms[i])
    # ---- batch-size sweep of the resident-input scoring call (SURVEY 8d: 1 024 ... 1 048 576 plus the reference's
    # own small batches); rank 0 only, short, reported as extra information
    sweep = {}
    if rank == 0 and args.sweep:
        with torch.no_grad():
            for rows_s in (64, 1024, 16384, 262144):
                for prec in ("bf16", "bf16x2", "tf32x3", "fp32"):
                    # bf16x2 = what the default precision ("auto") runs for D >= 128; fp32 FFMA only at small sizes
                    if (prec == "fp32" and rows_s > 16384) or (prec == "tf32x3" and rows_s < 16384):
                        continue
                    flow.precision = prec
                    xs = torch.randn(rows_s, D, device=dev)
                    if prec == "bf16":
                        flow.bf16_trust = True      # sweep entries are labelled by the kernels that ran
                    for _ in range(5):
                        flow.log_prob(xs)
                    torch.cuda.synchronize()
                    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    reps = 20 if rows_s <= 16384 else 5
                    h0.record()
                    for _ in range(reps):
                        flow.log_prob(xs)
                    h1.record()
                    torch.cuda.synchronize()
                    ms_s = h0.elapsed_time(h1) / reps
                    sweep[f"{prec}_rows{rows_s}"] = {"ms_per_call": ms_s, "samples_per_s": rows_s / (ms_s * 1e-3)}
            flow.precision = args.precision
            flow.bf16_trust = False
            flow.invalidate_cache()

    # ---- every other BASELINE.json config shape (north star: "throughput on synthetic data of EACH config's shape at 1, 2,
    # 4 and 8 GPUs ... as a fraction of the roofline"): short resident-input runs, every rank scores its own 65536 rows
    # (weak scaling like the headline), device-timed, max over ranks; reported under "configs"
    per_config = {}
    if args.configs:
        names = [n for n in CONFIGS if n != args.config]
        times = torch.zeros(len(names), device=dev, dtype=torch.float64)
        meta = []
        with torch.no_grad():
            for i, name in enumerate(names):
                kind_, d_, k_, cond_, base_, gain_, kw_, alg_, bound_ = CONFIGS[name]
                f_ = build_config_flow(P, name, dev)
                f_.precision = args.precision
                xs = torch.randn(ROWS_PER_GPU, d_, device=dev, generator=torch.Generator(device=dev).manual_seed(7 + rank))
                # warm-up with the call pattern of the timed steps (the result of the previous step is still alive when the
                # next one allocates its output: two alternating output buffers = two launch-chain graphs to capture)
                timed_steps_with_flush(lambda: f_.log_prob(xs), 8, dev)
                g0 = (ctypes.c_longlong * 4)()
                _lib.lib().usf_debug_graph_stats(g0, None, 0)
                ms_c, _ = timed_steps_with_flush(lambda: f_.log_prob(xs), 20, dev)
                g1 = (ctypes.c_longlong * 4)()
                _lib.lib().usf_debug_graph_stats(g1, None, 0)
                times[i] = ms_c / 20
                cs_ = f_._stack(True, dev, f_.effective_precision)
                fl_ = cs_.flops_per_row() if cs_ is not None else {}
                meta.append((f_.last_launches, f_.effective_precision, sum(v[1] for v in fl_.values()),
                             sum(v[0] for v in fl_.values()), int(g1[0] - g0[0]), int(g1[3] - g0[3])))
                del f_, xs, cs_
        if world > 1:
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
        peak_t, _ = measured_peak_tflops()
        peak_h, _ = measured_peak_hbm()
        for i, name in enumerate(names):
            kind_, d_, k_, cond_, base_, gain_, kw_, alg_, bound_ = CONFIGS[name]
            ms_c = float(times[i])
            launches_, eff_, useful_, executed_, replays_, eager_ = meta[i]
            entry = {"value": ROWS_PER_GPU * world / (ms_c * 1e-3), "unit": "samples/s", "ms_per_step": ms_c,
                     "rows_per_gpu": ROWS_PER_GPU, "launches_per_step": launches_, "effective_precision": eff_,
                     "graph_replays_of_20": replays_, "eager_chains_of_20": eager_,
                     "alg_mflop_per_sample": alg_, "bound": bound_}
            if bound_ == "tensor":
                ach = useful_ * ROWS_PER_GPU / (ms_c * 1e-3) / 1e12
                entry["roofline"] = {"achieved": ach, "peak": peak_t, "unit": "TFLOP/s", "frac": ach / peak_t,
                                     "frac_executed_padded": executed_ * ROWS_PER_GPU / (ms_c * 1e-3) / 1e12 / peak_t,
                                     "frac_algorithmic": alg_ * 1e6 * ROWS_PER_GPU / (ms_c * 1e-3) / 1e12 / peak_t,
                                     "note": "bf16 peak; a stack routed to 3xTF32 (effective_precision) is bound at 1/6 of it"}
            else:
                ach = (4 * d_ + 4) * ROWS_PER_GPU / (ms_c * 1e-3) / 1e9
                entry["roofline"] = {"achieved": ach, "peak": peak_h, "unit": "GB/s", "frac": ach / peak_h}
            per_config[name] = entry

    # ---- training step (second BASELINE metric): fwd + hand-written backward kernels + (DP all-reduce) + Adam
    train_ms, train_B, train_steps, train_graph = float("nan"), args.train_rows, args.train_steps, False
    train32_ms = train3_ms = train_small_ms = float("nan")
    if train_steps > 0:
        from nf4ad_b200.parallel import DataParallelTrainer
        from nf4ad_b200.optim import FusedAdam
        xb = x[:train_B]
        for prec in ("bf16", "tf32x3", "fp32"):
            # "bf16" = mixed precision: bf16 tensor-core GEMMs with fp32 accumulation, fp32 parameters / gradients /
            # Adam state, LU layers applied through their per-step dense inverse; "tf32x3" = the same step with
            # 3xTF32 tensor-core GEMMs (fp32-grade); "fp32" = the all-fp32 kernels
            tflow = build_config_flow(P, args.config, dev).train()
            tflow.precision = prec
            opt = FusedAdam(tflow.parameters(), lr=1e-4)   # torch.optim.Adam's update via usf_adam_step; the step replays as one CUDA graph
            trainer = DataParallelTrainer(tflow, opt)
            trainer.broadcast_parameters()
            for _ in range(5):          # 3 eager steps + capture + first replay (single rank), all untimed
                trainer.step(xb)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(train_steps):
                loss = trainer.step(xb)
            g1.record()
            barrier()
            if prec == "bf16":
                train_ms = g0.elapsed_time(g1)
                train_graph = trainer.graph_replays > 0
            elif prec == "tf32x3":
                train3_ms = g0.elapsed_time(g1)
            else:
                train32_ms = g0.elapsed_time(g1)
            assert bool(torch.isfinite(loss))
            del tflow, opt, trainer
        # the reference's own batch size (SURVEY 8d: training B per GPU = 64 and 4096; `adbench_wrapper.py:310`): the step
        # is launch / dependency-latency bound there, which is what the one-graph replay is for
        # (single-GPU line only: the multi-rank runs report the B = 4096 step above)
        if world == 1:
            try:
                xs = x[:TRAIN_SMALL_ROWS]
                tflow = build_config_flow(P, args.config, dev).train()
                tflow.precision = "bf16"
                opt = FusedAdam(tflow.parameters(), lr=1e-4)
                trainer = DataParallelTrainer(tflow, opt)
                for _ in range(5):
                    trainer.step(xs)
                torch.cuda.synchronize(dev)
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                for _ in range(train_steps):
                    loss = trainer.step(xs)
                g1.record()
                torch.cuda.synchronize(dev)
                if bool(torch.isfinite(loss)):
                    train_small_ms = g0.elapsed_time(g1)
                del tflow, opt, trainer
            except Exception as e:              # an extra line must not take the headline down
                print(f"bench: small-batch training line skipped ({type(e).__name__}: {e})", file=sys.stderr, flush=True)
    t = torch.tensor([ms_total, e2e_ms, train_ms, train32_ms, train3_ms, pageable_ms, h2d_only_ms, train_small_ms],
                     device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, train_ms, train32_ms, train3_ms, pageable_ms, h2d_only_ms, train_small_ms = (float(v) for v in t)

    if rank == 0:
        steps_prof = 3
        peak, peak_src = measured_peak_tflops()
        peak_hbm, peak_hbm_src = measured_peak_hbm()
        value = B * world * args.steps / (ms_total * 1e-3)
        e2e_value = B * world * args.steps / (e2e_ms * 1e-3)
        step_ms = ms_total / args.steps
        # ---- roofline on what the kernels execute: FLOPs per launch from the packed descriptors (CompiledStack.
        # flops_per_row: `useful` = the GEMM shapes without tile padding, `executed` = with it), time per launch from the
        # CUDA events usf_stack_run recorded around every launch of three profiled steps
        tag_kind = {0: "pack_input", 1: "affine_gemm", 2: "conditioner+coupling", 3: "conditioner+coupling",
                    4: "final_gemm+base", 5: "conditioner+coupling", 6: "whole_stack"}
        tag_name = {0: "pack_input", 1: "affine_gemm", 2: "mlp_hidden_gemm", 3: "mlp_last_gemm+coupling", 4: "final_gemm+base",
                    5: "fused_conditioner+coupling", 6: "whole_stack_kernel"}
        eff, fpr = eff_main, fpr_main
        dram, dram_src = ncu_dram_bytes()
        gemm_name = {"bf16": "usf_tc_gemm_kernel", "tf32x3": "usf_tc3_gemm_kernel", "bf16x2": "usf_tcb2_gemm_kernel",
                     "fp32": "usf_simt_gemm_kernel"}[eff]
        kernel_of = {"affine_gemm": gemm_name, "final_gemm+base": gemm_name,
                     "conditioner+coupling": "usf_tc_mlp_coupling_kernel" if 5 in per_tag else gemm_name}
        by_kind, kind_ms = {}, {}
        for tg, v in per_tag.items():
            kind_ms.setdefault(tag_kind[tg], []).extend(v)
        for kind, v in kind_ms.items():
            n_launch = len(v) / steps_prof
            avg_ms = sum(v) / len(v)
            e = {"launches_per_step": n_launch, "avg_launch_ms": avg_ms, "share_of_step": sum(v) / steps_prof / step_ms}
            if kind in fpr:
                ex, us = fpr[kind]
                e.update({"kernel": kernel_of[kind], "gflop_useful_per_launch": us * B / n_launch / 1e9,
                          "gflop_executed_per_launch": ex * B / n_launch / 1e9,
                          "achieved_tflops": us * B / n_launch / (avg_ms * 1e-3) / 1e12,
                          "frac": us * B / n_launch / (avg_ms * 1e-3) / 1e12 / peak,
                          "frac_executed_padded": ex * B / n_launch / (avg_ms * 1e-3) / 1e12 / peak,
                          "dram_bytes_per_launch_ncu": dram.get(kind)})
            elif kind == "whole_stack":   # small event shapes: ONE kernel, rows in shared memory across all layers
                bytes_ = B * (4 * D + 4)
                us = sum(v[1] for v in fpr.values())
                e.update({"kernel": "usf_small_stack_kernel", "achieved_gbs": bytes_ / (avg_ms * 1e-3) / 1e9,
                          "frac": bytes_ / (avg_ms * 1e-3) / 1e9 / peak_hbm, "bound": "hbm",
                          "achieved_tflops": us * B / (avg_ms * 1e-3) / 1e12, "note": "fp32 FFMA kernel"})
            else:   # pack_input: HBM-bound, reads 4*D and writes 2*ld (bf16) / 4*ld bytes per row
                ld = (D + 15) // 16 * 16
                bytes_ = B * (4 * D + (2 if eff == "bf16" else 4) * ld + 4)
                e.update({"kernel": "usf_convert_rows_kernel", "achieved_gbs": bytes_ / (avg_ms * 1e-3) / 1e9,
                          "frac": bytes_ / (avg_ms * 1e-3) / 1e9 / peak_hbm, "bound": "hbm"})
            by_kind[kind] = e
        tensor_kinds = [k for k in by_kind if k in fpr]
        if not tensor_kinds:           # whole-stack kernel: report it against the HBM roofline
            ws = by_kind["whole_stack"]
            by_kind["whole_stack"].update({"achieved_tflops": ws.get("achieved_tflops", 0.0)})
            fpr = dict(fpr, whole_stack=(sum(v[0] for v in fpr_main.values()), sum(v[1] for v in fpr_main.values())))
            for k in ("affine_gemm", "conditioner+coupling", "final_gemm+base"):
                fpr.pop(k, None)
            tensor_kinds = ["whole_stack"]
        dominant = max(tensor_kinds, key=lambda k: by_kind[k]["share_of_step"])
        exec_per_row = sum(v[0] for v in fpr.values())
        useful_per_row = sum(v[1] for v in fpr.values())
        gemm_ms_per_step = sum(sum(v) for k, v in kind_ms.items() if k in fpr) / steps_prof
        n_gemm_per_step = sum(len(v) for k, v in kind_ms.items() if k in fpr) / steps_prof
        dk = by_kind[dominant]
        line = {
            "metric": "log_prob samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "tf32x3": "tf32x3 (fp32 operands as hi+lo on tcgen05)", "fp32": "f32",
                      "bf16x2": "bf16x2 (bf16 hi+lo operand pairs on tcgen05, fp32-grade)"}[eff],
            "requested_precision": args.precision, "effective_precision": eff,
            "bf16_calibration_err": cal_err, "data": "synthetic", "config": config,
            "clocks": clocks, "host_enqueue_ms_per_step": host_enqueue_ms, "graph": graph_info,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(scorer.last_h2d_bytes),
                    "d2h_bytes_per_step": B * 4, "ms_per_step": e2e_ms / args.steps,
                    "api": "ShardedScorer.predict_score_host(pinned fp32 rows): the ADBenchFlow.predict_score call sequence",
                    "host_input_bytes_per_step": B * D * 4,
                    "h2d_copy_only": {"ms_per_step": h2d_only_ms / args.steps,
                                      "gbs_per_gpu": B * D * 4 / (h2d_only_ms / args.steps * 1e-3) / 1e9,
                                      "note": "the same pinned fp32 rows copied to the device and nothing else, all ranks "
                                              "at once: the floor the host -> device feed sets for one call"},
                    "host_narrowing": bool(scorer.host_bf16 and eff == "bf16"),
                    "host_threads": int(scorer.host_threads), "numa": numa,
                    "fp32_head_rows": (scorer._tune.get((B, D), {}).get("best", None) if scorer.host_bf16 else None)},
            "e2e_pageable": {"value": B * world * args.steps / (pageable_ms * 1e-3), "unit": "samples/s",
                             "ms_per_step": pageable_ms / args.steps, "h2d_bytes_per_step": pageable_h2d,
                             "d2h_bytes_per_step": B * 4,
                             "api": "nf4ad_b200.adbench.ADBenchFlow.predict_score(pageable numpy array) "
                                    "(adbench_wrapper.py:406-433), host wall clock" if world == 1 else
                                    "ShardedScorer.predict_score_host(pageable rows) per rank, host wall clock"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": dk.get("bound", "tensor"), "kernel": dk["kernel"], "kind": dominant,
                         "why_this_kernel": "largest share of the step's device time (launch_ms_by_kind)",
                         "achieved": dk["achieved_gbs"] if dk.get("bound") == "hbm" else dk["achieved_tflops"],
                         "peak": peak_hbm if dk.get("bound") == "hbm" else peak,
                         "unit": "GB/s" if dk.get("bound") == "hbm" else "TFLOP/s", "frac": dk["frac"],
                         "flop_basis": "executed useful FLOPs of this kernel per launch (GEMM shapes of the packed descriptors "
                                       "without tile padding) / its mean CUDA-event time",
                         "peak_source": peak_src + {"tf32x3": " -- bf16 figure; this run executed 3xTF32 MMAs (1/6 of it)",
                                                    "bf16x2": " -- bf16 figure; this run executed 3 bf16 MMAs per product (1/3 of it)"}.get(eff, ""),
                         "traffic": dram.get(dominant), "traffic_source": dram_src,
                         "by_kind": by_kind,
                         "step": {"flop_useful_per_sample": useful_per_row, "flop_executed_padded_per_sample": exec_per_row,
                                  "achieved": useful_per_row * B / (step_ms * 1e-3) / 1e12,
                                  "frac": useful_per_row * B / (step_ms * 1e-3) / 1e12 / peak,
                                  "gemm_share_of_step": gemm_ms_per_step / step_ms,
                                  "gemm_launches_per_step": n_gemm_per_step},
                         "frac_algorithmic": calg * 1e6 * B / (step_ms * 1e-3) / 1e12 / peak,
                         "alg_flop_per_sample": calg * 1e6,
                         "alg_note": "SURVEY 8d count (2 dense maps per block, conditioner once); the chain executes fewer FLOPs "
                                     "because adjacent affine maps are merged at weight-prep time",
                         "launch_ms_by_kind": {tag_name[k]: sum(v) / len(v) for k, v in sorted(per_tag.items())},
                         "launches_by_kind": {tag_name[k]: len(v) // steps_prof for k, v in sorted(per_tag.items())}},
        }
        if per_config:
            line["configs"] = per_config
        if sweep:
            line["sweep"] = sweep
        if train_steps > 0:
            line["train"] = {"metric": "train samples/sec (fwd + bwd + Adam; bf16 tensor-core GEMMs, fp32 accumulate / "
                                       "parameters / optimizer state)", "graph_replay": bool(train_graph),
                             "value": train_B * world * train_steps / (train_ms * 1e-3), "unit": "samples/s",
                             "batch_per_gpu": train_B, "steps": train_steps, "ms_per_step": train_ms / train_steps,
                             "tf32x3_path": {"value": train_B * world * train_steps / (train3_ms * 1e-3),
                                             "ms_per_step": train3_ms / train_steps},
                             "fp32_path": {"value": train_B * world * train_steps / (train32_ms * 1e-3),
                                           "ms_per_step": train32_ms / train_steps}}
            if world == 1 and train_small_ms == train_small_ms:          # (single-GPU line; not NaN: measured on this run)
                line["train"]["small_batch"] = {
                    "batch_per_gpu": TRAIN_SMALL_ROWS,
                    "value": TRAIN_SMALL_ROWS * world * train_steps / (train_small_ms * 1e-3),
                    "ms_per_step": train_small_ms / train_steps,
                    "note": "the reference's own batch size (adbench_wrapper.py:310), bf16 tier, one CUDA-graph replay per step"}
        if world == 1 and not args.no_cpu_baseline:
            # BASELINE.md section 3: B = 65536 (and 32), 3 warm-ups, median of 10 -- about 30 s of host work
            v, cores, cms, kind, _ = cpu_reference_run(10, 3, CPU_ROWS, args.config)
            v32, _, cms32, _, _ = cpu_reference_run(10, 3, CPU_SMALL_ROWS, args.config)
            line["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": cores, "kind": kind,
                                    "sample": f"{CPU_ROWS} rows per step, 3 warm-ups, median of 10 steps ({cms:.0f} ms), fp32, "
                                              f"{cores} threads; the reference's own NonUSFlow + MaskedAffineCoupling "
                                              "(oracle/_ref) on the oracle's src.usflows/pyro shim",
                                    "small_batch": {"rows": CPU_SMALL_ROWS, "value": v32, "ms_per_step": cms32}}
            # the same leg also checks the timed GPU path against the fp64 oracle on the first 256 rows
            import oracle
            fo = build_config_flow(oracle.load(), args.config, "cpu").double()
            with torch.no_grad():
                ref = fo.log_prob(x_host[:256].double())
                got = flow.log_prob(x[:256]).double().cpu()
            line["cpu_baseline"]["gpu_vs_oracle_fp64_max_rel_err"] = float(((got - ref).abs() / ref.abs().clamp_min(1.0)).max())
            # north star: "inverse(forward(x)) round-trip error reported" -- data -> latent -> data through both fused
            # directions of the timed flow, worst coordinate relative to its row's largest magnitude, per tier
            try:
                rt = {}
                keep = flow.precision
                with torch.no_grad():
                    xs = x[:256].float()
                    scale_ = xs.abs().amax(dim=1, keepdim=True).clamp_min(1.0)
                    for tier_ in dict.fromkeys((keep, "auto")):
                        flow.precision = tier_
                        back = flow.latent_to_data(flow.backward(xs))
                        rt[f"{tier_}->{flow.effective_precision}"] = float(((back - xs).abs() / scale_).max())
                flow.precision = keep
                line["cpu_baseline"]["round_trip_max_err"] = rt
            except Exception as e:
                flow.precision = keep
                line["cpu_baseline"]["round_trip_max_err"] = {"error": f"{type(e).__name__}: {e}"[:200]}
            # ... and records the stock GPU path beside the CPU one (SURVEY 8d): the same reference classes in torch eager on
            # this B200 (ATen + cuBLAS), none of our kernels
            line["cpu_baseline"]["torch_eager_b200"] = torch_eager_gpu_run(10, 3, CPU_ROWS, dev, args.config)
            # the second BASELINE metric's baselines (BASELINE.md section 3): the reference's training step at B = 64 and
            # 4096, on the host cores and in torch eager on this B200
            if train_steps > 0:
                line["cpu_baseline"]["train"] = {
                    "unit": "samples/s", "cores": cores,
                    "what": "reference classes, zero_grad + -log_prob.mean() + backward + torch.optim.Adam step + host read "
                            "of the loss (adbench_wrapper.py:375-392), torch eager, fp32, median of whole-step wall times",
                    "cpu": {f"B{b}": reference_train_run("cpu", b, n, 1, args.config) for b, n in ((TRAIN_SMALL_ROWS, 10), (train_B, 3))},
                    "torch_eager_b200": {f"B{b}": reference_train_run(dev, b, 10, 3, args.config) for b in (TRAIN_SMALL_ROWS, train_B)}}
        print(json.dumps(line), flush=True)
    if world > 1:
        # every rank has contributed to the line above (the max-over-ranks all_reduce); leave together, and leave through
        # os._exit: interpreter teardown with CUDA graphs that hold NCCL kernels alive next to a destroyed process group
        # hung a 2-GPU run of this file once (the line was printed, the processes never exited)
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
