"""Rows/s of `Flow.log_prob_and_grad` (the reverse launch chain) against the autograd route it replaces
(`x.requires_grad_()` + `log_prob` + `torch.autograd.grad` on the fp32 kernels), per shape at 65536 rows (inputs larger
than L2 at C2), device-event timing after warm-up, plus the grad-free `log_prob` of the same stack for scale and the
max per-row distance between the two gradients.  Card name and power limit are read in the same run.

    python scripts/grad_bench.py [out.json]        (default profiles/r3/grad_bench.json)
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import nf4ad_b200  # noqa: E402
from _cases import build_flow, randomize_constants, tame  # noqa: E402

SHAPES = [
    ("C2-D784", "NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-D64", "NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-D6", "NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
]
ROWS = 65536


def timed(fn, warmup=3, reps=10):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def autograd_route(flow, x):
    xr = x.clone().requires_grad_(True)
    lp = flow.log_prob(xr)
    return torch.autograd.grad(lp.sum(), xr)[0]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3", "grad_bench.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    P = nf4ad_b200.namespace()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi, "rows": ROWS, "shapes": []}
    for name, kind, D, K, cond, base, gain, kw in SHAPES:
        torch.manual_seed(D * 7 + K)
        flow = build_flow(P, kind, D, K, cond, base=base, **kw)
        tame(flow, gain)
        randomize_constants(flow, D * 7 + K)
        flow = flow.to("cuda").eval()
        x = torch.randn(ROWS, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
        _, g = flow.log_prob_and_grad(x)
        tier, launches = flow.last_grad_precision, flow.last_launches
        ms_fused = timed(lambda: flow.log_prob_and_grad(x))
        with torch.no_grad():
            ms_fwd = timed(lambda: flow.log_prob(x))
        fwd_tier = flow.effective_precision
        flow.precision = "fp32"
        g_a = autograd_route(flow, x)
        ms_auto = timed(lambda: autograd_route(flow, x), warmup=2, reps=5)
        err = float(((g.double() - g_a.double()).abs().amax(1) / g_a.double().abs().amax(1).clamp_min(1.0)).max())
        row = {"shape": name, "grad_tier": tier, "fused_ms": ms_fused, "fused_rows_per_s": ROWS / ms_fused * 1e3,
               "autograd_ms": ms_auto, "autograd_rows_per_s": ROWS / ms_auto * 1e3, "speedup": ms_auto / ms_fused,
               "log_prob_ms": ms_fwd, "log_prob_tier": fwd_tier, "grad_row_err_vs_autograd": err,
               "launches": launches}
        print(json.dumps(row), flush=True)
        res["shapes"].append(row)
        del flow, x, g, g_a
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "nvidia_smi": smi}))


if __name__ == "__main__":
    main()
