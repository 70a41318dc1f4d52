"""Cost of `Flow.log_prob_terms` against `log_prob` on the same flow and rows: log_prob with deterministic mode off (fp32
atomics), log_prob with it on (the slot form the terms call always runs) and log_prob_terms, taking turns in the same
process -- C2 at the bf16x2 and bf16 tiers, C4 D = 6 and D = 64 at "auto" (fp32), B = 65536 and 524288 rows.  Device
events around `REPS` calls after warm-up, the median of `ROUNDS` alternating rounds.  Card name and power limit are read
in the same run.

    python scripts/terms_bench.py [out.json]        (default profiles/r3/terms_bench.json)
"""
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import nf4ad_b200  # noqa: E402
from _cases import build_flow, randomize_constants, tame  # noqa: E402

CONFIGS = [
    # id, precision, kind, D, K, conditioner, base, gain, kwargs
    ("C2-D784", "bf16x2", "NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C2-D784", "bf16", "NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-D6", "auto", "NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-D64", "auto", "NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
]
ROWS = (65536, 524288)
ROUNDS, REPS = 5, 10


def timed(fn):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(REPS):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / REPS


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3", "terms_bench.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    P = nf4ad_b200.namespace()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi, "rounds": ROUNDS, "reps": REPS, "runs": []}
    for name, precision, kind, D, K, cond, base, gain, kw in CONFIGS:
        torch.manual_seed(D * 7 + K)
        flow = build_flow(P, kind, D, K, cond, base=base, **kw)
        tame(flow, gain)
        randomize_constants(flow, D * 7 + K)
        flow = flow.to("cuda").eval()
        flow.precision = precision
        for B in ROWS:
            x = torch.randn(B, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

            def lp(det):
                flow.deterministic = det
                return flow.log_prob(x)

            def terms():
                return flow.log_prob_terms(x)

            with torch.no_grad():
                lp(False)
                tier_lp, launches_lp = flow.effective_precision, flow.last_launches
                lp(True)
                launches_det = flow.last_launches
                t = terms()
                tier_t, launches_t = flow.effective_precision, flow.last_launches
                same = bool(torch.equal(t.log_prob, lp(True)))       # deterministic log_prob, bit for bit
                ms = {"log_prob": [], "log_prob_det": [], "terms": []}
                for _ in range(ROUNDS):
                    ms["log_prob"].append(timed(lambda: lp(False)))
                    ms["log_prob_det"].append(timed(lambda: lp(True)))
                    ms["terms"].append(timed(terms))
            med = {k: statistics.median(v) for k, v in ms.items()}
            row = {"config": name, "precision": precision, "tier": tier_t, "log_prob_tier": tier_lp, "rows": B,
                   "log_prob_ms": med["log_prob"], "log_prob_det_ms": med["log_prob_det"], "terms_ms": med["terms"],
                   "terms_over_log_prob": med["terms"] / med["log_prob"],
                   "terms_over_log_prob_det": med["terms"] / med["log_prob_det"],
                   "terms_rows_per_s": B / med["terms"] * 1e3,
                   "launches": {"log_prob": launches_lp, "log_prob_det": launches_det, "terms": launches_t},
                   "terms_log_prob_equals_det_log_prob": same,
                   "spread_ms": {k: [min(v), max(v)] for k, v in ms.items()}}
            print(json.dumps(row), flush=True)
            res["runs"].append(row)
            del x, t
            torch.cuda.empty_cache()
        del flow
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "nvidia_smi": smi}))


if __name__ == "__main__":
    main()
