"""`Flow.log_prob_and_grad` at fp32 on small event shapes: the one-kernel path (usf_small_stack_grad_kernel) against the
reverse launch chain it replaces, in the same GPU session.

The library reads USF_SMALL_STACK once per process, so the chain runs in a worker subprocess started with
USF_SMALL_STACK=0; the two processes take turns on the GPU (per shape and batch size: new, old, new, old, ...).  Both
build the same flow from the same seed and score the same seeded rows; the worker hands its outputs back for the
comparison.  Device-event timing after warm-up; card name and power limit are read in the same run.

    python scripts/small_grad_bench.py [out.json]        (default profiles/r3/small_grad_bench.json)
"""
import json
import os
import subprocess
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
sys.path.insert(0, os.path.join(HERE, ".."))

SHAPES = {
    # name: kind, D, K, conditioner, base, gain, kwargs
    "C4-D6": ("NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C4-D64": ("NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "fixture-D32": ("NonUSFlow", 32, 3, ("mlp", [128]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C1-D2": ("USFlow", 2, 10, ("densenn1", [128, 128]), "usnormal", 0.5,
              dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
}
BATCHES = (64, 4096, 65536, 524288)
ROUNDS = 3


def make_flow(name):
    import nf4ad_b200
    from _cases import build_flow, randomize_constants, tame
    kind, D, K, cond, base, gain, kw = SHAPES[name]
    torch.manual_seed(D * 7 + K)
    flow = build_flow(nf4ad_b200.namespace(), kind, D, K, cond, base=base, **kw)
    tame(flow, gain)
    randomize_constants(flow, D * 7 + K)
    flow = flow.to("cuda").eval()
    flow.precision = "fp32"
    return flow


def rows(name, B):
    return torch.randn(B, SHAPES[name][1], device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))


def time_call(flow, x):
    """ms per call: enough calls for >= ~0.2 s of GPU time after two warm-up calls."""
    for _ in range(2):
        flow.log_prob_and_grad(x)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    flow.log_prob_and_grad(x)
    b.record()
    b.synchronize()
    reps = max(5, min(500, int(200.0 / max(a.elapsed_time(b), 1e-3))))
    a.record()
    for _ in range(reps):
        flow.log_prob_and_grad(x)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


class Session:
    """One process's flows and rows, cached per shape / batch size."""

    def __init__(self):
        self.flows, self.x = {}, {}

    def time(self, name, B):
        if name not in self.flows:
            self.flows[name] = make_flow(name)
        if (name, B) not in self.x:
            self.x = {(name, B): rows(name, B)}          # one batch resident at a time
        flow = self.flows[name]
        ms = time_call(flow, self.x[(name, B)])
        return ms, flow.last_launches, flow.last_grad_precision

    def outputs(self, name, B):
        lp, g = self.flows[name].log_prob_and_grad(self.x[(name, B)])
        return lp.cpu(), g.cpu()


def worker():
    """The chain: reads 'name B path' lines, times, saves the outputs to path, answers with one JSON line."""
    s = Session()
    for line in sys.stdin:
        name, B, path = line.split()
        ms, n, prec = s.time(name, int(B))
        if path != "-":
            torch.save(s.outputs(name, int(B)), path)
        print(json.dumps({"ms": ms, "launches": n, "precision": prec}), flush=True)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3", "small_grad_bench.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    env = dict(os.environ, USF_SMALL_STACK="0")
    w = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker"], stdin=subprocess.PIPE,
                         stdout=subprocess.PIPE, text=True, env=env)
    s = Session()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi, "timing": "CUDA events, Flow.log_prob_and_grad at fp32",
           "rounds": ROUNDS, "results": []}
    tmp = tempfile.mkdtemp()
    try:
        for name in SHAPES:
            for B in BATCHES:
                new, old = [], []
                for r in range(ROUNDS):
                    ms, n_new, p_new = s.time(name, B)
                    new.append(ms)
                    path = os.path.join(tmp, "old.pt") if r == 0 else "-"
                    w.stdin.write(f"{name} {B} {path}\n")
                    w.stdin.flush()
                    reply = json.loads(w.stdout.readline())
                    old.append(reply["ms"])
                lp, g = s.outputs(name, B)
                lp_o, g_o = torch.load(os.path.join(tmp, "old.pt"))
                lp_d = float(((lp.double() - lp_o.double()).abs() / lp_o.double().abs().clamp_min(1.0)).max())
                scale = g_o.double().abs().amax(1).clamp_min(1e-30)
                g_row = (g.double() - g_o.double()).abs().amax(1) / scale
                r = {"shape": name, "B": B, "new_ms": min(new), "old_ms": min(old), "new_all_ms": new, "old_all_ms": old,
                     "speedup": min(old) / min(new), "new_launches": n_new, "old_launches": reply["launches"],
                     "precision": [p_new, reply["precision"]], "lp_max_rel_diff": lp_d,
                     "grad_row_rel_diff_max": float(g_row.max()), "grad_row_rel_diff_median": float(g_row.median()),
                     "grad_rows_over_1e-4": int((g_row > 1e-4).sum())}
                print(json.dumps(r), flush=True)
                res["results"].append(r)
    finally:
        w.stdin.close()
        w.wait()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    worker() if "--worker" in sys.argv else main()
