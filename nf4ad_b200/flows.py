"""`Flow`, `USFlow` (the `src.usflows.flows` names) and a `NonUSFlow` mirror on the B200 path.

`Flow.log_prob / sample / forward / backward` keep the surface nf4ad's wrappers use
(`/root/reference/src/nf4ad/adbench_wrapper.py:345,369,383,424`, `vaeflow.py:201,240`,
`flows.py:117-125`) and the semantics of `TransformedDistribution.log_prob / sample`
(torch `transformed_distribution.py:143-190`), but execute as:

  * inference (no autograd): ONE fused launch chain over a packed layer-descriptor array
    (`nf4ad_b200.stack` -> `usf_stack_run`) -- bf16 / bf16x2 / 3xTF32 tcgen05 GEMMs or fp32 FFMA kernels
    (`flow.precision`, resolved per weight version by `Flow._tier`), one whole-stack kernel for small event shapes;
  * training (autograd): the layer-wise kernels with their hand-written backward kernels (`nf4ad_b200.ops` autograd
    Functions); in the tensor-core tiers the affine runs between couplings are composed in weight space
    (`Flow._compose_affine_runs`) so the batch sees one GEMM per run.

CUDA tensors only -- a CPU tensor raises (`USFError`); the CPU restatement lives in `oracle/`.
"""
import contextlib
import os
from typing import Any, Dict, List, Optional, Type

import torch

from . import _lib, ops, stack
from .transforms import (
    BaseTransform, BlockAffineTransform, HouseholderTransform, InverseTransform, LUTransform, MaskedAffineCoupling,
    MaskedCoupling, ScaleTransform, SequentialAffineTransform, composing, context_dim, coupling_apply,
)

class _RunComposer:
    """Composes the affine runs of one training pass (`Flow._compose_affine_runs`), each chain forked from the step's
    start event.  `AHEAD` = how many runs are composed in advance of the one the batch-sized chain takes next.  Two
    orders follow the order in which this code runs on the host: a replayed CUDA graph dispatches its nodes roughly in
    capture order (~0.6 us per node; a step has ~1400), and autograd's backward pass visits nodes newest first -- so
    with a small `AHEAD` weight-space and batch-sized work alternate in both passes, with a large one (default: every
    run up front) all weight-space chains are dispatched first and visited last.  Measured on C2 / B = 4096
    (USF_COMPOSE_AHEAD = 1, 2, 3, all): 3.43 / 3.44 / 3.37 / 3.42 ms per step -- no difference: the step ends ~0.6 ms
    after the batch chain either way, which is the latency of ONE weight-space backward chain (~100 short kernels), not
    the order they are visited in.  Kept as a switch for other shapes."""

    AHEAD = int(os.environ.get("USF_COMPOSE_AHEAD", "99"))

    def __init__(self, flow, runs, probes, cur, start, pin):
        self.flow, self.runs, self.probes, self.cur, self.start, self.pin = flow, runs, probes, cur, start, pin
        self.done = []                       # per run, in order: the composed tuple or None

    def take(self, item):
        """The composed form of plan item `item` (None: not one of the composed runs), composing ahead first."""
        idx = next((i for i, r in enumerate(self.runs) if r is item), None)
        if idx is None:
            return None
        upto = min(len(self.runs), idx + 1 + max(0, self.AHEAD))
        while len(self.done) < upto:
            i = len(self.done)
            self.done.append(self.flow._compose_run(self.runs[i], i, self.probes, self.cur, self.start))
        return self.done[idx]


def _on_device(method):
    """Runs a `Flow` method with the CUDA device of its first tensor argument current: the C library launches on the
    current device's current stream (`_lib.stream`), so a flow living on cuda:1 must not be driven through cuda:0."""
    import functools

    @functools.wraps(method)
    def wrapped(self, x=None, *args, **kwargs):
        self.__dict__["_key_now"] = None          # the weights key is computed at most once per public call
        try:
            if isinstance(x, torch.Tensor) and x.is_cuda and x.device.index != torch.cuda.current_device():
                with torch.cuda.device(x.device):
                    return method(self, x, *args, **kwargs)
            return method(self, x, *args, **kwargs)
        finally:
            self.__dict__["_key_now"] = False
    return wrapped


_PRECISIONS = {"fp32": _lib.USF_PREC_FP32, "bf16": _lib.USF_PREC_BF16, "tf32x3": _lib.USF_PREC_TF32X3,
               "bf16x2": _lib.USF_PREC_BF16X2}
# `flow.precision`:
#   "auto"   (default) the <= 1e-4 tier on the fastest kernels that hold it: bf16x2 tensor-core kernels for D >= 128, fp32
#            FFMA kernels below (the one-kernel path for small event shapes)
#   "fp32"   fp32 FFMA kernels (the tightest: ~1e-6)
#   "tf32x3" 3xTF32 tcgen05 kernels (fp32 operands as hi + lo: <= 1e-4)
#   "bf16x2" bf16 tcgen05 kernels on (hi, lo) bf16 operand pairs, 3 MMAs per K step (<= 1e-4 at twice the 3xTF32 rate)
#   "bf16"   bf16 tcgen05 kernels, <= 1e-2 -- verified per weight version (Flow._tier)
_REQUESTS = ("auto",) + tuple(_PRECISIONS)


def _default_precision():
    p = os.environ.get("USF_PRECISION", "auto").lower()
    if p not in _REQUESTS:
        raise ValueError(f"USF_PRECISION must be one of {sorted(_REQUESTS)}, got {p!r}")
    return p


class Flow(torch.nn.Module):
    """Normalising flow = base distribution pushed through `layers` (generative order)."""

    export = "log_prob"

    def __init__(self, base_distribution, layers, soft_training: bool = False,
                 training_noise_prior=None, device="cpu", *args, **kwargs):
        preset = dict(self.__dict__)          # subclasses assign attributes first (flows.py:54-61)
        super().__init__()
        for k, v in preset.items():
            self.__dict__.setdefault(k, v)
        self.soft_training = soft_training
        self.training_noise_prior = training_noise_prior
        self.layers = list(layers)
        self.trainable_layers = torch.nn.ModuleList(
            [l for l in self.layers if isinstance(l, torch.nn.Module)])
        self.base_distribution = base_distribution
        self.device = device
        self.precision = _default_precision()   # "auto" (default) / "fp32" / "bf16x2" / "tf32x3" (<= 1e-4 tiers) or "bf16" (<= 1e-2, verified: _tier)
        self.effective_precision = self.precision
        self.bf16_calibration_err = None
        # run-to-run bit-identical log_prob (the reference's eager CPU path is deterministic): per-row partial sums go to
        # slots that are added in a fixed order instead of fp32 atomics (usf_set_deterministic).  Costs one small launch.
        self.deterministic = os.environ.get("USF_DETERMINISTIC", "0") == "1"
        # tensor-core training: compose the affine runs between couplings in weight space (`_compose_affine_runs`)
        self.compose_affine = os.environ.get("USF_COMPOSE_AFFINE", "1") != "0"
        self.last_launches = 0                  # kernels enqueued by the last fused call
        self.last_grad_precision = None         # tier of the last log_prob_and_grad: "bf16x2", "fp32" or "autograd"
        self._compiled = {}
        self._key_slots = None
        # the reference builds its flows with `device=...` and then scores device tensors without an explicit `.to()`
        # (`/root/reference/tests/conftest.py:123-125`, `tests/test_flows.py:57-60`): the constructor moves the parameters
        if str(device) != "cpu":
            self.to(device)

    # ------------------------------------------------------------------ helpers
    @property
    def event_shape(self):
        """Shape of one sample: `in_dims` of the stacked flows ([D], or image-shaped [C, H, W]); else read off the base
        distribution (USFlows wraps it as `Independent(base, len(batch_shape))`)."""
        if hasattr(self, "in_dims"):
            return tuple(int(d) for d in self.in_dims)
        base = self.base_distribution
        shp = tuple(getattr(base, "batch_shape", ())) + tuple(getattr(base, "event_shape", ()))
        return shp if shp else (int(self._infer_dim()),)

    @property
    def event_dim(self):
        n = 1
        for d in self.event_shape:
            n *= d
        return n

    def _infer_dim(self):
        for l in self.layers:
            if hasattr(l, "dim"):
                d = l.dim
                return d[0] if isinstance(d, (tuple, list)) else d
            if hasattr(l, "mask"):
                return l.mask.numel()
        raise ValueError("cannot infer the event dimension")

    def context_dim(self):
        """Width of the context the conditioners take (`ConditionalDenseNN.context_dim`); 0 = unconditional flow."""
        cd = self.__dict__.get("_ctx_dim")
        if cd is None:
            cd = 0
            for l in self.layers:
                cond = getattr(l, "conditioner", None)
                if cond is not None:
                    cd = max(cd, context_dim(cond))
            self.__dict__["_ctx_dim"] = cd
        return cd

    def _soft_context(self, x2, context):
        """USFlows soft training: the conditioners take the per-sample noise level as context, and scoring without one
        means noise level 0 (upstream behaviour as recalled; see oracle/shim/src/usflows/flows.py)."""
        if context is None and self.soft_training:
            return torch.zeros(x2.shape[0], 1, dtype=torch.float32, device=x2.device)
        if context is not None:
            context = torch.as_tensor(context, device=x2.device, dtype=torch.float32)
            if context.dim() == 0:
                context = context.reshape(1, 1)
            elif context.dim() == 1:
                context = context.reshape(-1, 1) if context.shape[0] == x2.shape[0] else context.reshape(1, -1)
        return context

    def _scan_key_slots(self):
        """(owner dict, name) of every parameter / buffer / base-distribution tensor.  Walking the module tree costs
        ~0.2 ms, comparable to a whole small-batch scoring call, so it is done once (and again whenever the module
        is moved, re-moded or `invalidate_cache()`d) and `_weights_key` only looks the slots up."""
        slots = []
        for m in self.modules():
            slots += [(m._parameters, k) for k, v in m._parameters.items() if v is not None]
            slots += [(m._buffers, k) for k, v in m._buffers.items() if v is not None]
        base, seen = self.base_distribution, set()
        while base is not None and id(base) not in seen and not isinstance(base, torch.nn.Module):
            seen.add(id(base))
            slots += [(base.__dict__, k) for k, v in base.__dict__.items() if isinstance(v, torch.Tensor)]
            base = getattr(base, "base_dist", None)
        self._key_slots = slots
        return slots

    def invalidate_cache(self):
        """Forget the packed weights and the parameter scan (call after replacing sub-modules of a built flow)."""
        self._compiled = {}
        self._key_slots = None
        self.__dict__.pop("_ctx_dim", None)
        self.__dict__.pop("_tier_cache", None)
        self.__dict__.pop("_small_cache", None)

    def _weights_key(self):
        memo = self.__dict__.get("_key_now", False)
        if memo:                         # inside one public call (log_prob / backward / latent_to_data): computed already
            return memo
        slots = self.__dict__.get("_key_slots") or self._scan_key_slots()
        key = [_lib.weights_epoch()]     # raw-pointer / graph-replayed optimizer steps (optim.FusedAdam, DataParallelTrainer)
        for d, k in slots:
            t = d.get(k)
            key.append((id(t), t._version if t is not None else -1))
        key = tuple(key)
        if memo is None:
            self.__dict__["_key_now"] = key
        return key

    def train(self, mode: bool = True):
        if mode != self.training:
            self._key_slots = None
        return super().train(mode)

    # ---- which tier a grad-free call really runs ---------------------------------------------------------------
    # `precision = "bf16"` promises log_prob within 1e-2 of the fp64 result (BASELINE.json north star).  bf16 operands
    # hold that on the large trained-flow-like stacks (D >= 128: 1e-3 .. 6e-3) but not on every stack: the small ADBench /
    # GMM shapes (D < 128) and ill-conditioned untrained stacks amplify the 2^-9 operand rounding past it (4e-2 at D = 6).
    # So the tier is not taken on trust:
    #   * small event shapes (D + context <= 64, widths <= 128) run the ONE-kernel fp32 path (csrc/usf_small.cu) whatever
    #     tier was asked for -- those shapes are launch-latency bound, it is both the fastest and the most accurate form;
    #   * other stacks with D < 128 run the 3xTF32 kernels (fp32-grade; the tensor-core rate does not matter there);
    #   * for the rest the first scoring call after every weight change scores its first rows (<= 256) at both tiers and
    #     keeps bf16 only if the two agree within `BF16_CALIBRATION_TOL` on every row.
    # `effective_precision` reports the outcome; USF_BF16_CALIBRATE=0 / `bf16_trust` run the bf16 kernels regardless.
    BF16_CALIBRATION_TOL = 5e-3
    BF16_MIN_DIM = 128
    SMALL_MAX_DIM = 64
    SMALL_MAX_ROWS = 8192       # (for stacks with layers wider than 32; see _small_ok)
    # the tensor-core tier that stands in for fp32 ("auto", and where bf16 is not trusted): bf16 (hi, lo) operand pairs.
    # Measured on every BASELINE shape with D >= 128 (scripts/bf16x2_check.py, profiles/r2/bf16x2.txt): log_prob max-row
    # error 5e-6 .. 2.8e-5 (3xTF32: 5e-6 .. 5.6e-5) at 2.0-2.5x the 3xTF32 rate (C2: 3.39 vs 6.66 ms per 65536 rows).
    FP32_GRADE_TC = "bf16x2"

    SMALL_ALWAYS = False        # (measurement switch: take the one-kernel path whenever the stack is eligible)

    def _small_ok(self, device, rows=None):
        """Does the one-kernel path take this stack (both directions share the shapes), and does it pay at this batch
        size?  Measured against the split-operand tensor-core chain (scripts/bench_small.py, profiles/r2/small_stack.txt):
        one kernel instead of 11 launches wins at every batch size while the layers are at most 32 wide (D = 6: 1.6-1.8x,
        D = 20: 1.5x from 65536 rows on).  With 64-128 wide layers its fp32 FFMA arithmetic (paced by shared-memory reads)
        loses to the tensor cores beyond 8192 rows (0.4-0.6x at 65536 rows), so there it is kept for batches of up to
        8192 rows, where it is 1.03-1.17x and one launch means the lowest latency and a deterministic sum."""
        if self.event_dim + self.context_dim() > self.SMALL_MAX_DIM or len(self.event_shape) != 1:
            return False
        key = self._weights_key()
        hit = self.__dict__.get("_small_cache")
        if hit is None or hit[0] != key:
            cs = self._stack(True, device, "fp32")
            if cs is None or not cs.single_kernel:
                hit = (key, False, 0)
            else:
                widest = 0
                for j in range(cs.desc.n_blocks):
                    blk = cs.blocks[j]
                    widest = max([widest, blk.G.N] + [blk.mlp[l].N for l in range(blk.n_mlp - 1)])
                hit = (key, True, widest)
            self.__dict__["_small_cache"] = hit
        _, eligible, widest = hit
        if not eligible:
            return False
        return rows is None or self.SMALL_ALWAYS or rows <= self.SMALL_MAX_ROWS or widest <= 32

    def _tier(self, x2=None, context_rows=None):
        want = self.precision
        if want == "auto":
            want = self.FP32_GRADE_TC if self.event_dim >= self.BF16_MIN_DIM else "fp32"
        if want == "fp32" or (want == "bf16" and self.__dict__.get("bf16_trust", False)) or \
                (want == "bf16" and os.environ.get("USF_BF16_CALIBRATE", "1") == "0"):
            self.effective_precision = want
            return want
        key = self._weights_key()
        device = x2.device if x2 is not None else next(self.parameters()).device
        if self._small_ok(device, None if x2 is None else x2.shape[0]):     # (depends on the batch size: not cached below)
            self.effective_precision = "fp32"
            return "fp32"
        hit = self.__dict__.get("_tier_cache")
        if hit is not None and hit[0] == (key, want) and (hit[2] or x2 is None):
            self.effective_precision = hit[1]
            return hit[1]
        tier, calibrated, err = want, False, None
        if want in ("tf32x3", "bf16x2"):
            calibrated = True
        elif self.event_dim < self.BF16_MIN_DIM:
            tier, calibrated = self.FP32_GRADE_TC, True
        elif x2 is not None and x2.shape[0] > 0 and not self._needs_grad(x2):
            rows = (x2 if context_rows is None else context_rows)[:256]
            lo = self._stack(True, device, "bf16")
            hi = self._stack(True, device, self.FP32_GRADE_TC) or self._stack(True, device, "fp32")
            if lo is None or lo.desc.base_kind < 0 or hi is None:
                calibrated = True                      # no fused bf16 path at all / nothing to compare with
            else:
                a = lo.run(rows, want_logprob=True)[0].double()
                b = hi.run(rows.float(), want_logprob=True)[0].double()
                err = float(((a - b).abs() / b.abs().clamp_min(1.0)).nan_to_num(nan=float("inf")).max())
                if not err <= self.BF16_CALIBRATION_TOL:
                    tier = self.FP32_GRADE_TC if hi.precision != _lib.USF_PREC_FP32 else "fp32"
                calibrated = True
                # the packed weights of the tier that lost are not needed until the weights change again
                self._compiled.pop((True, lo.precision if tier != "bf16" else hi.precision), None)
        if tier in ("tf32x3", "bf16x2") and self._stack(True, device, tier) is None and \
                self._stack(True, device, "fp32") is not None:
            tier = "fp32"                              # shapes the split-operand kernels do not take (N > 1024)
        self.__dict__["_tier_cache"] = ((key, want), tier, calibrated, err)
        self.effective_precision = tier
        self.bf16_calibration_err = err
        return tier

    def cached_precision(self):
        """The resolved tier of the current weights, or None when it has not been calibrated since they changed."""
        if self.precision == "fp32":
            return "fp32"
        hit = self.__dict__.get("_tier_cache")
        return hit[1] if hit is not None and hit[2] and hit[0][0] == self._weights_key() else None

    def resolve_precision(self, x):
        """The tier grad-free calls on these weights run at ("bf16" may resolve to "tf32x3" / "fp32", see above);
        `x`: a few device rows to calibrate on when that has not happened since the last weight change."""
        x2, _ = self._prep(x)
        ctx = self._soft_context(x2, None)
        if self.context_dim() > 0 and ctx is not None:
            xin = torch.cat([x2.float(), ctx.expand(x2.shape[0], self.context_dim())], dim=1)
        else:
            xin = None
        return self._tier(x2, xin)

    def _stack(self, inverse, device, precision=None, grad=False):
        """Compiled (packed) stack for this direction / precision / weight version, or None.  `grad`: the inverse stack
        with the transposed matrices of the reverse chain as well (`log_prob_and_grad`)."""
        precision = precision or self.precision
        if precision == "auto":
            precision = self.FP32_GRADE_TC if self.event_dim >= self.BF16_MIN_DIM else "fp32"
        prec = _PRECISIONS[precision]
        slot = ("grad", prec) if grad else (bool(inverse), prec)
        key = (self._weights_key(), str(device))
        hit = self._compiled.get(slot)
        if hit is not None and hit[0] == key:
            return hit[1]
        try:
            if len(self.event_shape) != 1:
                raise stack.Unsupported("image-shaped event: the layer-wise kernels are used")
            cs = stack.CompiledStack(self.layers, self.base_distribution, self.event_dim, device, inverse, prec, grad=grad)
        except stack.Unsupported as e:
            cs = None
            self._unsupported_reason = str(e)
        self._compiled[slot] = (key, cs)
        return cs

    def _needs_grad(self, x):
        if not torch.is_grad_enabled():
            return False
        return x.requires_grad or any(p.requires_grad for p in self.parameters())

    def _prep(self, x):
        """(*batch, *event) -> (rows (B, prod(event)), leading batch shape)."""
        _lib.require_cuda(x)
        ev = self.event_shape
        n = len(ev)
        if x.dim() < n or (n > 1 and tuple(x.shape[x.dim() - n:]) != ev):
            raise ValueError(f"input of shape {tuple(x.shape)} does not end in the event shape {ev}")
        lead = tuple(x.shape[:x.dim() - n])
        width = 1
        for d in x.shape[x.dim() - n:]:
            width *= int(d)
        return x.reshape(-1, width), lead

    def _unflat(self, rows):
        """(B, prod(event)) rows -> (B, *event) as the layers of an image-shaped flow expect."""
        ev = self.event_shape
        return rows if len(ev) == 1 else rows.reshape(rows.shape[0], *ev)

    def _fused(self, x2, context, inverse):
        """-> (compiled stack | None, input rows incl. context columns).  The fused launch chain serves the grad-free
        calls of flat-event flows; a conditional flow carries its context as extra activation columns."""
        if self._needs_grad(x2):
            return None, x2
        cd = self.context_dim()
        if cd == 0 and context is not None:
            return None, x2                   # unconditional conditioners handed a context: evaluated as given, layer-wise
        if cd > 0 and context is None:
            raise ValueError("this flow's conditioners take a context (ConditionalDenseNN): pass `context=` or build the "
                             "flow with soft_training=True")
        xin = x2
        if cd > 0:
            ctx = context if context.dim() == 2 else context.reshape(-1, cd)
            xin = torch.cat([x2.to(torch.float32), ctx.to(torch.float32).expand(x2.shape[0], cd)], dim=1)
        tier = self._tier(x2 if inverse else None, xin if inverse else None)
        cs = self._stack(inverse, x2.device, tier)
        if cs is None or cs.ctx_dim != cd:
            return None, x2
        return cs, xin

    # ------------------------------------------------------------------ density path
    @_on_device
    def log_prob(self, x, context=None):
        x2, lead = self._prep(x)
        context = self._soft_context(x2, context)
        cs, xin = self._fused(x2, context, True)
        if cs is not None and cs.desc.base_kind >= 0:
            lp, _, _, n = cs.run(xin, want_logprob=True, deterministic=self.deterministic)
            self.last_launches = n
            return lp.reshape(lead)
        # autograd (training) pass; "bf16" / "tf32x3" select the tensor-core forms of its GEMMs (ops.tc_training);
        # "auto" trains on the fp32 kernels (the reference's arithmetic)
        mode = {"bf16": 1, "tf32x3": 2}.get(self.precision, 0) if torch.is_grad_enabled() else 0
        with ops.tc_training(mode):
            z, neg_ladj = self._inverse_layers(self._unflat(x2), context)
            lp = self._base_log_prob(z.reshape(z.shape[0], -1)) + neg_ladj
        return lp.reshape(lead)

    @_on_device
    def log_prob_and_grad(self, x, context=None):
        """(log p(x), d log p(x) / dx) per row, the weights taken as constants: `lp` has the leading batch shape, `g` the
        shape of `x` (fp32).  Equal to `torch.autograd.grad(self.log_prob(x).sum(), x)` in exact arithmetic (relu'(0) = 0,
        sign(0) = 0 for a Laplace base); builds no autograd graph, touches no `p.grad`, works under `torch.no_grad()`.
        The gradient is the per-feature attribution of the anomaly score -log p (the context gradient is not formed).

        Flat-event stacks run the reverse launch chain of the fused path in one library call: at bf16x2 when the request
        is "auto" with D >= BF16_MIN_DIM, or "bf16x2" / "bf16" / "tf32x3" (a gradient at bf16 operand precision would be
        of little use), else on the fp32 SIMT kernels.  Other flows (image-shaped events, opaque conditioners, softplus
        scales, a context handed to an unconditional flow) differentiate the layer-wise pass with autograd.
        `last_grad_precision` reports which: "bf16x2", "fp32" or "autograd"."""
        x2, lead = self._prep(x)
        ctx = self._soft_context(x2, context)
        cs, xin = self._grad_stack(x2, ctx)
        if cs is None:
            self.last_grad_precision = "autograd"
            with torch.enable_grad():
                xr = x.detach().to(torch.float32).requires_grad_(True)
                lp = self.log_prob(xr, context)
                g, = torch.autograd.grad(lp.sum(), xr)
            return lp.detach(), g
        lp, g, n = cs.run_grad(xin, deterministic=self.deterministic)
        self.last_grad_precision = "bf16x2" if cs.precision == _lib.USF_PREC_BF16X2 else "fp32"
        self.last_launches = n
        return lp.reshape(lead), g.reshape(x.shape)

    def _grad_stack(self, x2, context):
        """-> (compiled stack with its transposed matrices | None, input rows incl. context columns) for
        `log_prob_and_grad`, by the tier rule there."""
        cd = self.context_dim()
        if len(self.event_shape) != 1 or (cd == 0 and context is not None):
            return None, x2
        if cd > 0 and context is None:
            raise ValueError("this flow's conditioners take a context (ConditionalDenseNN): pass `context=` or build the "
                             "flow with soft_training=True")
        xin = x2.to(torch.float32)
        if cd > 0:
            ctx = context if context.dim() == 2 else context.reshape(-1, cd)
            xin = torch.cat([xin, ctx.to(torch.float32).expand(x2.shape[0], cd)], dim=1)
        want = self.precision
        tc = (want == "auto" and self.event_dim >= self.BF16_MIN_DIM) or want in ("bf16x2", "bf16", "tf32x3")
        for tier in (("bf16x2", "fp32") if tc else ("fp32",)):
            cs = self._stack(True, x2.device, tier, grad=True)
            if cs is not None and cs.ctx_dim == cd and cs.desc.base_kind >= 0:
                return cs, xin
        return None, x2

    def _prefetch_lu_inverses(self, y):
        """Mixed-precision training: the dense inverses of all LU layers this pass will apply are independent of the
        data and of each other, and one inversion (two 25-CTA triangular solves on the identity) cannot fill the GPU.
        They are therefore issued up front on a few side streams (fork / join from the current stream; their backward
        nodes run on the same streams), and `LUTransform.backward` picks its matrix up from `_A_pre`."""
        B = y.shape[0]
        mods, seen = [], set()
        for layer in self.layers:
            if not isinstance(layer, torch.nn.Module):
                continue
            for m in layer.modules():
                if isinstance(m, LUTransform):
                    m.__dict__.pop("_A_pre", None)          # never carry a matrix over from an interrupted pass
                    # a layer wrapped in InverseTransform is applied through its forward map: no inverse needed
                    if not isinstance(layer, InverseTransform) and id(m) not in seen and m.dim % 16 == 0:
                        seen.add(id(m))
                        mods.append(m)
        if not y.is_cuda or B < 8 or B % 8 or len(mods) < 2:
            return
        cur = torch.cuda.current_stream(y.device)
        used = self._side(y.device, len(mods))
        for s in used:
            s.wait_stream(cur)
        # in the order the pass will need them (it walks the layers backwards); each consumer joins only its own stream
        for i, lu in enumerate(reversed(mods)):
            st = used[i % len(used)]
            with torch.cuda.stream(st):
                A = ops.LUInverseFn.apply(lu.L_raw, lu.U_raw)
            A.record_stream(cur)
            lu.__dict__["_A_pre"] = (A, st)

    _PROBES = {}                 # (device, D) -> (I_D, 8 zero rows): what an affine run is composed on

    def _side(self, device, n):
        """`n` (at most 32) side streams of this flow for the weight-space chains.  Every stream the flow creates is
        also listed in `_side_streams`, which a trainer joins; the lists only ever hold streams a pass has forked into,
        so joining "all of the flow's side streams" never waits on one outside a capture."""
        n = max(1, min(32, n))
        streams = self.__dict__.get("_run_streams")
        if streams is None or (streams and streams[0].device != device):
            streams = self.__dict__["_run_streams"] = []
            self.__dict__["_side_streams"] = []
            for k in ("_cond_stream", "_acc_stream"):
                self.__dict__.pop(k, None)
            # the factor gradients are produced on the side streams on purpose; autograd syncs them with the
            # accumulation stream, it only warns that this costs a synchronisation
            warn_off = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
            if warn_off is not None:
                warn_off(False)
        while len(streams) < n:
            # two streams per affine run, in the order the batch-sized chain consumes the runs: the earlier a run is
            # needed, the more urgent its stream (the chain itself runs above all of them: DataParallelTrainer)
            st = _lib.pooled_stream(device, ("run", len(streams)), priority=min(0, -4 + len(streams) // 2))
            streams.append(st)
            self.__dict__["_side_streams"].append(st)
        return streams[:n]

    def _extra_stream(self, key, device, priority):
        """A further stream of the flow's own (conditioner operands, gradient accumulation), created once per device."""
        self._side(device, 1)                                        # (resets everything on a device change)
        st = self.__dict__.get(key)
        if st is None:
            st = self.__dict__[key] = _lib.pooled_stream(device, key, priority=priority)
            self.__dict__["_side_streams"].append(st)
        return st

    def _compose_affine_runs(self, y):
        """Mixed-precision training: every maximal run of affine layers between two couplings (LU solve / product,
        Householder reflections, scale -- with affine conjugation the tail of one block and the head of the next) is a
        single map x -> x M^T + c that does not depend on the data.  Each run is evaluated ONCE per step in weight space:
        its layers are applied, with autograd, to probe rows on a side stream (M^T = the identity through the linear parts,
        c = the image of 0, the parameter-only log-dets summed there too), and the batch then sees ONE tensor-core GEMM per
        run instead of a GEMM / reflection / scale kernel per layer.  The runs are independent of each other, so their
        chains -- forward here, backward wherever autograd reaches them: a node's backward runs on its forward's
        stream -- overlap each other and the batch-sized chain.  -> (plan, composer | None): the runs are composed by
        `_RunComposer.take`, a few ahead of the batch-sized chain."""
        plan, run = [], []
        for layer in reversed(self.layers):
            if isinstance(layer, BaseTransform) and getattr(layer, "is_affine", False) and not stack._is_coupling(layer):
                run.append(layer)
                continue
            if run:
                plan.append(run)
                run = []
            plan.append(layer)
        if run:
            plan.append(run)
        B, D = y.shape[0], y.shape[-1]
        if not (y.is_cuda and y.dim() == 2 and B >= 8 and B % 8 == 0 and D % 16 == 0 and getattr(self, "compose_affine", True)):
            return plan, None
        runs = [r for r in plan if isinstance(r, list)
                and any(isinstance(m, LUTransform) for layer in r for m in layer.modules())]
        if not runs:
            return plan, None
        dev = y.device
        probes = Flow._PROBES.get((dev, D))
        if probes is None:
            probes = Flow._PROBES[(dev, D)] = (torch.eye(D, device=dev, dtype=torch.float32),
                                               torch.zeros(8, D, device=dev, dtype=torch.float32))
        cur = torch.cuda.current_stream(dev)
        # A parameter's gradient accumulator runs on the stream that is current when the parameter first enters a graph,
        # and autograd sums the contributions of different nodes there.  Every affine layer sits in TWO runs (tail of
        # one, head of the next): were the accumulator created inside a run, the partial sums of the neighbouring
        # run's gradients would be queued on this run's stream ahead of its own backward chain -- and the nine chains
        # would execute one after the other (measured: a 2.1 ms tail).  So the accumulators are created here, on a stream
        # of their own -- not the calling one either: with the runs composed a few ahead, their backward chains are
        # visited BETWEEN the blocks of the batch-sized chain, and an accumulation queued on the batch chain's stream
        # would hold it up until that weight-space chain has finished.  The graphs built later keep the accumulators
        # alive (`pin` lives as long as the composer).
        start = torch.cuda.Event()
        start.record(cur)
        acc = self._extra_stream("_acc_stream", dev, -8)
        acc.wait_event(start)
        with torch.cuda.stream(acc):
            pin = [p.view_as(p) for r in runs for layer in r for p in layer.parameters() if p.requires_grad]
        return plan, _RunComposer(self, runs, probes, cur, start, pin)

    def _compose_run(self, r, i, probes, cur, start):
        """One affine run -> (M^T, c, log-det, streams, bf16 operands of M | None) or None, on the run's own two streams, forked from `start`."""
        dev = probes[0].device
        used = self._side(dev, 2 * (i + 1))
        st, st_c = used[2 * i], used[2 * i + 1]     # the matrix pass / the shift pass (waits for the factors of the first)
        st.wait_event(start)
        st_c.wait_event(start)
        with composing() as comp:
            comp["eye"], comp["aux"] = probes[0], st_c
            # the matrix: the identity through the run's linear parts (shifts off -- taking them from the same rows
            # and subtracting would make every shift gradient a difference of D bf16-rounded sums) ...
            with torch.cuda.stream(st):
                comp["linear_only"] = True
                Mt = probes[0]
                for layer in r:
                    Mt = layer.backward(Mt)
            # ... and the shift: the zero row through the full maps (8 rows: the GEMM's row granularity).
            # (Issuing this pass first would put the LU factor nodes and their long backward on its stream, beside
            # the matrix pass's backward chain -- measured: the tail shrinks by 90 us, but the replayed graph then
            # starts the nine inversions three at a time instead of together: +500 us before the first coupling.)
            with torch.cuda.stream(st_c):
                comp["linear_only"] = False
                # the parameter-only log-dets first: created before the shift chain, their backward nodes are visited
                # after it, so the ~15 tiny kernels of their gradients do not sit between the chain's backward and the
                # factor gradients that wait for it (an affine layer's log-det does not look at its arguments)
                z, const = probes[1], None
                for layer in r:
                    l = layer.log_abs_det_jacobian(z, z)
                    if torch.is_tensor(l) and l.dim() > 0:
                        const = False                  # a data-dependent log-det: not an affine run after all
                        break
                    l = torch.as_tensor(l, device=dev, dtype=torch.float32)
                    const = l if const is None else const + l
                if const is not False:
                    for layer in r:
                        z = layer.backward(z)
                c = None if const is False else z[0]
        if const is False:
            cur.wait_stream(st)
            cur.wait_stream(st_c)
            return None
        operands = None
        if ops._TC_TRAIN == 1:
            # the bf16 operand forms of the composed matrix, on the run's stream rather than in front of the batch's GEMM
            with torch.cuda.stream(st):
                operands = ops.weight_operands(Mt.detach(), w_transposed=True)
            for t in operands:
                t.record_stream(cur)
        for t in (Mt, c, const):
            t.record_stream(cur)
        return Mt, c, const, (st, st_c), operands

    def _prefetch_conditioners(self, y):
        """Tensor-core training: the bf16 operand forms of the conditioner weights (first layer with the coupling mask
        folded in) do not depend on the batch: converted up front on one side stream instead of in front of every GEMM
        of the batch-sized chain.  Single use: `run_conditioner` pops `_usf_pre`."""
        from .transforms import conditioner_weights
        if ops._TC_TRAIN != 1 or not y.is_cuda or y.dim() != 2 or y.shape[0] < 8 or y.shape[0] % 8:
            return
        todo = []
        for layer in self.layers:
            cond = getattr(layer, "conditioner", None)
            if stack._is_coupling(layer) and isinstance(cond, torch.nn.Module):
                cond.__dict__.pop("_usf_pre", None)
                if layer.mask.numel() == y.shape[1] and all(p.is_cuda for p in cond.parameters()):
                    todo.append((layer, cond))
        if not todo:
            return
        cur = torch.cuda.current_stream(y.device)
        st = self._extra_stream("_cond_stream", y.device, -8)       # short and needed first
        st.wait_stream(cur)
        with torch.cuda.stream(st):
            for layer, cond in todo:
                ws = conditioner_weights(cond, layer.mask)
                if ws is None or any(W.shape[0] % 16 or W.shape[1] % 16 for W, _ in ws):
                    continue
                pre = []
                for W, b in ws:
                    Wb, WT = ops.weight_operands(W)
                    for t in (W, Wb, WT):
                        t.record_stream(cur)
                    pre.append((W, b, (Wb, WT)))
                cond.__dict__["_usf_pre"] = (pre, st)
        self.__dict__["_cond_pending"] = st

    def _inverse_layers(self, y, context=None):
        """Layer-wise data -> latent with the accumulated -sum(ladj) (autograd-capable)."""
        # (fp32 training -- the reference's arithmetic -- stays layer-wise: composed, its C2 step takes 14.2 instead of
        # 23.2 ms, but the reflection vectors' gradients, differences of large terms of dM, end up 4.6e-3 from the fp64
        # oracle's instead of 7e-5; the tensor-core tiers are at that level in either form)
        if ops.tc_train_enabled() and y.dim() == 2:
            plan, composer = self._compose_affine_runs(y)
            self._prefetch_conditioners(y)
        else:
            plan, composer = list(reversed(self.layers)), None
        if ops.tc_train_enabled() and composer is None:
            self._prefetch_lu_inverses(y)
        total = torch.zeros(y.shape[0], device=y.device, dtype=torch.float32)
        consts = []
        for item in plan:
            hit = composer.take(item) if (composer is not None and isinstance(item, list)) else None
            if hit is not None:
                Mt, c, const, sts, operands = hit
                for st in sts:
                    torch.cuda.current_stream(y.device).wait_stream(st)
                y = ops.linear_fn(y, Mt, c, False, w_transposed=True, operands=operands)
                consts.append(const)
                continue
            for layer in (item if isinstance(item, list) else (item,)):
                if hasattr(layer, "inverse_and_ladj"):
                    x, ladj = layer.inverse_and_ladj(y, context)
                elif stack._is_coupling(layer):
                    # a foreign coupling class (the reference's own MaskedAffineCoupling): same arithmetic, our kernels
                    x, ladj = coupling_apply(layer, y, True, context)
                else:
                    x = layer.backward(y) if context is None else layer.backward(y, context)
                    ladj = layer.log_abs_det_jacobian(x, y)
                total = total - ladj
                y = x
        if consts:
            total = total - torch.stack(consts).sum()
        pending = self.__dict__.pop("_cond_pending", None)
        if pending is not None:              # (joined even if no conditioner picked its operands up)
            torch.cuda.current_stream(y.device).wait_stream(pending)
        if composer is not None:
            # the accumulation stream was forked into this pass (it carries no forward work): join it, so that a
            # forward-only call inside someone's stream capture leaves no unjoined stream behind
            torch.cuda.current_stream(y.device).wait_stream(self.__dict__["_acc_stream"])
        return y, total

    def _forward_layers(self, z, context=None):
        for layer in self.layers:
            if stack._is_coupling(layer) and not hasattr(layer, "forward_and_ladj"):
                z = coupling_apply(layer, z, False, context)[0]        # foreign coupling class
            else:
                z = layer.forward(z) if context is None else layer.forward(z, context)
        return z

    def _base_log_prob(self, z):
        base = self.base_distribution
        bp = stack.base_params(base, z.shape[1], z.device)
        if bp is not None:
            kind, _, _ = bp
            inner = base
            while isinstance(inner, torch.distributions.Independent):
                inner = inner.base_dist
            loc = torch.as_tensor(inner.loc, device=z.device)
            scale = torch.as_tensor(inner.scale, device=z.device)
            return ops.BaseLogProbFn.apply(z, loc.expand(z.shape[1]) if loc.numel() == 1 else loc, scale, kind)
        lp = base.log_prob(z)                      # unsupported base: evaluated as given
        while lp.dim() > 1:
            lp = lp.sum(-1)
        return lp

    @_on_device
    def backward(self, x, context=None):
        """data -> latent."""
        x2, lead = self._prep(x)
        context = self._soft_context(x2, context)
        cs, xin = self._fused(x2, context, True)
        if cs is not None:
            _, z, _, n = cs.run(xin, want_y=True)
            self.last_launches = n
        else:
            z, _ = self._inverse_layers(self._unflat(x2), context)
        return z.reshape(*lead, *self._tail(x, z))

    @_on_device
    def latent_to_data(self, z, context=None):
        z2, lead = self._prep(z)
        context = self._soft_context(z2, context)
        cs, zin = self._fused(z2, context, False)
        if cs is not None:
            _, x, _, n = cs.run(zin, want_y=True)
            self.last_launches = n
        else:
            x = self._forward_layers(self._unflat(z2), context)
        return x.reshape(*lead, *self._tail(z, x))

    def _tail(self, given, result):
        """Event dims of the result: the event shape (image-shaped flows), else the caller's own last dimension."""
        ev = self.event_shape
        return ev if len(ev) > 1 else (result.shape[-1],)

    def sample(self, sample_shape=None, context=None):
        shape = torch.Size() if sample_shape is None else torch.Size(sample_shape)
        with torch.no_grad():
            z = self.base_distribution.sample(shape)
            return self.latent_to_data(z, context)

    def rsample(self, sample_shape=None, context=None):
        shape = torch.Size() if sample_shape is None else torch.Size(sample_shape)
        return self.latent_to_data(self.base_distribution.rsample(shape), context)

    def forward(self, x=None, context=None):
        """`export` switch (`visualization.py:85-86`)."""
        if self.export == "log_prob":
            return self.log_prob(x, context)
        if self.export == "sample":
            return self.sample()
        if self.export == "backward":
            return self.backward(x, context)
        return self.latent_to_data(x, context)

    # ------------------------------------------------------------------ housekeeping
    def is_feasible(self) -> bool:
        return all(bool(l.is_feasible()) for l in self.layers if hasattr(l, "is_feasible"))

    def add_jitter(self, jitter: float = 1e-6) -> None:
        for l in self.layers:
            if hasattr(l, "jitter"):
                l.jitter(jitter)

    def log_prior(self):
        total = 0.0
        for l in self.layers:
            if hasattr(l, "log_prior"):
                total = total + l.log_prior()
        return total

    def _apply(self, fn, *a, **kw):
        out = super()._apply(fn, *a, **kw)
        for base in (self.base_distribution, self.training_noise_prior):      # plain distributions: move their tensors
            if base is None or isinstance(base, torch.nn.Module):
                continue
            seen = set()
            while base is not None and id(base) not in seen:
                seen.add(id(base))
                for k, v in list(base.__dict__.items()):
                    if isinstance(v, torch.Tensor):
                        base.__dict__[k] = fn(v)
                base = getattr(base, "base_dist", None)
        self._compiled = {}
        self._key_slots = None
        return out

    def to(self, *args, **kwargs):
        out = super().to(*args, **kwargs)
        if args and isinstance(args[0], (str, torch.device)):
            self.device = args[0]
        elif "device" in kwargs:
            self.device = kwargs["device"]
        return out

    def soft_noise(self, batch, generator=None):
        """USFlows soft training (SoftFlow-style; upstream behaviour as recalled, fixed by the oracle shim): one noise level
        per sample from `training_noise_prior`, the sample is perturbed by N(0, level^2) noise and the level is handed to
        the conditioners as context.  -> (noisy batch, context (B, 1))."""
        B = batch.shape[0]
        level = self.training_noise_prior.sample([B]).reshape(B).to(batch)
        eps = torch.randn(batch.shape, dtype=batch.dtype, device=batch.device, generator=generator)
        return batch + level.reshape(B, *([1] * (batch.dim() - 1))) * eps, level.reshape(B, 1).detach()

    def fit(self, data_train, optim=torch.optim.Adam, optim_params=None, batch_size=32, shuffle=True,
            gradient_clip=None, device=None, jitter=1e-6, epochs=1):
        """Feasibility check + jitter, then minimise -mean log_prob (- log_prior / N): USFlows `Flow.fit` as nf4ad's runner
        calls it (`explib/hyperopt.py:71-77`).  Returns the per-epoch mean loss.

        The data set is gathered once and kept on the device; batches are drawn there, the step -- (soft-training noise,)
        forward, hand-written backward kernels, clipping, optimizer update -- runs through `DataParallelTrainer` (one
        CUDA-graph replay per step for Adam / AdamW / SophiaG, which run as fused capturable kernels), and the host reads
        the loss once per epoch.  The feasibility check (a host read of the LU diagonals) runs at the start of every epoch
        instead of every step.  Under `torch.distributed` every rank trains on its shard of the same global batches."""
        from .parallel import DataParallelTrainer, rank_batches, shared_permutation
        if device is not None:
            self.to(device)
        dev = next(self.parameters()).device
        if isinstance(data_train, torch.Tensor):
            X = data_train
        elif isinstance(data_train, torch.utils.data.TensorDataset):
            X = data_train.tensors[0]
        elif hasattr(data_train, "__array__"):
            X = torch.as_tensor(data_train.__array__())
        else:                                        # a map-style dataset of rows or (row, label, ...) tuples
            rows = [data_train[j] for j in range(len(data_train))]
            X = torch.stack([torch.as_tensor(r[0] if isinstance(r, (tuple, list)) else r) for r in rows])
        X = X.to(device=dev, dtype=torch.float32)
        n = X.shape[0]
        params = dict(optim_params or {})
        from .optim import FusedAdam, SophiaG
        if dev.type == "cuda" and optim in (torch.optim.Adam, torch.optim.AdamW) and \
                set(params) <= {"lr", "betas", "eps", "weight_decay"}:
            # the same update through usf_adam_step (AdamW: decoupled decay, default 1e-2)
            if optim is torch.optim.AdamW:
                params.setdefault("weight_decay", 1e-2)
            opt = FusedAdam(self.parameters(), decoupled=optim is torch.optim.AdamW, **params)
        else:
            if dev.type == "cuda" and optim in (torch.optim.Adam, torch.optim.AdamW):
                params.setdefault("capturable", True)
                params.setdefault("fused", True)
            opt = optim(self.parameters(), **params)
        with_prior = getattr(self, "prior_scale", None) is not None
        soft = bool(self.soft_training) and self.training_noise_prior is not None

        def loss_fn(batch):
            ctx = None
            if soft:
                batch, ctx = self.soft_noise(batch)          # device RNG: capturable (the graph advances the generator)
            loss = -self.log_prob(batch, ctx).mean()
            if with_prior:
                loss = loss - self.log_prior() / n
            if isinstance(opt, SophiaG):
                opt.note_batch(batch.shape[0])
            return loss

        guard = torch.cuda.device(dev) if dev.type == "cuda" else contextlib.nullcontext()
        with guard:
            trainer = DataParallelTrainer(self, opt, gradient_clip=gradient_clip, loss_fn=loss_fn)
            trainer.broadcast_parameters()
            gen = torch.Generator(device=dev)
            gen.manual_seed(int(torch.initial_seed()) & 0x7FFFFFFF)
            losses = []
            for _ in range(epochs):
                while not self.is_feasible():
                    self.add_jitter(jitter)
                perm = shared_permutation(n, dev, gen, shuffle, trainer.group)
                total = torch.zeros((), device=dev)
                seen = 0
                for idx in rank_batches(perm, batch_size, trainer.rank, trainer.world):
                    batch = X.index_select(0, idx)
                    total += trainer.step(batch) * batch.shape[0]
                    seen += batch.shape[0]
                losses.append(float(total.cpu()) / max(seen, 1))         # one device -> host read per epoch
        self.fit_graph_replays = trainer.graph_replays
        return losses


def _parity_mask(in_dims, channel_only=False, invert=False):
    """`create_checkerboard_mask` / `create_channel_mask` (`nf4ad/flows.py:127-145`)."""
    grids = torch.meshgrid(*[torch.arange(d, dtype=torch.int32) for d in in_dims], indexing="ij")
    idx = torch.stack(grids)
    m = torch.fmod(idx[0] if channel_only else idx.sum(dim=0), 2).to(torch.float32).view(1, *in_dims)
    return 1 - m if invert else m


class _StackedFlow(Flow):
    """Shared builder of USFlow / NonUSFlow: per block
    `BlockAffine(Sequential(LU x lu, Householder))`, coupling, `Inverse(block)` if conjugated,
    alternating masks; tail `BlockAffine(LU)`, `Scale`  (`nf4ad/flows.py:78-114`)."""

    MASKTYPE = ("checkerboard", "channel")
    _coupling_cls = None

    def __init__(self, base_distribution, in_dims: List[int], coupling_blocks: int,
                 conditioner_cls: Type[torch.nn.Module], conditioner_args: Dict[str, Any],
                 soft_training: bool = False, prior_scale: Optional[float] = None,
                 training_noise_prior=None, affine_conjugation: bool = False, nonlinearity=None,
                 lu_transform: int = 1, householder: int = 1, masktype: str = "checkerboard",
                 device="cpu", *args, **kwargs):
        self.coupling_blocks, self.in_dims = coupling_blocks, list(in_dims)
        self.conditioner_cls, self.conditioner_args = conditioner_cls, conditioner_args
        self.prior_scale = prior_scale
        if masktype not in self.MASKTYPE:
            raise ValueError(f"Unknown mask type {masktype}")
        if lu_transform < 0:
            raise ValueError("Number of LU transforms must be non-negative")
        if householder < 0:
            raise ValueError("Number of Householder vectors transforms must be non-negative")
        self.lu_transform, self.householder = lu_transform, householder
        D = in_dims[0]          # the affine layers act along the leading event dim (image-shaped: per-pixel C x C maps)
        mask = _parity_mask(in_dims, masktype == "channel")
        layers = []
        for _ in range(coupling_blocks):
            affine = [LUTransform(D, prior_scale) for _ in range(lu_transform)]
            if householder > 0:
                affine.append(HouseholderTransform(dim=D, nvs=householder, device="cpu"))
            conj = BlockAffineTransform(in_dims, SequentialAffineTransform(affine)) if affine else None
            if conj is not None:
                layers.append(conj)
            layers.append(self._coupling_cls(mask, conditioner_cls(**conditioner_args)))
            if affine_conjugation and conj is not None:
                layers.append(InverseTransform(conj))
            mask = 1 - mask
        layers.append(BlockAffineTransform(in_dims, LUTransform(D, prior_scale)))
        layers.append(ScaleTransform(in_dims))
        super().__init__(base_distribution, layers, soft_training=soft_training,
                         training_noise_prior=training_noise_prior, device=device)

    create_checkerboard_mask = staticmethod(lambda in_dims, invert=False: _parity_mask(in_dims, False, invert))
    create_channel_mask = staticmethod(lambda in_dims, invert=False: _parity_mask(in_dims, True, invert))

    def log_prior(self):
        if self.prior_scale is None:
            return 0
        return super().log_prior()

    def log_abs_det_jacobian(self, x):
        """`NonUSFlow.log_abs_det_jacobian(x)` (`nf4ad/flows.py:160-169`), quirk included: every layer is
        evaluated at the data point `x` (it is never advanced through the stack), so the value is the true
        log-det only for data-independent layers (USFlow).  Only the evaluation notebook calls it."""
        total = 0
        for layer in reversed(self.layers):
            try:
                total = total - layer.log_abs_det_jacobian(layer.backward(x), x)
            except Exception:
                continue
        return total


class USFlow(_StackedFlow):
    """`src.usflows.flows.USFlow`: additive couplings => data-independent total log-det."""

    _coupling_cls = MaskedCoupling


class NonUSFlow(_StackedFlow):
    """Mirror of `nf4ad.flows.NonUSFlow` (`nf4ad/flows.py:27-125`): affine couplings."""

    _coupling_cls = MaskedAffineCoupling
