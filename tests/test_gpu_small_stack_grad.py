"""The one-kernel input-gradient path (`usf_small_stack_grad_kernel`, csrc/usf_small.cu): log p and d log p / dx of a
small event shape (D + context <= 64) in one launch, against the fp64 interpreter of the packed stack and the harness of
test_gpu_stack_grad_kernels.py (NaN-filled, misaligned workspace of exactly the queried size, sentinels, ldx > D with NaN
pads), and at the Flow level against the fp64 oracle.

Beyond the interpreter bounds, the path has to give:
  * log p bit-identical to usf_stack_run's on the same descriptor, without deterministic mode (both run the same forward
    code on the same staged weights);
  * a gradient that is bit-identical from run to run and does not depend on how the rows are split into calls;
  * launches == 1 wherever usf_stack_grad_is_single_kernel says so, and the launch chain where it refuses a stack.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from _cases import build_flow, randomize_constants, tame
from test_gpu_stack_grad_kernels import K, P, LP_TOL, assert_grad_rows, call_grad, call_run, grad_stack, inputs as _inputs, \
    lp_err, ref_grad  # noqa: F401  (K, P: fixtures)
import test_gpu_stack_grad_kernels as base

pytestmark = pytest.mark.gpu

CASES = {
    # name: kind, D, K, conditioner, base, gain, kwargs
    "C4-D6": ("NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C4-D64": ("NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "fixture-D32": ("NonUSFlow", 32, 3, ("mlp", [128]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C1-D2": ("USFlow", 2, 10, ("densenn1", [128, 128]), "usnormal", 0.5,
              dict(affine_conjugation=True, householder=0, prior_scale=1.0)),                     # additive couplings
    "laplace-D6": ("NonUSFlow", 6, 3, ("mlp", [6]), "laplace", 0.25, dict(affine_conjugation=True)),
    "cond-D20": ("NonUSFlow", 20, 4, ("cond2", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    # five 96-wide hidden layers: the scoring kernel takes it, the gradient kernel's five hidden slots do not fit
    "deep96-D16": ("NonUSFlow", 16, 1, ("mlp", [96] * 5), "normal", 0.25, dict(affine_conjugation=True)),
}
REFUSED = ("deep96-D16",)
# the small cases of test_gpu_stack_grad_kernels.py that the one-kernel path takes (D1 has Da = 0: the scoring kernel
# refuses it, and so does the gradient kernel)
EXISTING = ("nohid40", "deep24", "D3", "cond16")
ALL = [n for n in CASES if n not in REFUSED] + list(EXISTING)


def case_flow(O, P, name):
    if name in EXISTING:
        return base.flows(O, P, name)[1]
    if name not in base._FLOWS:
        kind, D, nb, cond, bd, gain, kw = CASES[name]
        seed = D * 7 + nb
        torch.manual_seed(seed)
        fo = build_flow(O, kind, D, nb, cond, base=bd, **kw)
        tame(fo, gain)
        randomize_constants(fo, seed)
        fp = build_flow(P, kind, D, nb, cond, base=bd, **kw)
        fp.load_state_dict(fo.state_dict())
        base._FLOWS[name] = (fo.double(), fp.to("cuda").eval())
    return base._FLOWS[name][1]


def case_rows(name, B=256, seed=5):
    if name in EXISTING:
        x, ctx = _inputs(name, B, seed)
    else:
        D, cond = CASES[name][1], CASES[name][3]
        x = torch.randn(B, D, generator=torch.Generator().manual_seed(seed))
        ctx = torch.rand(B, 1, generator=torch.Generator().manual_seed(seed + 1)) * 0.2 if cond[0] == "cond2" else None
    return (x if ctx is None else torch.cat([x, ctx], 1)).float().cuda()


def query(K, cs):
    return K.lib().usf_stack_grad_is_single_kernel(C.byref(cs.desc), C.byref(cs.grad_desc), K.USF_PREC_FP32)


@pytest.mark.parametrize("name", ALL)
def test_single_kernel_matches_interpreter(K, O, P, name):
    """One launch; log p torch.equal to usf_stack_run's (not deterministic mode); log p and every qualifying gradient
    row within the fp32 bounds of the launch chain against the interpreter."""
    cs = grad_stack(case_flow(O, P, name), "fp32")
    assert cs.single_kernel and query(K, cs) == 1 and cs.grad_single_kernel
    xin = case_rows(name)
    lp, g, n = call_grad(K, cs, "fp32", xin)
    assert n == 1
    lq, _ = call_run(K, cs, "fp32", xin)
    assert torch.equal(lp, lq), float(lp_err(lp, lq).max())
    lp_ref, g_ref, margin = ref_grad(cs, "fp32", xin)
    assert float(lp_err(lp, lp_ref).max()) <= LP_TOL["fp32"]
    assert_grad_rows(name, "fp32", g, g_ref, margin)


@pytest.mark.parametrize("name", ["C4-D6", "C4-D64", "C1-D2", "cond-D20"])
def test_bitwise_repeat_and_row_split(K, O, P, name):
    """More row tiles than the grid holds: the same bits twice, and the same bits for the rows of calls of 1, 63, 64 and
    65 rows at tile-straddling offsets; B = 0 writes nothing."""
    cs = grad_stack(case_flow(O, P, name), "fp32")
    B = torch.cuda.get_device_properties(0).multi_processor_count * 8 * 64 + 100
    xin = case_rows(name, B=B, seed=11)
    lp, g, n = call_grad(K, cs, "fp32", xin)
    lp2, g2, _ = call_grad(K, cs, "fp32", xin)
    assert n == 1 and torch.equal(lp, lp2) and torch.equal(g, g2)
    for r0, rows in ((0, 1), (5, 63), (64, 64), (100, 65), (B - 65, 65)):
        lpc, gc, _ = call_grad(K, cs, "fp32", xin[r0:r0 + rows])
        assert torch.equal(lpc, lp[r0:r0 + rows]) and torch.equal(gc, g[r0:r0 + rows]), (r0, rows)
    call_grad(K, cs, "fp32", xin[:0])


def test_workspace(K, O, P):
    """A stack whose saved rows live in the workspace (C1-D2: eleven blocks) and one whose rows stay in shared memory:
    the queried bytes at any offset succeed, one byte short returns USF_E_WORKSPACE and writes nothing."""
    for name in ("C1-D2", "C4-D6"):
        cs = grad_stack(case_flow(O, P, name), "fp32")
        xin = case_rows(name, B=70)
        for off in (0, 3, 255):
            call_grad(K, cs, "fp32", xin, ws_off=off)
        call_grad(K, cs, "fp32", xin, short=1, expect=-3)


@pytest.mark.parametrize("name", REFUSED)
def test_refused_stack_keeps_the_chain(K, O, P, name):
    """The scoring kernel takes the stack, the gradient kernel does not: the gradient runs the launch chain, correctly."""
    cs = grad_stack(case_flow(O, P, name), "fp32")
    assert cs.single_kernel and query(K, cs) == 0 and not cs.grad_single_kernel
    xin = case_rows(name)
    lp, g, n = call_grad(K, cs, "fp32", xin)
    assert n > 1
    lp_ref, g_ref, margin = ref_grad(cs, "fp32", xin)
    assert float(lp_err(lp, lp_ref).max()) <= LP_TOL["fp32"]
    assert_grad_rows(name, "fp32", g, g_ref, margin)


def test_query_is_fp32_only(K, O, P):
    """usf_stack_grad_is_single_kernel is 0 at the tensor-core tier, the one-kernel path is fp32 only."""
    cs = grad_stack(case_flow(O, P, "C4-D6"), "bf16x2")
    assert K.lib().usf_stack_grad_is_single_kernel(C.byref(cs.desc), C.byref(cs.grad_desc), K.USF_PREC_BF16X2) == 0


# ------------------------------------------------------------------------------------------------------------------
# Flow level
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["C4-D6", "fixture-D32"])
def test_flow_auto(O, P, name):
    """Flow.log_prob_and_grad under "auto": one launch at fp32, lp torch.equal to the fused log_prob (no_grad: with
    trainable parameters and grad mode on, log_prob differentiates the layer-wise pass instead), both within the bounds
    of test_full_depth_against_oracle; ADBenchFlow.score_gradients is -g."""
    from test_gpu_log_prob_grad import FP32_TOL, GRAD_TOL, oracle_grad, rel, row_err
    from nf4ad_b200.adbench import ADBenchFlow
    case_flow(O, P, name)
    fo, fp = base._FLOWS[name]
    fp.precision = "auto"
    D = CASES[name][1]
    x = torch.randn(256, D, generator=torch.Generator().manual_seed(5))
    xc = x.cuda()
    lp, g = fp.log_prob_and_grad(xc)
    assert fp.last_grad_precision == "fp32" and fp.last_launches == 1
    with torch.no_grad():
        lq = fp.log_prob(xc)
    assert fp.last_launches == 1 and torch.equal(lp, lq)
    lp_ref, g_ref, kink = oracle_grad(fo, x)
    e = row_err(g, g_ref)
    bad = e > GRAD_TOL
    assert float(e.median()) <= 1e-4 and bool((kink[bad] < 1e-4).all()), (e[bad], kink[bad])
    assert rel(lp, lp_ref) <= FP32_TOL and rel(lq, lp_ref) <= FP32_TOL
    model = ADBenchFlow(fp, batch_size=256, epochs=1, lr=1e-3, device="cuda", verbose=False)
    sg = model.score_gradients(x.numpy(), chunk_rows=100)
    assert np.array_equal(sg, (-g).cpu().numpy())
