"""`Flow.log_prob_and_grad`: log p(x) and d log p(x) / dx per row on the reverse launch chain (fp32 SIMT and bf16x2
tensor-core tiers), against the golden fp64 gradients, the fp64 oracle's autograd at full depth, and the product's own
autograd route; its invariants (determinism, no autograd state, shapes, chunking, weight updates), the autograd fallback
of the stacks the fused path does not take, and `ADBenchFlow.score_gradients`."""
import numpy as np
import pytest
import torch

from _cases import build_flow, flow_from_case, flow_from_r2_case, golden_names, load_golden, load_golden_r2, \
    randomize_constants, tame

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
GRAD_TOL = 1e-3
CHUNK = 16384        # rows per pass of the reverse chain (csrc/usf_grad.cu kGradChunkRows)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float(((a - b).abs() / b.abs().clamp_min(1.0)).max())


def relmax(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def row_err(a, b):
    a, b = a.detach().double().cpu().flatten(1), b.detach().double().cpu().flatten(1)
    return (a - b).abs().amax(1) / b.abs().amax(1).clamp_min(1.0)


@pytest.fixture(scope="module")
def P():
    assert torch.cuda.is_available()
    import nf4ad_b200
    return nf4ad_b200.namespace()


def _pair(O, P, kind, D, K, cond, base, gain, seed, **kw):
    torch.manual_seed(seed)
    fo = build_flow(O, kind, D, K, cond, base=base, **kw)
    tame(fo, gain)
    randomize_constants(fo, seed)
    fp = build_flow(P, kind, D, K, cond, base=base, **kw)
    fp.load_state_dict(fo.state_dict())
    return fo.double(), fp.to("cuda").eval()


def oracle_grad(fo, x, ctx=None):
    """fp64 (log p, d log p / dx) and, per row, the smallest |pre-activation| of any ReLU of the pass (inf: none seen)."""
    mins = []
    hooks = [m.register_forward_hook(lambda m, i, o: mins.append(i[0].detach().abs().flatten(1).amin(1)))
             for m in fo.modules() if isinstance(m, torch.nn.ReLU)]
    try:
        xd = x.double().clone().requires_grad_(True)
        lp = fo.log_prob(xd) if ctx is None else fo.log_prob(xd, ctx.double())
        g, = torch.autograd.grad(lp.sum(), xd)
    finally:
        for h in hooks:
            h.remove()
    kink = torch.stack(mins).amin(0) if mins else torch.full((x.shape[0],), float("inf"), dtype=torch.float64)
    return lp.detach(), g, kink


def autograd_route(fp, x, ctx=None):
    """The route the method replaces: x.requires_grad_() + log_prob + autograd.grad on the fp32 kernels."""
    prev, fp.precision = fp.precision, "fp32"
    try:
        xr = x.clone().requires_grad_(True)
        lp = fp.log_prob(xr) if ctx is None else fp.log_prob(xr, ctx)
        g, = torch.autograd.grad(lp.sum(), xr)
    finally:
        fp.precision = prev
    return lp.detach(), g


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
@pytest.mark.parametrize("name", golden_names())
def test_golden_grad(P, name, tier):
    """g["grad_x"] is the fp64 gradient of -mean(log p): the per-row gradient of log p is -B grad_x."""
    g = load_golden(name)
    flow = flow_from_case(P, g["case"])
    flow.load_state_dict({k: v.float() for k, v in g["state_dict"].items()})
    flow = flow.to("cuda").eval()
    flow.precision = tier
    x = g["x"].float().cuda()
    lp, gx = flow.log_prob_and_grad(x)
    assert flow.last_grad_precision == tier
    assert rel(lp, g["log_prob"]) < FP32_TOL
    assert relmax(gx, -x.shape[0] * g["grad_x"]) < 2e-3


FULL = [
    # id, kind, D, K, conditioner, base, gain, kwargs -- BASELINE.json configs at full depth
    ("C2-D784", "NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C3-D784", "NonUSFlow", 784, 11, ("mlp", [200, 200, 200]), "laplace", 0.25, dict(affine_conjugation=True, householder=0)),
    ("C1-D128", "USFlow", 128, 10, ("densenn1", [128, 128]), "usnormal", 0.5,
     dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
    ("C4-D500", "NonUSFlow", 500, 3, ("mlp", [128]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-D6", "NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("cond2-D16", "NonUSFlow", 16, 3, ("cond2", [32]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
]


@pytest.mark.parametrize("cfg", FULL, ids=lambda c: c[0])
def test_full_depth_against_oracle(O, P, cfg):
    """Every row's gradient within 1e-3 of the fp64 oracle's autograd (relative to the row's scale) and log p within
    1e-4, at the tier "auto" resolves to and at fp32; the same bound against the product's own autograd route.

    The gradient of a ReLU conditioner jumps where a hidden pre-activation crosses 0.  At bf16x2 the hidden activations
    carry ~1e-5 of error, so a row with a unit that close to its kink takes the other branch of the gradient (on C2 at
    256 rows: 5 rows of 1.5e-3 .. 1.2e-2, every one with a pre-activation within 2e-5 of 0 in the fp64 pass; median row
    8.5e-5).  Rows beyond 1e-3 are allowed only if the fp64 pass has a pre-activation within 1e-4 of the kink."""
    name, kind, D, K, cond, base, gain, kw = cfg
    fo, fp = _pair(O, P, kind, D, K, cond, base, gain, seed=D * 7 + K, **kw)
    B = 256
    x = torch.randn(B, D, generator=torch.Generator().manual_seed(5))
    ctx = torch.rand(B, 1, generator=torch.Generator().manual_seed(6)) * 0.2 if cond[0] == "cond2" else None
    lp_ref, g_ref, kink = oracle_grad(fo, x, ctx)
    xc, cc = x.cuda(), (ctx.cuda() if ctx is not None else None)
    for precision in ("auto", "fp32"):
        fp.precision = precision
        lp, g = fp.log_prob_and_grad(xc, cc)
        want = "bf16x2" if (precision == "auto" and D >= fp.BF16_MIN_DIM) else "fp32"
        assert fp.last_grad_precision == want
        assert g.shape == x.shape and g.dtype == torch.float32 and lp.shape == (B,)
        e = row_err(g, g_ref)
        print(f"{name} {want}: grad row_err max {float(e.max()):.2e} median {float(e.median()):.2e}, "
              f"log_prob {rel(lp, lp_ref):.2e}")
        bad = e > GRAD_TOL
        assert float(e.median()) <= 1e-4 and bool((kink[bad] < 1e-4).all()), (e[bad], kink[bad])
        assert rel(lp, lp_ref) <= FP32_TOL
    lp_a, g_a = autograd_route(fp, xc, cc)
    e = row_err(g, g_a)
    assert float(e.median()) <= 1e-4 and bool((kink[e > GRAD_TOL] < 1e-4).all())
    assert rel(lp, lp_a) <= FP32_TOL


@pytest.mark.parametrize("precision,D,hidden", [("fp32", 50, [256, 256]), ("bf16x2", 128, [256, 256])])
def test_invariants(O, P, precision, D, hidden):
    _, fp = _pair(O, P, "NonUSFlow", D, 4, ("mlp", hidden), "normal", 0.25, seed=11, affine_conjugation=True)
    fp.precision = precision
    fp.deterministic = True
    x = torch.randn(1000, D, generator=torch.Generator().manual_seed(7)).cuda()
    lp, g = fp.log_prob_and_grad(x)
    assert fp.last_grad_precision == precision
    # deterministic mode: log p bit-identical to the launch chain of log_prob at the fp32 tier; at bf16x2 the two agree
    # to the tier's accuracy (measured 3e-6) but not bit for bit
    with torch.no_grad():
        lq = fp.log_prob(x)
    assert fp.effective_precision == precision
    assert torch.equal(lp, lq) if precision == "fp32" else rel(lp, lq) < FP32_TOL
    # run to run: bit-identical
    lp2, g2 = fp.log_prob_and_grad(x)
    assert torch.equal(g, g2) and torch.equal(lp, lp2)
    # no autograd state, under no_grad too
    assert lp.grad_fn is None and g.grad_fn is None and not g.requires_grad
    assert all(p.grad is None for p in fp.parameters())
    with torch.no_grad():
        lp3, g3 = fp.log_prob_and_grad(x)
    assert torch.equal(g3, g)
    # B = 0
    lp0, g0 = fp.log_prob_and_grad(x[:0])
    assert lp0.shape == (0,) and g0.shape == (0, D)
    # leading batch dimensions, non-contiguous rows
    lpl, gl = fp.log_prob_and_grad(x[:600].reshape(3, 200, D))
    assert lpl.shape == (3, 200) and gl.shape == (3, 200, D)
    assert torch.equal(gl.reshape(600, D), g[:600]) and torch.equal(lpl.reshape(600), lp[:600])
    xt = x.t().contiguous().t()
    assert not xt.is_contiguous()
    assert torch.equal(fp.log_prob_and_grad(xt)[1], g)
    # more than two internal chunks plus a ragged tail == chunk-by-chunk calls
    big = torch.randn(2 * CHUNK + 123, D, generator=torch.Generator().manual_seed(8)).cuda()
    lpb, gb = fp.log_prob_and_grad(big)
    for i in range(0, big.shape[0], CHUNK):
        lpi, gi = fp.log_prob_and_grad(big[i:i + CHUNK])
        assert torch.equal(gi, gb[i:i + CHUNK]) and torch.equal(lpi, lpb[i:i + CHUNK])


def test_fallback_autograd(P):
    """Stacks the fused path does not take (image-shaped events, softplus scales, an opaque conditioner) return the
    autograd gradient of the layer-wise pass."""
    flows = []
    for name in ("nonus_img_c3_4x4_k3_channel_laplace", "nonus_d8_k2_softplus"):
        case = load_golden_r2(name)
        f = flow_from_r2_case(P, case["case"])
        f.load_state_dict({k: v.float() for k, v in case["state_dict"].items()})
        flows.append((f.to("cuda").eval(), case["x"].float().cuda()))
    torch.manual_seed(3)
    f = build_flow(P, "NonUSFlow", 8, 2, ("mlp", [16]), affine_conjugation=True)
    for layer in f.layers:                       # Tanh instead of ReLU: not a Linear/ReLU chain
        net = getattr(getattr(layer, "conditioner", None), "net", None)
        if net is not None:
            net[1] = torch.nn.Tanh()
    flows.append((f.to("cuda").eval(), torch.randn(64, 8, device="cuda")))
    for flow, x in flows:
        lp, g = flow.log_prob_and_grad(x)
        assert flow.last_grad_precision == "autograd"
        xr = x.clone().requires_grad_(True)
        lp_a = flow.log_prob(xr)
        g_a, = torch.autograd.grad(lp_a.sum(), xr)
        assert g.shape == x.shape and lp.shape == lp_a.shape
        assert torch.allclose(g, g_a) and torch.allclose(lp, lp_a.detach())
        assert lp.grad_fn is None and all(p.grad is None for p in flow.parameters())


def test_score_gradients_and_weight_updates(P):
    """`ADBenchFlow.score_gradients` is -g of log_prob_and_grad; after `fit` (FusedAdam steps) the packed transposes
    are rebuilt: the gradient follows the new weights."""
    from nf4ad_b200.adbench import ADBenchFlow
    torch.manual_seed(4)
    flow = build_flow(P, "NonUSFlow", 64, 3, ("mlp", [64]), affine_conjugation=True, prior_scale=1.0).to("cuda")
    data = np.random.default_rng(0).standard_normal((2048, 64)).astype(np.float32)
    X = torch.from_numpy(data[:512]).cuda()
    model = ADBenchFlow(flow, batch_size=256, epochs=1, lr=1e-3, device="cuda", verbose=False)
    flow.eval()
    _, g_before = flow.log_prob_and_grad(X)
    model.fit(data)
    flow.eval()
    lp, g = flow.log_prob_and_grad(X)
    assert not torch.equal(g, g_before)
    lp_a, g_a = autograd_route(flow, X)
    assert float(row_err(g, g_a).max()) <= GRAD_TOL and rel(lp, lp_a) <= FP32_TOL
    sg = model.score_gradients(data[:512], chunk_rows=200)
    assert sg.shape == (512, 64) and sg.dtype == np.float32
    assert np.array_equal(sg, (-g).cpu().numpy())
