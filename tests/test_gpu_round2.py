"""GPU parity, round 2: the rows of SURVEY.md section 8 the first round left partial -- every BASELINE.json config at
FULL depth with a max-row tolerance, the softplus / same-shape / ValueError branches of `_parse_params`, the
`log_abs_det_jacobian(x)` quirk, the `export` switch, conditional (context) flows and soft training, image-shaped
events, SophiaG, and the score -> train -> score weight-cache sequence."""
import numpy as np
import pytest
import torch

from _cases import (build_flow, flow_from_r2_case, golden_r2_names, load_golden, load_golden_r2, flow_from_case,
                    randomize_constants, tame)

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_TOL = 1e-2


def lp_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs() / b.abs().clamp_min(1.0)


def row_err(a, b):
    a, b = a.detach().double().cpu().flatten(1), b.detach().double().cpu().flatten(1)
    return (a - b).abs().amax(1) / b.abs().amax(1).clamp_min(1.0)


def relmax(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


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


# BASELINE.json configs (SURVEY 8d "Config -> concrete stack") at their FULL depth
FULL_DEPTH = [
    ("C1-gmm-D2", "USFlow", 2, 10, ("densenn1", [128, 128]), "usnormal", 0.5, dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
    ("C1-gmm-D128", "USFlow", 128, 10, ("densenn1", [128, 128]), "usnormal", 0.5, dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
    ("C2-mnist-D784", "NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C3-fashion-D784", "NonUSFlow", 784, 11, ("mlp", [200, 200, 200]), "laplace", 0.25, dict(affine_conjugation=True, householder=0)),
    ("C4-adbench-D6", "NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-adbench-D64", "NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-adbench-D500-K3", "NonUSFlow", 500, 3, ("mlp", [128]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    ("C4-adbench-D500-K8", "NonUSFlow", 500, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True)),
    ("C5-mvtec-D128", "USFlow", 128, 10, ("densenn1", [512, 256]), "normal", 0.5, dict(affine_conjugation=True, householder=0)),
    ("C5-mvtec-D256", "NonUSFlow", 256, 10, ("mlp", [512, 256]), "normal", 0.25, dict(affine_conjugation=True)),
]


@pytest.mark.parametrize("cfg", FULL_DEPTH, ids=lambda c: c[0])
def test_full_depth_configs_max_row(O, P, cfg):
    """Every BASELINE.json config shape at full depth: EVERY row's log_prob within 1e-4 (fp32 / 3xTF32) and 1e-2
    (`precision="bf16"`) of the fp64 oracle; round trip reported."""
    name, kind, D, K, cond, base, gain, kw = cfg
    fo, fp = _pair(O, P, kind, D, K, cond, base, gain, seed=D * 13 + K, **kw)
    B = 192
    x = torch.randn(B, D, generator=torch.Generator().manual_seed(42))
    with torch.no_grad():
        ref = fo.log_prob(x.double())
        z_ref = fo.backward(x.double())
        xc = x.cuda()
        for precision, tol in (("fp32", FP32_TOL), ("auto", FP32_TOL), ("bf16x2", FP32_TOL), ("tf32x3", 2e-4), ("bf16", BF16_TOL)):
            fp.precision = precision
            lp = fp.log_prob(xc)
            assert fp.last_launches > 0, "fused CUDA path did not run"
            e = lp_err(lp, ref)
            z = fp.backward(xc)
            rt = row_err(fp.latent_to_data(z), x)
            print(f"[{name} {precision} -> {fp.effective_precision}] launches {fp.last_launches} log_prob max-row err "
                  f"{float(e.max()):.2e} latent {float(row_err(z, z_ref).max()):.2e} round-trip max {float(rt.max()):.2e}")
            assert float(e.max()) < tol, (name, precision, float(e.max()))


@pytest.mark.parametrize("name", golden_r2_names())
def test_round2_golden(P, name):
    """Image-shaped events (per-pixel LU blocks, N-D masks, conv conditioner, 2C-channel split), softplus scale activation,
    same-shape conditioner output, conditional flow: the product on CUDA against what the reference's own classes
    produced in fp64 (tests/golden/make_golden_r2.py) -- values, latents, samples and every gradient."""
    g = load_golden_r2(name)
    flow = flow_from_r2_case(P, g["case"])
    flow.load_state_dict({k: v.float() for k, v in g["state_dict"].items()})
    flow = flow.to("cuda").eval()
    x = g["x"].float().cuda()
    ctx = None if g["context"] is None else g["context"].float().cuda()
    with torch.no_grad():
        lp = flow.log_prob(x, ctx)
        assert lp.shape == (g["case"]["B"],)
        assert float(lp_err(lp, g["log_prob"]).max()) < FP32_TOL
        fused = flow.last_launches > 0 and isinstance(g["case"]["D"], int) and not g["case"].get("scale_activation")
        z = flow.backward(x, ctx)
        assert z.shape == x.shape and relmax(z, g["latent"]) < FP32_TOL
        xs = flow.latent_to_data(g["z_sample"].float().cuda(), ctx)
        assert relmax(xs, g["x_from_z"]) < FP32_TOL
        if g["ladj_quirk"] is not None:          # NonUSFlow.log_abs_det_jacobian(x): flows.py:160-169, x never advanced
            q = torch.as_tensor(flow.log_abs_det_jacobian(x))
            assert relmax(q, g["ladj_quirk"]) < FP32_TOL
        if g["case"].get("context"):
            assert fused, "a conditional flow must run the fused chain (context columns)"
            for prec, tol in (("bf16x2", FP32_TOL), ("tf32x3", 2e-4), ("bf16", BF16_TOL)):
                flow.precision = prec
                assert float(lp_err(flow.log_prob(x, ctx), g["log_prob"]).max()) < tol
            flow.precision = "fp32"
    # training path: hand-written backward kernels against the reference's autograd
    flow.train()
    xg = x.clone().requires_grad_(True)
    lp = flow.log_prob(xg, ctx)
    assert float(lp_err(lp, g["log_prob"]).max()) < FP32_TOL
    (-lp.mean()).backward()
    assert relmax(xg.grad, g["grad_x"]) < 2e-3
    for n, p in flow.named_parameters():
        ref = g["grad_params"][n]
        if ref is None:
            continue
        got = p.grad
        assert got is not None, n
        if n.endswith("L_raw"):
            got, ref = got.tril(-1), ref.tril(-1)
        if n.endswith("U_raw"):
            got, ref = got.triu(), ref.triu()
        assert relmax(got, ref) < 2e-3, n


def test_parse_params_branches_on_cuda(O, P):
    """a9: a conditioner whose output fits none of the three accepted forms raises the reference's ValueError
    (`transforms.py:57-60`); an unknown scale_activation raises `Unsupported scale_activation` (`:86-87`)."""
    from _cases import MLP
    T = P.transforms
    mask = (torch.arange(6) % 2).float().view(1, 6)
    bad = T.MaskedAffineCoupling(mask, MLP(6, [8], 9)).to("cuda")
    with pytest.raises(ValueError, match="Conditioner output shape not compatible"):
        bad.forward(torch.randn(4, 6, device="cuda"))
    odd = T.MaskedAffineCoupling(mask, MLP(6, [8], 12), scale_activation="sigmoid").to("cuda")
    with pytest.raises(ValueError, match="Unsupported scale_activation"):
        odd.backward(torch.randn(4, 6, device="cuda"))
    # the (s, t) tuple form and the 2C form agree when they carry the same numbers
    torch.manual_seed(0)
    net = MLP(6, [8], 12).cuda()

    class Pair(torch.nn.Module):
        def forward(self, x):
            p = net(x)
            return p[:, :6], p[:, 6:]

    a = T.MaskedAffineCoupling(mask, net).cuda()
    b = T.MaskedAffineCoupling(mask, Pair()).cuda()
    x = torch.randn(5, 6, device="cuda")
    with torch.no_grad():
        assert torch.allclose(a.forward(x), b.forward(x), atol=1e-6)
        assert torch.allclose(a.log_abs_det_jacobian(x, a.forward(x)), b.log_abs_det_jacobian(x, b.forward(x)), atol=1e-6)


def test_export_switch(O, P):
    """a3: `model.export = "backward"; model.forward(x)` (`visualization.py:85-86`) and the other three settings."""
    g = load_golden("nonus_d8_k2_conj_hh1")
    flow = flow_from_case(P, g["case"])
    flow.load_state_dict({k: v.float() for k, v in g["state_dict"].items()})
    flow = flow.to("cuda").eval()
    x = g["x"].float().cuda()
    with torch.no_grad():
        assert flow.export == "log_prob"
        assert relmax(flow(x), g["log_prob"]) < FP32_TOL
        flow.export = "backward"
        assert relmax(flow.forward(x), g["latent"]) < FP32_TOL
        flow.export = "forward"
        assert relmax(flow(g["z_sample"].float().cuda()), g["x_from_z"]) < FP32_TOL
        flow.export = "sample"
        s = flow()
        assert s.shape == (8,) and s.is_cuda and bool(torch.isfinite(s).all())


def test_context_on_an_unconditional_flow_is_passed_as_given(O, P):
    """A non-None context on a flow whose conditioners are opaque modules taking `(x, context)` runs the layer-wise
    kernels with the conditioner evaluated as given (`transforms.py:71-74`) -- checked against the oracle."""
    class CtxCond(torch.nn.Module):
        def __init__(self, d):
            super().__init__()
            self.a = torch.nn.Linear(d, 2 * d)
            self.c = torch.nn.Linear(1, 2 * d)

        def forward(self, x, context=None):
            out = self.a(x)
            return out if context is None else out + torch.tanh(self.c(context))

    D = 10
    torch.manual_seed(2)
    bd = lambda ns: ns.dist.Normal(torch.zeros(D), torch.ones(D))
    fo = O.NonUSFlow(bd(O), [D], 2, CtxCond, dict(d=D), affine_conjugation=True)
    fp = P.NonUSFlow(bd(P), [D], 2, CtxCond, dict(d=D), affine_conjugation=True)
    tame(fo, 0.25)
    fp.load_state_dict(fo.state_dict())
    fo, fp = fo.double(), fp.to("cuda").eval()
    x = torch.randn(9, D)
    ctx = torch.rand(9, 1)
    with torch.no_grad():
        ref = fo.log_prob(x.double(), ctx.double())
        got = fp.log_prob(x.cuda(), ctx.cuda())
        assert float(lp_err(got, ref).max()) < FP32_TOL
        assert float(lp_err(fp.log_prob(x.cuda()), fo.log_prob(x.double())).max()) < FP32_TOL     # and without one
        assert float((fp.log_prob(x.cuda(), ctx.cuda()) - fp.log_prob(x.cuda())).abs().max()) > 1e-3


def test_soft_training_fit_and_scoring(O, P):
    """f2: `soft_training=True` -- `Flow.fit` perturbs each sample with its own noise level drawn from
    `training_noise_prior` and conditions on it; scoring without a context means noise level 0.  Scoring agrees with the
    oracle (same weights), the conditional flow runs the fused chain, training lowers the loss and replays as a graph."""
    D = 16
    torch.manual_seed(1)
    prior = lambda ns, dev: ns.dist.Uniform(torch.tensor(0.0, device=dev), torch.tensor(0.2, device=dev))
    kw = dict(affine_conjugation=True, prior_scale=1.0, soft_training=True)
    fo = build_flow(O, "NonUSFlow", D, 3, ("cond2", [32]), training_noise_prior=prior(O, "cpu"), **kw)
    tame(fo, 0.25)
    fp = build_flow(P, "NonUSFlow", D, 3, ("cond2", [32]), training_noise_prior=prior(P, "cpu"), **kw)
    fp.load_state_dict(fo.state_dict())
    fo, fp = fo.double(), fp.to("cuda").eval()
    assert fp.training_noise_prior.low.is_cuda                      # moved with the flow
    x = torch.randn(64, D, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        got = fp.log_prob(x.cuda())
        assert fp.last_launches > 0
        assert float(lp_err(got, fo.log_prob(x.double())).max()) < FP32_TOL
        ctx = torch.full((64, 1), 0.1)
        assert float(lp_err(fp.log_prob(x.cuda(), ctx.cuda()), fo.log_prob(x.double(), ctx.double())).max()) < FP32_TOL
        s = fp.sample([5])
        assert s.shape == (5, D) and bool(torch.isfinite(s).all())
    data = torch.randn(512, D, generator=torch.Generator().manual_seed(4)) * 0.5 + 0.3
    losses = fp.fit(data, torch.optim.Adam, {"lr": 2e-3}, batch_size=64, epochs=6)
    assert len(losses) == 6 and np.all(np.isfinite(losses)) and losses[-1] < losses[0]
    assert fp.fit_graph_replays >= 8 * 6 - 4
    with torch.no_grad():                                            # the cache followed the training (ADVICE r1 high)
        after = fp.eval().log_prob(x.cuda())
    assert float((after - got).abs().mean()) > 1e-2


def test_score_train_score_sees_the_new_weights(P):
    """ADVICE r1 (high): predict_score -> fit -> predict_score must score with the TRAINED weights: FusedAdam writes the
    parameters through raw pointers and the step is replayed as a CUDA graph, neither of which bumps torch's version
    counters.  The fused scores after training must equal the layer-wise path's on the same weights."""
    from nf4ad_b200.adbench import ADBenchFlow
    rng = np.random.RandomState(0)
    Xtr = (rng.randn(256, 20) * 0.5 + 1.0).astype(np.float32)
    Xte = rng.randn(64, 20).astype(np.float32)
    torch.manual_seed(0)
    flow = build_flow(P, "NonUSFlow", 20, 3, ("mlp", [32]), affine_conjugation=True, prior_scale=1.0)
    tame(flow, 0.25)
    w = ADBenchFlow(flow_model=flow, epochs=3, batch_size=32, lr=2e-3, device="cuda", verbose=False)
    for precision in ("fp32", "bf16"):
        flow.precision = precision
        s0 = w.predict_score(Xte)                       # populates the packed-weight cache
        w.fit(Xtr)
        s1 = w.predict_score(Xte)
        assert np.abs(s1 - s0).mean() > 1e-2, "scores did not move after training: stale packed weights"
        flow.train()                                    # layer-wise kernels on the live parameters
        with torch.no_grad():
            z, neg_ladj = flow._inverse_layers(torch.from_numpy(Xte).cuda())
            ref = -(flow._base_log_prob(z) + neg_ladj)
        flow.eval()
        assert float(lp_err(torch.from_numpy(s1), ref).max()) < (FP32_TOL if precision == "fp32" else BF16_TOL)
        w.fit(Xtr)                                      # and again: fit -> score -> fit -> score
        s2 = w.predict_score(Xte)
        assert np.abs(s2 - s1).mean() > 1e-3
    # Flow.fit with scoring in between epochs
    flow.precision = "fp32"
    with torch.no_grad():
        a = flow.log_prob(torch.from_numpy(Xte).cuda()).clone()
    flow.fit(torch.from_numpy(Xtr), torch.optim.Adam, {"lr": 2e-3}, batch_size=64, epochs=2)
    with torch.no_grad():
        b = flow.eval().log_prob(torch.from_numpy(Xte).cuda())
    assert float((a - b).abs().mean()) > 1e-3


def test_sophia_matches_its_definition(P):
    """`src.usflows.sophia.SophiaG` as a fused kernel against the update rule written out in torch (fp64)."""
    from nf4ad_b200.optim import SophiaG
    torch.manual_seed(0)
    ps = [torch.nn.Parameter(torch.randn(n, device="cuda")) for n in (5, 1000, 8193)]
    ref = [p.detach().double().clone() for p in ps]
    m = [torch.zeros_like(r) for r in ref]
    h = [torch.zeros_like(r) for r in ref]
    lr, b1, b2, rho, wd, k, bs = 1e-2, 0.965, 0.99, 0.04, 0.1, 3, 64.0
    opt = SophiaG(ps, lr=lr, betas=(b1, b2), rho=rho, weight_decay=wd, hessian_interval=k, bs=bs)
    for step in range(1, 8):
        gs = [torch.randn_like(p) * 0.1 for p in ps]
        for p, g in zip(ps, gs):
            p.grad = g.clone()
        opt.step()
        for i, g in enumerate(gs):
            g = g.double()
            if (step - 1) % k == 0:
                h[i] = b2 * h[i] + (1 - b2) * g * g
            ref[i] = ref[i] * (1 - lr * wd)
            m[i] = b1 * m[i] + (1 - b1) * g
            ratio = (m[i].abs() / (rho * bs * h[i] + 1e-15)).clamp(max=1.0)
            ref[i] = ref[i] - lr * m[i].sign() * ratio
    for p, r in zip(ps, ref):
        assert float((p.detach().double() - r).abs().max()) < 1e-5
    # and it trains a flow through Flow.fit as a captured step
    flow = build_flow(P, "USFlow", 8, 2, ("densenn1", [16]), affine_conjugation=True, prior_scale=1.0).to("cuda")
    data = torch.randn(256, 8) * 0.5 + 0.5
    losses = flow.fit(data, SophiaG, {"lr": 5e-3, "weight_decay": 0.0}, batch_size=64, epochs=8)
    assert np.all(np.isfinite(losses)) and losses[-1] < losses[0] and flow.fit_graph_replays > 0


def test_image_shaped_flow_trains_and_samples(P):
    """f4: an image-shaped NonUSFlow (`in_dims=[C, H, W]`, conv conditioner) end to end on the device: sample shape,
    finite scores, a few optimizer steps lower the loss, state_dict round trip (checkpoint keys, `hyperopt.py:206,324`)."""
    torch.manual_seed(0)
    flow = build_flow(P, "NonUSFlow", [4, 8, 8], 2, ("conv", [8]), affine_conjugation=True, prior_scale=1.0, device="cuda")
    tame(flow, 0.25)
    x = torch.randn(32, 4, 8, 8, device="cuda") * 0.5
    s = flow.sample([6])
    assert s.shape == (6, 4, 8, 8) and s.is_cuda
    opt = torch.optim.Adam(flow.parameters(), lr=2e-3)
    first = None
    for _ in range(15):
        opt.zero_grad()
        loss = -flow.log_prob(x).mean()
        loss.backward()
        opt.step()
        first = float(loss.detach()) if first is None else first
    assert float(loss.detach()) < first
    sd = flow.state_dict()
    assert any(k.endswith("L_raw") for k in sd) and any(k.endswith("conditioner.net.0.weight") for k in sd)
    twin = build_flow(P, "NonUSFlow", [4, 8, 8], 2, ("conv", [8]), affine_conjugation=True, prior_scale=1.0, device="cuda")
    twin.load_state_dict(sd)
    with torch.no_grad():
        assert torch.allclose(twin.eval().log_prob(x), flow.eval().log_prob(x), rtol=1e-5, atol=1e-4)


SMALL = [
    # kind, D, K, conditioner, base, kwargs -- shapes the one-kernel path takes (D + context <= 64, widths <= 128)
    ("NonUSFlow", 2, 4, ("mlp", [16]), "normal", dict(affine_conjugation=True)),
    ("USFlow", 2, 10, ("densenn1", [128, 128]), "usnormal", dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
    ("NonUSFlow", 6, 3, ("mlp", [6]), "laplace", dict(affine_conjugation=True, prior_scale=1.0)),
    ("NonUSFlow", 20, 3, ("mlp", [20]), "normal", dict(affine_conjugation=True, prior_scale=1.0)),
    ("NonUSFlow", 32, 3, ("mlp", [128]), "normal", dict(affine_conjugation=True, prior_scale=1.0)),
    ("NonUSFlow", 33, 2, ("densenn2", [40]), "normal", dict(affine_conjugation=False, lu_transform=2, householder=2)),
    ("USFlow", 50, 5, ("mlp_add", [64, 64, 64]), "normal", dict(affine_conjugation=True)),
    ("NonUSFlow", 64, 3, ("mlp", [64]), "normal", dict(affine_conjugation=True, prior_scale=1.0)),
    ("NonUSFlow", 16, 3, ("cond2", [32]), "normal", dict(affine_conjugation=True, soft_training=True)),
]


@pytest.mark.parametrize("cfg", SMALL, ids=lambda c: f"{c[0]}-D{c[1]}-K{c[2]}-{c[3][0]}")
def test_small_stack_single_kernel(O, P, cfg):
    """Small event shapes run the WHOLE stack as one kernel (csrc/usf_small.cu), whatever tier is requested: fp32-grade
    against the fp64 oracle in both directions, ragged batches, deterministic (bit-identical repeats: no atomics)."""
    kind, D, K, cond, base, kw = cfg
    fo, fp = _pair(O, P, kind, D, K, cond, base, 0.5, seed=D * 3 + K, **kw)
    g = torch.Generator().manual_seed(11)
    for B in (1, 63, 64, 65, 1000):
        x = torch.randn(B, D, generator=g)
        zs = torch.randn(B, D, generator=g)
        with torch.no_grad():
            ref, z_ref, xs_ref = fo.log_prob(x.double()), fo.backward(x.double()), fo.latent_to_data(zs.double())
            for precision in ("auto", "fp32", "tf32x3", "bf16x2", "bf16"):
                fp.precision = precision
                lp = fp.log_prob(x.cuda())
                assert fp.last_launches == 1 and fp.effective_precision == "fp32", (precision, fp.last_launches, fp.effective_precision)
                assert float(lp_err(lp, ref).max()) < FP32_TOL
            z = fp.backward(x.cuda())
            assert fp.last_launches == 1 and float(row_err(z, z_ref).max()) < FP32_TOL
            xs = fp.latent_to_data(zs.cuda())
            assert fp.last_launches == 1 and float(row_err(xs, xs_ref).max()) < FP32_TOL
            assert torch.equal(fp.log_prob(x.cuda()), lp) and torch.equal(fp.log_prob(x.cuda()), lp)      # deterministic
    # a row's score does not depend on the batch it travels in
    with torch.no_grad():
        big = torch.randn(70000, D, generator=g).cuda()
        lp = fp.log_prob(big)
        big_tier = fp.effective_precision        # wide layers at this batch size go to the FP32_GRADE_TC chain (Flow._small_ok)
        part = fp.log_prob(big[12345:12400].contiguous())
        if big_tier == "fp32":
            assert fp.last_launches == 1 and torch.equal(lp[12345:12400], part)
        else:
            # two tiers on the same rows (the untrained stress stacks reach |log_prob| ~ 1e9: ill-conditioned)
            assert big_tier == "bf16x2" and float(lp_err(lp[12345:12400], part).max()) < 1e-3
        assert bool(torch.isfinite(lp).all())


def test_deterministic_mode_is_bit_identical(O, P):
    """`flow.deterministic = True` (usf_set_deterministic): the per-row log-det / log-density partial sums go to slots that
    one last kernel adds in a fixed order, instead of fp32 atomics -- log_prob is bit-identical run to run on every tier (as
    the reference's is), equal to the atomic form up to the rounding of the different summation order, and still right."""
    for kind, D, K, cond, base, kw in (
            ("NonUSFlow", 784, 2, ("mlp", [256, 256]), "normal", dict(affine_conjugation=True)),
            ("NonUSFlow", 200, 3, ("mlp", [300]), "laplace", dict(affine_conjugation=True)),        # unfused (hidden > 256)
            ("USFlow", 128, 3, ("densenn1", [64, 64]), "usnormal", dict(affine_conjugation=True, householder=0))):
        fo, fp = _pair(O, P, kind, D, K, cond, base, 0.25, seed=D + K, **kw)
        x = torch.randn(5000, D, generator=torch.Generator().manual_seed(9))
        xc = x.cuda()
        with torch.no_grad():
            ref = fo.log_prob(x[:200].double())
            # ("bf16" is forced onto these untrained stacks here -- bf16_trust -- to exercise its kernels: sanity bound only)
            for tier, tol in (("bf16", 5 * BF16_TOL), ("bf16x2", FP32_TOL), ("tf32x3", 2e-4), ("fp32", FP32_TOL)):
                fp.precision = tier
                fp.bf16_trust = True
                fp.deterministic = False
                loose = fp.log_prob(xc)
                n_loose = fp.last_launches
                fp.deterministic = True
                a = fp.log_prob(xc)
                assert fp.last_launches == n_loose + 1               # the slot-summing kernel
                for _ in range(4):
                    assert torch.equal(fp.log_prob(xc), a), tier
                assert float(lp_err(a, loose).max()) < 1e-5
                assert float(lp_err(a[:200], ref).max()) < tol, (tier, float(lp_err(a[:200], ref).max()))
                # small batch (the fp32 tier's split-K form sums atomically: not used in this mode)
                b = fp.log_prob(xc[:33].contiguous())
                assert torch.equal(fp.log_prob(xc[:33].contiguous()), b) and float(lp_err(b, ref[:33]).max()) < tol
                fp.deterministic = False
