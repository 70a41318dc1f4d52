"""`Flow.log_prob_terms` and `usf_stack_log_prob_terms`: the base log-density and every coupling's log-det term behind
log p(x), from the fused pass of `log_prob`.

The C ABI call is checked with the hostile harness of test_gpu_stack_grad_kernels.py (NaN pads, sentinels, a NaN-filled
misaligned workspace of exactly the queried size) against its fp64 interpreter of the packed stack.  The interpreter sums
the coupling terms of all blocks; a block's own term is the difference of the sums of two prefixes of the stack
(`interp_terms`).  The flow-level terms are checked against the fp64 oracle walked layer by layer.
"""
import ctypes as C
import types

import numpy as np
import pytest
import torch

import test_gpu_stack_grad_kernels as G
from _cases import build_flow, flow_from_case, flow_from_r2_case, load_golden, load_golden_r2, randomize_constants, tame

pytestmark = pytest.mark.gpu

CHUNK = 131072                 # rows per pass of the launch chain (csrc/usf_api.cu kChunkRows)
EPS32 = float(np.finfo(np.float32).eps)

CASES = {
    # name: kind, D, K, conditioner, base, gain, kwargs
    "C1-D2": ("USFlow", 2, 4, ("densenn1", [8]), "usnormal", 0.5, dict(affine_conjugation=True, householder=0,
                                                                       prior_scale=1.0)),
    "C4-D6": ("NonUSFlow", 6, 3, ("mlp", [6]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C4-D64": ("NonUSFlow", 64, 3, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "cond20": ("NonUSFlow", 20, 3, ("cond2", [32]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
}
SINGLE = ("C1-D2", "C4-D6", "C4-D64", "cond20", "fixture-D32", "deep24")   # the one-kernel path at fp32 (D = 1: the chain)
# z at the bf16 tier against the fp32 interpreter, relative to the row's max |z|: the bf16 activations of eight blocks
# (measured 3.0e-2 on C2 on a B200); the bf16 tier's promise is about log p, whose terms stay within 1e-2 (4.5e-3)
BF16_Z_TOL = 5e-2


@pytest.fixture(scope="module")
def K():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from nf4ad_b200 import _lib
    assert _lib.lib().usf_device_ok() == 1, "expected an sm_100 device"
    return _lib


@pytest.fixture(scope="module")
def P():
    import nf4ad_b200
    return nf4ad_b200.namespace()


_FLOWS = {}


def flows(O, P, name):
    """(fp64 oracle flow, product flow on cuda): the cases of test_gpu_stack_grad_kernels.py, the ones above and the
    golden D = 32 fixture."""
    if name in G.CASES:
        return G.flows(O, P, name)
    if name not in _FLOWS:
        if name == "fixture-D32":
            g = load_golden("nonus_d32_k3_fixture")
            fo, fp = flow_from_case(O, g["case"]), flow_from_case(P, g["case"])
            fo.load_state_dict({k: v.double() for k, v in g["state_dict"].items()})
            fp.load_state_dict({k: v.float() for k, v in g["state_dict"].items()})
            _FLOWS[name] = (fo.double(), fp.to("cuda").eval())
        else:
            kind, D, nb, cond, base, gain, kw = CASES[name]
            seed = D * 7 + nb
            torch.manual_seed(seed)
            fo = build_flow(O, kind, D, nb, cond, base=base, **kw)
            tame(fo, gain)
            randomize_constants(fo, seed)
            fp = build_flow(P, kind, D, nb, cond, base=base, **kw)
            fp.load_state_dict(fo.state_dict())
            _FLOWS[name] = (fo.double(), fp.to("cuda").eval())
    return _FLOWS[name]


def inputs(fp, B=G.ROWS, seed=5):
    """(x (B, D), context (B, 1) or None) on the CPU."""
    x = torch.randn(B, fp.event_dim, generator=torch.Generator().manual_seed(seed))
    ctx = torch.rand(B, 1, generator=torch.Generator().manual_seed(seed + 1)) * 0.2 if fp.context_dim() else None
    return x, ctx


def prec(K, tier):
    return {"fp32": K.USF_PREC_FP32, "tf32x3": K.USF_PREC_TF32X3, "bf16x2": K.USF_PREC_BF16X2, "bf16": K.USF_PREC_BF16}[tier]


# ------------------------------------------------------------------------------------------------------------------
# the interpreter, per block
# ------------------------------------------------------------------------------------------------------------------
def _prefix(cs, n):
    """The first n blocks of a packed stack as the interpreter reads it.  The next block's affine map stands in for the
    final map: it reads the layout block n - 1 leaves, so the pass goes through; only its coupling sum is used."""
    st = cs.desc
    desc = types.SimpleNamespace(D=st.D, n_blocks=n, G_final=cs.blocks[n].G, loc=st.loc, inv_scale=st.inv_scale,
                                 base_kind=st.base_kind, const_term=st.const_term)
    return types.SimpleNamespace(desc=desc, blocks=cs.blocks, _keep=cs._keep, _mlp_widths=cs._mlp_widths)


def interp_terms(cs, tier, xin):
    """fp64 (terms (n_blocks + 1, B) in the layout of out_terms, z (B, D)) of the packed stack."""
    nb = cs.desc.n_blocks
    full = G.interpret(cs, tier, xin)
    sums = [torch.zeros_like(full.ladj)] + [G.interpret(_prefix(cs, j), tier, xin).ladj for j in range(1, nb)] + [full.ladj]
    rows = [sums[j + 1] - sums[j] for j in range(nb)]
    rows.append(full.lp - float(cs.desc.const_term) - full.ladj)
    return torch.stack(rows), full.z


# ------------------------------------------------------------------------------------------------------------------
# the C ABI call, with the hostile harness
# ------------------------------------------------------------------------------------------------------------------
def call_terms(K, cs, tier, xin, ws_off=3, short=0, expect=0, deterministic=False):
    """usf_stack_log_prob_terms -> (log p (B,), terms (n_blocks + 1, B), z (B, D), launches); checks everything outside
    the outputs.  `deterministic`: usf_set_deterministic around the call (the call must not depend on it)."""
    lib = K.lib()
    D, din, B, nt = cs.D, cs.D + cs.ctx_dim, xin.shape[0], cs.desc.n_blocks + 1
    ldx, ldz, ldt = din + 5, D + 3, B + 3
    xb = torch.full((B + 1, ldx), G.NAN, dtype=torch.float32, device="cuda")
    xb[:B, :din] = xin
    tb = torch.full((nt + 1, ldt), G.SENTINEL, dtype=torch.float32, device="cuda")
    tb[:nt, :B] = G.NAN
    zb = torch.full((B + 1, ldz), G.SENTINEL, dtype=torch.float32, device="cuda")
    zb[:B, :D] = G.NAN
    lb = torch.full((B + 1,), G.SENTINEL, dtype=torch.float32, device="cuda")
    lb[:B] = G.NAN
    t0, z0, l0 = tb.clone(), zb.clone(), lb.clone()
    prev = lib.usf_set_deterministic(int(deterministic))
    try:
        nbytes = lib.usf_stack_terms_workspace_bytes(C.byref(cs.desc), B, prec(K, tier))
        assert nbytes > 0, lib.usf_last_error()
        buf, wp = G._ws(nbytes, ws_off)
        n = C.c_int(-1)
        rc = lib.usf_stack_log_prob_terms(C.byref(cs.desc), C.c_void_p(xb.data_ptr()), ldx, B, C.c_void_p(lb.data_ptr()),
                                          C.c_void_p(tb.data_ptr()), ldt, C.c_void_p(zb.data_ptr()), ldz, wp,
                                          nbytes - short, prec(K, tier), C.byref(n), K.stream())
        torch.cuda.synchronize()
    finally:
        lib.usf_set_deterministic(prev)
    assert rc == expect, (rc, lib.usf_last_error())
    assert G._ws_untouched(buf, nbytes, ws_off), "wrote outside the workspace"
    bits = lambda t: t.view(torch.int32)
    if rc != 0 or B == 0:
        assert torch.equal(bits(tb), bits(t0)) and torch.equal(bits(zb), bits(z0)) and torch.equal(bits(lb), bits(l0))
        return None, None, None, n.value
    assert torch.equal(bits(tb[:, B:]), bits(t0[:, B:])) and torch.equal(bits(tb[nt]), bits(t0[nt])), "wrote outside out_terms"
    assert torch.equal(bits(zb[:B, D:]), bits(z0[:B, D:])) and torch.equal(bits(zb[B]), bits(z0[B])), "wrote outside out_z"
    assert lb[B].item() == G.SENTINEL, "wrote past out_logprob"
    lp, t, z = lb[:B].clone(), tb[:nt, :B].clone(), zb[:B, :D].clone()
    for v in (lp, t, z):
        assert bool(torch.isfinite(v).all()), "an output element was not written"
    return lp, t, z, n.value


def stack_of(fp, tier):
    cs = fp._stack(True, "cuda", tier)
    assert cs is not None, fp._unsupported_reason
    return cs


def row_scale(cs, t):
    """max(|const_term| + sum |terms|, 1) per row."""
    return (abs(float(cs.desc.const_term)) + t.double().abs().sum(0)).clamp_min(1.0).cpu()


def recombined_gap(cs, lp, t):
    """|log p - (const_term + sum of the rows)| against 64 eps (|const_term| + sum |row|), per row (identity 5)."""
    gap = (lp.double() - (float(cs.desc.const_term) + t.double().sum(0))).abs().cpu()
    return gap, 64 * EPS32 * row_scale(cs, t)


# ------------------------------------------------------------------------------------------------------------------
# 1. the terms against the interpreter
# ------------------------------------------------------------------------------------------------------------------
TIER_CASES = [("C2", t) for t in ("fp32", "bf16x2", "tf32x3", "bf16")] + \
    [(n, "fp32") for n in ("C1-D2", "C1", "C3", "C4-D6", "C4-D64", "fixture-D32", "cond20", "D1", "deep24")]


@pytest.mark.parametrize("name,tier", TIER_CASES)
def test_terms_match_interpreter(K, O, P, name, tier):
    """Every term row within the tier's log p bound of the fp64 interpreter of the same packs (bf16: of the fp32 packs,
    1e-2), relative to the row scale max(|const_term| + sum |terms|, 1), and z within the tier's z bound; additive
    blocks exactly 0.0."""
    _, fp = flows(O, P, name)
    cs = stack_of(fp, tier)
    assert cs.single_kernel == (name in SINGLE and tier == "fp32"), name
    x, ctx = inputs(fp)
    xin = G.rows_in(x, ctx)
    lp, t, z, n = call_terms(K, cs, tier, xin)
    assert n == 1 if cs.single_kernel else n > 1
    ref_cs, ref_tier = (stack_of(fp, "fp32"), "fp32") if tier == "bf16" else (cs, tier)
    t_ref, z_ref = interp_terms(ref_cs, ref_tier, xin.double())
    scale = row_scale(cs, t_ref)
    et = ((t.double().cpu() - t_ref.cpu()).abs() / scale).amax(1)
    ez = G.row_err(z, z_ref)
    lp_tol = 1e-2 if tier == "bf16" else G.tol(G.LP_TOL, tier, name)
    z_tol = BF16_Z_TOL if tier == "bf16" else G.tol(G.Z_TOL, tier, name)
    print(f"[terms] {name} {tier} single={cs.single_kernel}: worst term row {float(et.max()):.2e} "
          f"(per row {[f'{float(e):.1e}' for e in et]}), z {float(ez.max()):.2e}")
    assert float(et.max()) <= lp_tol, (name, tier, et)
    assert float(ez.max()) <= z_tol, (name, tier, float(ez.max()))
    for j in range(cs.desc.n_blocks):
        if not cs.blocks[j].affine:
            assert bool((t[j] == 0).all()), (name, j)
    gap, bound = recombined_gap(cs, lp, t)
    assert bool((gap <= bound).all()), (name, tier, float((gap / bound).max()))


# ------------------------------------------------------------------------------------------------------------------
# 2. identities
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["fp32", "bf16x2", "tf32x3", "bf16"])
def test_chain_logprob_and_z_identity(K, O, P, tier):
    """Launch chain: out_logprob and z are usf_stack_run's in deterministic mode bit for bit (with the library's mode
    off or on around the terms call), and the rows recombine to log p within 64 eps of the row scale."""
    _, fp = flows(O, P, "C2")
    cs = stack_of(fp, tier)
    assert not cs.single_kernel
    x, _ = inputs(fp)
    xin = G.rows_in(x, None)
    lq, zq = G.call_run(K, cs, tier, xin, deterministic=True) if tier != "bf16" else _run_bf16(K, cs, xin)
    for det in (False, True):
        lp, t, z, _ = call_terms(K, cs, tier, xin, deterministic=det)
        assert torch.equal(lp, lq), float(G.lp_err(lp, lq).max())
        assert torch.equal(z, zq)
        gap, bound = recombined_gap(cs, lp, t)
        print(f"[recombine] C2 {tier}: worst gap / bound {float((gap / bound).max()):.3f}")
        assert bool((gap <= bound).all())


def _run_bf16(K, cs, xin):
    """usf_stack_run at the bf16 tier, deterministic (G.call_run's tier table has no bf16 entry)."""
    lib = K.lib()
    B, D = xin.shape[0], cs.D
    lp = torch.empty(B, device="cuda")
    z = torch.empty(B, D, device="cuda")
    prev = lib.usf_set_deterministic(1)
    try:
        nbytes = lib.usf_stack_workspace_bytes(C.byref(cs.desc), B, K.USF_PREC_BF16)
        ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        K.check(lib.usf_stack_run(C.byref(cs.desc), C.c_void_p(xin.data_ptr()), xin.shape[1], B, C.c_void_p(lp.data_ptr()),
                                  C.c_void_p(z.data_ptr()), D, None, C.c_void_p(ws.data_ptr()), nbytes, K.USF_PREC_BF16,
                                  None, K.stream()), "usf_stack_run")
        torch.cuda.synchronize()
    finally:
        lib.usf_set_deterministic(prev)
    return lp, z


@pytest.mark.parametrize("name", ["C1-D2", "C4-D6", "C4-D64", "fixture-D32", "cond20"])
def test_single_kernel_identities(K, O, P, name):
    """One-kernel path, in either library mode: out_logprob and z are usf_stack_run's bit for bit, and
    const_term + row 0 + ... + row n_blocks added in that order in fp32 is out_logprob bit for bit."""
    _, fp = flows(O, P, name)
    cs = stack_of(fp, "fp32")
    assert cs.single_kernel
    x, ctx = inputs(fp)
    xin = G.rows_in(x, ctx)
    for det in (False, True):
        lq, zq = G.call_run(K, cs, "fp32", xin, deterministic=det)
        lp, t, z, n = call_terms(K, cs, "fp32", xin, deterministic=det)
        assert n == 1
        assert torch.equal(lp, lq) and torch.equal(z, zq)
        acc = torch.full_like(lp, float(cs.desc.const_term))
        for row in t:
            acc = acc + row
        assert torch.equal(acc, lp), float((acc - lp).abs().max())


@pytest.mark.parametrize("name,tier", [("cond200", "bf16x2"), ("C4-D6", "fp32")])
def test_run_to_run_and_split(K, O, P, name, tier):
    """Bit-identical run to run, and one call of 131072 + 77 rows (two chunks of the chain) equals two calls split at
    the chunk boundary."""
    _, fp = flows(O, P, name)
    cs = stack_of(fp, tier)
    B = CHUNK + 77
    x, ctx = inputs(fp, B=B, seed=11)
    xin = G.rows_in(x, ctx)
    lp, t, z, _ = call_terms(K, cs, tier, xin)
    lp2, t2, z2, _ = call_terms(K, cs, tier, xin, ws_off=0)
    assert torch.equal(lp, lp2) and torch.equal(t, t2) and torch.equal(z, z2)
    la, ta, za, _ = call_terms(K, cs, tier, xin[:CHUNK])
    lb, tb, zb, _ = call_terms(K, cs, tier, xin[CHUNK:])
    assert torch.equal(lp, torch.cat([la, lb])) and torch.equal(t, torch.cat([ta, tb], 1)) and \
        torch.equal(z, torch.cat([za, zb]))


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
def test_workspace_and_empty_batch(K, O, P, tier):
    """Exactly the queried bytes at misaligned pointers succeed; one byte short returns USF_E_WORKSPACE and writes
    nothing (also on the one-kernel path); B = 0 returns OK and writes nothing."""
    for name in ("cond200", "C4-D6"):
        _, fp = flows(O, P, name)
        cs = stack_of(fp, tier if name == "cond200" else "fp32")
        x, ctx = inputs(fp, B=40)
        xin = G.rows_in(x, ctx)
        for off in (0, 3, 255):
            call_terms(K, cs, tier if name == "cond200" else "fp32", xin, ws_off=off)
        call_terms(K, cs, tier if name == "cond200" else "fp32", xin, short=1, expect=-3)
        call_terms(K, cs, tier if name == "cond200" else "fp32", xin[:0])


# ------------------------------------------------------------------------------------------------------------------
# 3. Flow.log_prob_terms against the fp64 oracle
# ------------------------------------------------------------------------------------------------------------------
def _is_coupling(layer):
    return hasattr(layer, "mask") and hasattr(layer, "conditioner")


def oracle_terms(fo, x, ctx=None):
    """fp64 (couplings (B, K) in layer order, base log p at the oracle's z, affine, log p) of the oracle flow, walked
    as its log_prob walks it."""
    context = fo._soft_context(x, ctx)
    y, coup, aff = x, [], 0.0
    for layer in reversed(fo.layers):
        xin = layer.backward(y) if context is None else layer.backward(y, context)
        ladj = layer.log_abs_det_jacobian(xin, y) if context is None else layer.log_abs_det_jacobian(xin, y, context)
        if _is_coupling(layer):
            coup.append(-torch.as_tensor(ladj, dtype=torch.float64).expand(x.shape[0]))
        else:
            aff = aff - ladj
        y = xin
    base = fo._event_base.log_prob(y)
    lp = fo.log_prob(x) if ctx is None else fo.log_prob(x, ctx)
    return torch.stack(coup[::-1], 1), base, torch.as_tensor(aff, dtype=torch.float64), lp


def _check_against_oracle(fo, fp, x, ctx, what):
    with torch.no_grad():
        c_ref, b_ref, a_ref, lp_ref = oracle_terms(fo, x.double(), None if ctx is None else ctx.double())
        t = fp.log_prob_terms(x.cuda(), None if ctx is None else ctx.cuda())
        lq = fp.log_prob(x.cuda(), None if ctx is None else ctx.cuda())
    B = x.shape[0]
    assert t.couplings.shape == c_ref.shape and t.base.shape == (B,) and t.log_prob.shape == (B,)
    assert t.affine.shape == () and t.z.shape == x.shape
    scale = lp_ref.abs().clamp_min(1.0)
    ec = float(((t.couplings.double().cpu() - c_ref).abs().amax(1) / scale).max())
    eb = float(((t.base.double().cpu() - b_ref).abs() / scale).max())
    ea = abs(float(t.affine) - float(a_ref)) / max(abs(float(a_ref)), 1.0)
    el = float(((t.log_prob.double().cpu() - lp_ref).abs() / scale).max())
    print(f"[oracle] {what} ({fp.effective_precision}, {fp.last_launches} launches): couplings {ec:.2e}, base {eb:.2e}, "
          f"affine {ea:.2e}, log p {el:.2e}")
    for e in (ec, eb, ea, el):
        assert e <= 1e-4, what
    lq = lq.cpu()
    gap = (lq.double() - (t.base.double().cpu() + t.couplings.double().cpu().sum(1) + float(t.affine))).abs()
    bound = 64 * EPS32 * (abs(float(t.affine)) + t.base.double().abs().cpu() + t.couplings.double().abs().cpu().sum(1))
    assert bool((gap <= bound.clamp_min(64 * EPS32)).all()), (what, float((gap / bound).max()))
    return t


@pytest.mark.parametrize("name", ["C2", "C4-D6"])
def test_flow_terms_against_oracle_auto(O, P, name):
    """C2 "auto" (bf16x2 chain) and C4 D = 6 "auto" (one kernel): per-coupling terms in layer order, base log p at the
    oracle's z and the affine constant within the log p bound of test_full_depth_against_oracle (1e-4); the terms
    recombine to log_prob; in deterministic mode terms.log_prob is log_prob and terms.z is backward, bit for bit."""
    fo, fp = flows(O, P, name)
    fp.precision = "auto"
    x, _ = inputs(fp)
    t = _check_against_oracle(fo, fp, x, None, name)
    assert fp.effective_precision == ("bf16x2" if name == "C2" else "fp32")
    assert fp.last_launches == 1 if name == "C4-D6" else fp.last_launches > 1
    prev, fp.deterministic = fp.deterministic, True
    try:
        with torch.no_grad():
            t2 = fp.log_prob_terms(x.cuda())
            lq = fp.log_prob(x.cuda())
            zq = fp.backward(x.cuda())
    finally:
        fp.deterministic = prev
    assert torch.equal(t2.log_prob, lq) and torch.equal(t2.z, zq)
    assert torch.equal(t2.couplings, t.couplings) and torch.equal(t2.base, t.base)


def test_flow_terms_conditional(O, P):
    """A conditional flow with a context; a soft-training flow scored without one; the conditional flow without a
    context raises log_prob's ValueError, a CPU tensor USFError."""
    fo, fp = flows(O, P, "cond20")
    x, ctx = inputs(fp)
    _check_against_oracle(fo, fp, x, ctx, "cond20 with context")
    with pytest.raises(ValueError):
        fp.log_prob_terms(x.cuda())
    from nf4ad_b200._lib import USFError
    with pytest.raises(USFError):
        fp.log_prob_terms(x, ctx)
    torch.manual_seed(21)
    kw = dict(affine_conjugation=True, prior_scale=1.0, soft_training=True)
    fo = build_flow(O, "NonUSFlow", 16, 3, ("cond2", [32]), **kw)
    tame(fo, 0.25)
    randomize_constants(fo, 21)
    fp = build_flow(P, "NonUSFlow", 16, 3, ("cond2", [32]), **kw)
    fp.load_state_dict(fo.state_dict())
    fo, fp = fo.double(), fp.to("cuda").eval()
    _check_against_oracle(fo, fp, torch.randn(128, 16, generator=torch.Generator().manual_seed(3)), None, "soft, no context")


def _r2_pair(O, P, name):
    case = load_golden_r2(name)
    fo, fp = flow_from_r2_case(O, case["case"]), flow_from_r2_case(P, case["case"])
    fo.load_state_dict({k: v.double() for k, v in case["state_dict"].items()})
    fp.load_state_dict({k: v.float() for k, v in case["state_dict"].items()})
    return fo.double(), fp.to("cuda").eval(), case["x"].float()


def test_flow_terms_layerwise_route(O, P):
    """Flows without a fused stack -- an image-shaped event, a softplus scale, an opaque (Tanh) conditioner -- collect
    the terms from the layer-wise pass; terms.log_prob is log_prob's there."""
    pairs = [_r2_pair(O, P, n) for n in ("nonus_img_c3_4x4_k3_channel_laplace", "nonus_d8_k2_softplus")]
    torch.manual_seed(3)
    fo = build_flow(O, "NonUSFlow", 8, 2, ("mlp", [16]), affine_conjugation=True)
    fp = build_flow(P, "NonUSFlow", 8, 2, ("mlp", [16]), affine_conjugation=True)
    fp.load_state_dict(fo.state_dict())
    for f in (fo, fp):
        for layer in f.layers:
            net = getattr(getattr(layer, "conditioner", None), "net", None)
            if net is not None:
                net[1] = torch.nn.Tanh()
    pairs.append((fo.double(), fp.to("cuda").eval(), torch.randn(64, 8, generator=torch.Generator().manual_seed(4))))
    for fo, fp, x in pairs:
        assert fp._stack(True, "cuda", "fp32") is None
        t = _check_against_oracle(fo, fp, x, None, type(fp).__name__ + str(tuple(x.shape[1:])))
        with torch.no_grad():
            assert torch.equal(t.log_prob, fp.log_prob(x.cuda()))
        assert t.log_prob.grad_fn is None and t.couplings.grad_fn is None


# ------------------------------------------------------------------------------------------------------------------
# 4. ADBenchFlow.score_terms
# ------------------------------------------------------------------------------------------------------------------
def test_adbench_score_terms(O, P):
    """Shapes and score sign; the parts add up to predict_score within identity 5's bound; column k is the k-th
    coupling of flow.layers (a coupling whose conditioner outputs zeros contributes exactly 0 in its own column)."""
    from nf4ad_b200.adbench import ADBenchFlow
    torch.manual_seed(9)
    flow = build_flow(P, "NonUSFlow", 20, 3, ("mlp", [32]), affine_conjugation=True, prior_scale=1.0)
    tame(flow, 0.25)
    couplings = [l for l in flow.layers if _is_coupling(l)]
    with torch.no_grad():
        last = couplings[1].conditioner.net[-1]
        last.weight.zero_()
        last.bias.zero_()
    model = ADBenchFlow(flow, device="cuda", verbose=False)
    X = np.random.default_rng(1).standard_normal((1000, 20)).astype(np.float32)
    st = model.score_terms(X, chunk_rows=300)
    assert st["score"].shape == (1000,) and st["base"].shape == (1000,) and st["couplings"].shape == (1000, 3)
    assert isinstance(st["affine"], float)
    assert np.all(st["couplings"][:, 1] == 0) and np.all(st["couplings"][:, [0, 2]] != 0)
    ps = model.predict_score(X).astype(np.float64)
    parts = st["base"].astype(np.float64) + st["couplings"].astype(np.float64).sum(1) + st["affine"]
    bound = 64 * EPS32 * (abs(st["affine"]) + np.abs(st["base"]) + np.abs(st["couplings"]).sum(1))
    assert np.all(np.abs(ps - parts) <= bound), float(np.max(np.abs(ps - parts) / bound))
    with torch.no_grad():
        t = flow.log_prob_terms(torch.from_numpy(X[:300]).cuda())
    assert np.array_equal(st["score"][:300], (-t.log_prob).cpu().numpy())
    assert np.array_equal(st["couplings"][:300], (-t.couplings).cpu().numpy())
