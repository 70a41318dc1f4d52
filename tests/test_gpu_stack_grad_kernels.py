"""GPU parity of the fused input-gradient chain (`usf_stack_log_prob_grad`, csrc/usf_grad.cu) and of the forward chain
(`usf_stack_run`) against an fp64 interpreter of the PACKED descriptor they run.

The interpreter (`interpret`) evaluates an inverse-direction `usf_stack_desc` in float64 from the very device tensors its
descriptors point at (found in `CompiledStack._keep` by data pointer).  Per tier it multiplies the effective weights the
kernels multiply: fp32 `W`; tf32x3 and bf16x2 the sum of the high and low rows (exact in fp64).  So what it measures is
the kernels' arithmetic error alone, not the error of packing the weights (the fp32 run matrices of the affine layers).
Its gradient is `torch.autograd.grad` of its log p.  It is anchored to the fp64 oracle flow on every case
(`test_interpreter_matches_oracle`), so a wrong interpreter cannot agree with a wrong kernel.

Harness rules, as in test_gpu_backward_kernels.py:
  * x sits in a buffer with ldx > D + ctx_dim, NaN pad columns and a NaN row below;
  * out_grad has ldg > D and a row below, holding a sentinel that must come back bit-identical; out_logprob has a
    sentinel element behind it; both start as NaN inside, so every element must be written;
  * the workspace is filled with NaN (0xFF bytes: NaN as fp32 and as bf16) before every call and passed misaligned by
    3 bytes with exactly `usf_stack_grad_workspace_bytes` bytes (the 256-byte alignment slack); bytes past it must be
    unchanged.

Gradient rows are compared relative to the row's max-abs value, on the rows whose fp64 ReLU margin (smallest |hidden
pre-activation| of the pass) is above MARGIN[tier]: a unit closer to its kink than the kernels' activation error may
land on the other side of it, and then the row takes the other branch of a discontinuous gradient.  At least
MIN_QUALIFIED[tier] of the rows must qualify; the others are only required to be finite.

Measured on an NVIDIA B200 at a 1000 W power limit, 256 rows per case (largest error over the cases, bound in brackets):
  * gradient, qualifying rows: fp32 7.3e-6 on C2 and 1.5e-5 on the D = 40 stack without hidden layers [3e-5]; bf16x2
    1.4e-4 on C2 [3e-4], 2.6e-4 and 2.9e-4 on the two ILL_CONDITIONED stacks [3e-3].
  * rows that left the bound took the other side of a kink: the largest fp64 margin among them was 1.4e-6 at fp32 and
    2.5e-5 at bf16x2, hence MARGIN = 1e-5 and 5e-5.  At those margins C3 (6600 ReLU units per row) keeps 34 % of its rows
    at bf16x2 and 82 % at fp32, the other cases 73 % .. 100 %.
  * log p: fp32 1.5e-5 [3e-5]; tf32x3 1.0e-4 (C2) [2e-4]; bf16x2 5.9e-5 (C2) [1e-4], 3.2e-4 ILL_CONDITIONED [1e-3].
  * z: fp32 8.6e-6 [3e-5]; tf32x3 1.1e-4 (C2) [3e-4]; bf16x2 7.9e-5 (C2) [2e-4], 3.1e-4 ILL_CONDITIONED [2e-3].
  * the interpreter against the oracle (the packing error): gradient median 2.5e-6 or less and log p 9.2e-6 or less on
    every case; single rows reach 4.3e-4 (C1) and 2.6e-3 (D = 1) where the packing moves a row across a kink or a
    near-zero row.
The file runs in about 10 s on the B200.
"""
import ctypes as C
import math

import pytest
import torch

from _cases import build_flow, randomize_constants, tame

pytestmark = pytest.mark.gpu

NAN = float("nan")
SENTINEL = -12345.5          # exactly representable: bit comparisons are meaningful
CHUNK = 16384                # rows per pass of the gradient chain (csrc/usf_grad.cu kGradChunkRows)
ROWS = 256

GRAD_TOL = {"fp32": 3e-5, "bf16x2": 3e-4}        # per qualifying row, relative to the row's max |g|
MARGIN = {"fp32": 1e-5, "bf16x2": 5e-5}          # |ReLU pre-activation| a row needs to qualify
MIN_QUALIFIED = {"fp32": 0.6, "bf16x2": 0.3}
LP_TOL = {"fp32": 3e-5, "tf32x3": 2e-4, "bf16x2": 1e-4}   # log p, relative to max(|log p|, 1)
Z_TOL = {"fp32": 3e-5, "tf32x3": 3e-4, "bf16x2": 2e-4}    # latent z per row, relative to the row's max |z|
# stacks whose affine runs amplify operand rounding most (their fp32 packing error in log p is 7e-6 .. 9e-6, ten times
# the other cases'): the tensor-core tiers get ten times the bounds there
ILL_CONDITIONED = ("nohid40", "cond16")


def tol(table, tier, name):
    return table[tier] * (10 if tier != "fp32" and name in ILL_CONDITIONED else 1)


CASES = {
    # name: kind, D, K, conditioner, base, gain, kwargs
    "C2": ("NonUSFlow", 784, 8, ("mlp", [256, 256]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "C3": ("NonUSFlow", 784, 11, ("mlp", [200, 200, 200]), "laplace", 0.25, dict(affine_conjugation=True, householder=0)),
    "C1": ("USFlow", 128, 10, ("densenn1", [128, 128]), "usnormal", 0.5,
           dict(affine_conjugation=True, householder=0, prior_scale=1.0)),
    "add130": ("NonUSFlow", 130, 3, ("mlp_add", [64]), "normal", 0.25, dict(affine_conjugation=True)),     # ragged last tile
    "nohid40": ("NonUSFlow", 40, 3, ("mlp", []), "normal", 0.25, dict(affine_conjugation=True)),           # n_mlp == 1
    "deep24": ("NonUSFlow", 24, 2, ("mlp", [32] * 7), "laplace", 0.25, dict(affine_conjugation=True)),     # n_mlp == 8
    "D1": ("NonUSFlow", 1, 1, ("mlp", [8]), "normal", 0.25, dict(affine_conjugation=True)),                # Da == 0
    "D3": ("NonUSFlow", 3, 2, ("mlp", [8]), "laplace", 0.25, dict(affine_conjugation=True)),
    "cond16": ("NonUSFlow", 16, 3, ("cond2", [32]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "cond200": ("NonUSFlow", 200, 2, ("cond2", [64]), "normal", 0.25, dict(affine_conjugation=True, prior_scale=1.0)),
    "D1040": ("NonUSFlow", 1040, 1, ("mlp", [64]), "normal", 0.25, dict(affine_conjugation=True)),       # bf16x2 refused
}
NAMES = list(CASES)


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
    """(fp64 oracle flow, product flow on cuda) of a case, built once per module."""
    if name not in _FLOWS:
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


def inputs(name, B=ROWS, seed=5):
    """(x (B, D), context (B, 1) or None) on the CPU."""
    D, cond = CASES[name][1], CASES[name][3]
    x = torch.randn(B, D, generator=torch.Generator().manual_seed(seed))
    ctx = torch.rand(B, 1, generator=torch.Generator().manual_seed(seed + 1)) * 0.2 if cond[0] == "cond2" else None
    return x, ctx


def rows_in(x, ctx):
    return (x if ctx is None else torch.cat([x, ctx], 1)).float().cuda()


def prec(K, tier):
    return {"fp32": K.USF_PREC_FP32, "tf32x3": K.USF_PREC_TF32X3, "bf16x2": K.USF_PREC_BF16X2}[tier]


# ------------------------------------------------------------------------------------------------------------------
# the fp64 interpreter of a packed inverse-direction stack
# ------------------------------------------------------------------------------------------------------------------
def _keep(cs):
    return {t.data_ptr(): t for t in cs._keep}


def _rows_of(t, n, ldw, start=0):
    return t.reshape(-1)[start * ldw:(start + n) * ldw].view(n, ldw)


def weights(cs, L, tier):
    """(W (N, K), bias (N) or None) in fp64: exactly the matrix the kernels of `tier` multiply."""
    m = _keep(cs)
    N, Kd, ldw = L.N, L.K, L.ldw
    if tier == "fp32":
        W = _rows_of(m[L.W], N, ldw)[:, :Kd].double()
    else:
        t = m[L.W] if tier == "tf32x3" else m[L.Wb]
        W = _rows_of(t, N, ldw)[:, :Kd].double() + _rows_of(t, N, ldw, N)[:, :Kd].double()     # hi + lo, exact in fp64
    b = m[L.bias].reshape(-1)[:N].double() if L.bias else None
    return W, b


class Interp:
    pass


def interpret(cs, tier, x):
    """fp64 pass of x (B, D + ctx_dim) through the packed stack: .lp (log p), .ladj (the coupling log-det terms),
    .z (latent, (B, D)) and .margin (per row, the smallest |pre-activation| of any real ReLU unit; inf if none)."""
    st, m = cs.desc, _keep(cs)
    D, B = st.D, x.shape[0]
    act = x
    ladj = torch.zeros(B, dtype=torch.float64, device=x.device)
    margin = torch.full((B,), math.inf, dtype=torch.float64, device=x.device)
    for j in range(st.n_blocks):
        blk = cs.blocks[j]
        W, b = weights(cs, blk.G, tier)
        u = act[:, :blk.G.K] @ W.t() + b                       # [a | ctx | pad | b] layout, G.N columns
        h = u[:, :blk.mlp[0].K]
        for l in range(blk.n_mlp - 1):
            W, b = weights(cs, blk.mlp[l], tier)
            pre = h[:, :W.shape[1]] @ W.t() + b                # (the padded units of h are not read)
            real = cs._mlp_widths[j][l]                        # the padded units are constant 0
            margin = torch.minimum(margin, pre[:, :real].detach().abs().amin(1))
            h = torch.relu(pre)
        W, b = weights(cs, blk.mlp[blk.n_mlp - 1], tier)
        p = h[:, :W.shape[1]] @ W.t() + b                      # per tile [s(C) | t(C)], or [t(C)] when additive
        Cc, Db, bo = blk.C, blk.Db, blk.b_off
        q = torch.arange(Db, device=x.device)
        tile, w = q // Cc, q % Cc
        ub = u[:, bo:bo + Db]
        if blk.affine:
            s, t = p[:, tile * 2 * Cc + w], p[:, tile * 2 * Cc + Cc + w]
            ls = blk.clamp * torch.tanh(s)
            xb = (ub - t) * torch.exp(-ls)
            ladj = ladj - ls.sum(1)
        else:
            xb = ub - p[:, tile * Cc + w]
        act = torch.cat([u[:, :bo], xb, u[:, bo + Db:]], 1)
    W, b = weights(cs, st.G_final, tier)
    z = act[:, :st.G_final.K] @ W[:D].t() + b[:D]
    loc = m[st.loc].reshape(-1)[:D].double()
    inv = m[st.inv_scale].reshape(-1)[:D].double()
    d = (z - loc) * inv
    base = (-0.5 * d * d).sum(1) if st.base_kind == 0 else (-d.abs()).sum(1)
    r = Interp()
    r.z, r.ladj, r.margin = z, ladj, margin
    r.lp = float(st.const_term) + ladj + base
    r.loc, r.inv = loc, inv
    return r


def ref_grad(cs, tier, xin, ties=None):
    """fp64 (log p, d log p / dx (B, D), ReLU margin) of the packed stack.  `ties`: a (B, D) bool mask of z == loc
    entries, where the Laplace base gradient is sign(0) = 0."""
    xd = xin.double().clone().requires_grad_(True)
    r = interpret(cs, tier, xd)
    if ties is None:
        obj = r.lp.sum()
    else:
        gz = -torch.sign(r.z.detach() - r.loc) * r.inv
        gz[ties] = 0.0
        obj = r.ladj.sum() + (r.z * gz).sum()
    g, = torch.autograd.grad(obj, xd)
    return r.lp.detach(), g[:, :cs.D], r.margin


def row_err(got, ref):
    """Max error of each row relative to the row's max |ref|, but to no less than half the median row scale: a row
    whose values nearly cancel to 0 (D = 1) measures the cancellation, not the kernel."""
    got, ref = got.double().cpu(), ref.double().cpu()
    scale = ref.abs().amax(1)
    return (got - ref).abs().amax(1) / scale.clamp_min(0.5 * float(scale.median())).clamp_min(1e-30)


def lp_err(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return (got - ref).abs() / ref.abs().clamp_min(1.0)


def assert_grad_rows(name, tier, g, g_ref, margin, min_qualified=None):
    """Per-row check on the rows whose ReLU margin clears MARGIN[tier]; the rest only finite."""
    bound = tol(GRAD_TOL, tier, name)
    min_qualified = MIN_QUALIFIED[tier] if min_qualified is None else min_qualified
    assert bool(torch.isfinite(g).all()), (name, tier, "non-finite gradient")
    e = row_err(g, g_ref)
    ok = margin.cpu() > MARGIN[tier]
    frac = float(ok.double().mean())
    worst = float(e[ok].max()) if bool(ok.any()) else 0.0
    flips = e > bound
    print(f"[grad] {name} {tier}: qualified {frac:.2f}, max row err {worst:.2e}, median {float(e.median()):.2e}, "
          f"excluded max {float(e[~ok].max()) if bool((~ok).any()) else 0.0:.2e}, rows beyond tol {int(flips.sum())} "
          f"with margins up to {float(margin.cpu()[flips].max()) if bool(flips.any()) else 0.0:.2e}")
    assert frac >= min_qualified, (name, tier, frac)
    assert worst <= bound, (name, tier, worst, e[ok].topk(min(5, int(ok.sum()))))


# ------------------------------------------------------------------------------------------------------------------
# the C ABI calls, with the hostile harness
# ------------------------------------------------------------------------------------------------------------------
def _ws(nbytes, off):
    """A NaN-filled workspace and the misaligned pointer into it."""
    buf = torch.full((nbytes + off + 512,), 0xFF, dtype=torch.uint8, device="cuda")
    return buf, C.c_void_p(buf.data_ptr() + off)


def _ws_untouched(buf, nbytes, off):
    return bool((buf[:off] == 0xFF).all()) and bool((buf[off + nbytes:] == 0xFF).all())


def call_grad(K, cs, tier, xin, deterministic=False, ws_off=3, short=0, expect=0):
    """usf_stack_log_prob_grad on xin (B, D + ctx) -> (log p (B,), gradient (B, D), launches); checks everything outside
    the outputs.  `short`: bytes fewer than the workspace query; `expect`: the return code."""
    lib = K.lib()
    D, din, B = cs.D, cs.D + cs.ctx_dim, xin.shape[0]
    ldx, ldg = din + 5, D + 3
    xb = torch.full((B + 1, ldx), NAN, dtype=torch.float32, device="cuda")
    xb[:B, :din] = xin
    gb = torch.full((B + 1, ldg), SENTINEL, dtype=torch.float32, device="cuda")
    gb[:B, :D] = NAN
    lb = torch.full((B + 1,), SENTINEL, dtype=torch.float32, device="cuda")
    lb[:B] = NAN
    g0, l0 = gb.clone(), lb.clone()
    prev = lib.usf_set_deterministic(int(deterministic))
    try:
        nbytes = lib.usf_stack_grad_workspace_bytes(C.byref(cs.desc), C.byref(cs.grad_desc), B, prec(K, tier))
        assert nbytes > 0, lib.usf_last_error()
        buf, wp = _ws(nbytes, ws_off)
        n = C.c_int(-1)
        rc = lib.usf_stack_log_prob_grad(C.byref(cs.desc), C.byref(cs.grad_desc), C.c_void_p(xb.data_ptr()), ldx, B,
                                         C.c_void_p(lb.data_ptr()), C.c_void_p(gb.data_ptr()), ldg, wp, nbytes - short,
                                         prec(K, tier), C.byref(n), K.stream())
        torch.cuda.synchronize()
    finally:
        lib.usf_set_deterministic(prev)
    assert rc == expect, (rc, lib.usf_last_error())
    assert _ws_untouched(buf, nbytes, ws_off), "wrote outside the workspace"
    if rc != 0 or B == 0:
        assert torch.equal(gb.view(torch.int32), g0.view(torch.int32)) and torch.equal(lb.view(torch.int32),
                                                                                       l0.view(torch.int32))
        return None, None, n.value
    gi, g0i = gb.view(torch.int32), g0.view(torch.int32)
    assert torch.equal(gi[:B, D:], g0i[:B, D:]) and torch.equal(gi[B], g0i[B]), "wrote outside out_grad"
    assert lb[B].item() == SENTINEL, "wrote past out_logprob"
    lp, g = lb[:B].clone(), gb[:B, :D].clone()
    assert bool(torch.isfinite(lp).all()) and bool(torch.isfinite(g).all()), "an output element was not written"
    return lp, g, n.value


def call_run(K, cs, tier, xin, deterministic=False):
    """usf_stack_run -> (log p (B,), z (B, D)), with the same harness."""
    lib = K.lib()
    D, din, B = cs.D, cs.D + cs.ctx_dim, xin.shape[0]
    ldx, ldy = din + 5, D + 3
    xb = torch.full((B + 1, ldx), NAN, dtype=torch.float32, device="cuda")
    xb[:B, :din] = xin
    yb = torch.full((B + 1, ldy), SENTINEL, dtype=torch.float32, device="cuda")
    yb[:B, :D] = NAN
    lb = torch.full((B + 1,), SENTINEL, dtype=torch.float32, device="cuda")
    lb[:B] = NAN
    y0 = yb.clone()
    prev = lib.usf_set_deterministic(int(deterministic))
    try:
        nbytes = lib.usf_stack_workspace_bytes(C.byref(cs.desc), B, prec(K, tier))
        assert nbytes > 0, lib.usf_last_error()
        buf, wp = _ws(nbytes, 3)
        n = C.c_int(-1)
        K.check(lib.usf_stack_run(C.byref(cs.desc), C.c_void_p(xb.data_ptr()), ldx, B, C.c_void_p(lb.data_ptr()),
                                  C.c_void_p(yb.data_ptr()), ldy, None, wp, nbytes, prec(K, tier), C.byref(n), K.stream()),
                "usf_stack_run")
        torch.cuda.synchronize()
    finally:
        lib.usf_set_deterministic(prev)
    assert _ws_untouched(buf, nbytes, 3), "wrote outside the workspace"
    yi, y0i = yb.view(torch.int32), y0.view(torch.int32)
    assert torch.equal(yi[:B, D:], y0i[:B, D:]) and torch.equal(yi[B], y0i[B]), "wrote outside out_y"
    assert lb[B].item() == SENTINEL
    lp, z = lb[:B].clone(), yb[:B, :D].clone()
    assert bool(torch.isfinite(lp).all()) and bool(torch.isfinite(z).all()), "an output element was not written"
    return lp, z


def grad_stack(fp, tier):
    return fp._stack(True, "cuda", tier, grad=True)


# ------------------------------------------------------------------------------------------------------------------
# 1. the interpreter against the fp64 oracle: the packing error
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_interpreter_matches_oracle(O, P, name):
    """The interpreter on the fp32 packs against the oracle flow's log p and autograd gradient.  What differs is the
    packing error (fp32 run matrices of the affine layers); an interpreter that mis-read the layout would be off by
    O(1) on every row."""
    fo, fp = flows(O, P, name)
    x, ctx = inputs(name)
    cs = grad_stack(fp, "fp32")
    assert cs is not None, fp._unsupported_reason
    lp, g, margin = ref_grad(cs, "fp32", rows_in(x, ctx).double())
    xd = x.double().clone().requires_grad_(True)
    lo = fo.log_prob(xd) if ctx is None else fo.log_prob(xd, ctx.double())
    go, = torch.autograd.grad(lo.sum(), xd)
    e, el = row_err(g, go), lp_err(lp, lo.detach())
    print(f"[pack] {name}: log p {float(el.max()):.2e}, grad row err max {float(e.max()):.2e} "
          f"median {float(e.median()):.2e} 90% {float(e.quantile(0.9)):.2e}")
    assert float(el.max()) <= 1e-4
    assert float(e.median()) <= 1e-3 and float(e.quantile(0.9)) <= 2e-3


# ------------------------------------------------------------------------------------------------------------------
# 2. the transposed packs, bit for bit
# ------------------------------------------------------------------------------------------------------------------
def _pairs(cs):
    """(forward desc, transposed desc, what) for every matrix of the chain."""
    out = []
    for j in range(cs.desc.n_blocks):
        blk, gb = cs.blocks[j], cs.grad_blocks[j]
        out.append((blk.G, gb.G, f"block {j} G"))
        out += [(blk.mlp[l], gb.mlp[l], f"block {j} mlp {l}") for l in range(blk.n_mlp)]
    out.append((cs.desc.G_final, cs.grad_desc.G_final, "G_final"))
    return out


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
@pytest.mark.parametrize("name", NAMES)
def test_transposed_packs_bitwise(P, O, name, tier):
    """T.N = round_up(K, 16), T.K = T.ldw = N; rows below K hold the forward matrix transposed (fp32: W; bf16x2: hi and
    lo each), the padded rows are zero."""
    _, fp = flows(O, P, name)
    cs = grad_stack(fp, tier)
    if cs is None:
        assert name == "D1040" and tier == "bf16x2", fp._unsupported_reason
        return
    m = _keep(cs)
    for F, T, what in _pairs(cs):
        assert T.N == (F.K + 15) // 16 * 16 and T.K == F.N and T.ldw == F.N, what
        assert not T.bias, what
        parts = [(m[F.W], m[T.W], 0)] if tier == "fp32" else [(m[F.Wb], m[T.Wb], 0), (m[F.Wb], m[T.Wb], 1)]
        for f, t, half in parts:
            fw = _rows_of(f, F.N, F.ldw, half * F.N)[:, :F.K]
            tw = _rows_of(t, T.N, T.ldw, half * T.N)
            iv = torch.int32 if f.dtype == torch.float32 else torch.int16
            assert torch.equal(tw[:F.K].contiguous().view(iv), fw.t().contiguous().view(iv)), (what, half)
            assert bool((tw[F.K:] == 0).all()), (what, half, "padded rows not zero")



# ------------------------------------------------------------------------------------------------------------------
# 3. usf_stack_log_prob_grad through the C ABI
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
@pytest.mark.parametrize("name", NAMES)
def test_grad_chain_matches_interpreter(K, O, P, name, tier):
    """log p and every qualifying row of the gradient against the interpreter of the same packs."""
    _, fp = flows(O, P, name)
    cs = grad_stack(fp, tier)
    if cs is None:
        assert name == "D1040" and tier == "bf16x2", fp._unsupported_reason
        return
    x, ctx = inputs(name)
    xin = rows_in(x, ctx)
    lp, g, n = call_grad(K, cs, tier, xin)
    assert n > 0
    lp_ref, g_ref, margin = ref_grad(cs, tier, xin)
    el = lp_err(lp, lp_ref)
    print(f"[lp] {name} {tier}: {float(el.max()):.2e}")
    assert float(el.max()) <= tol(LP_TOL, tier, name), (name, tier, float(el.max()))
    assert_grad_rows(name, tier, g, g_ref, margin)


def test_bf16x2_refused_falls_back_to_fp32(K, O, P):
    """D = 1040: G_final.N > 1024, so the bf16x2 packs are refused; a "bf16x2" request runs the fp32 chain and matches
    its interpreter."""
    _, fp = flows(O, P, "D1040")
    assert grad_stack(fp, "bf16x2") is None and "1024" in fp._unsupported_reason
    x, _ = inputs("D1040")
    prev, fp.precision = fp.precision, "bf16x2"
    try:
        lp, g = fp.log_prob_and_grad(x.cuda())
    finally:
        fp.precision = prev
    assert fp.last_grad_precision == "fp32"
    lp_ref, g_ref, margin = ref_grad(grad_stack(fp, "fp32"), "fp32", x.cuda())
    assert float(lp_err(lp, lp_ref).max()) <= LP_TOL["fp32"]
    assert_grad_rows("D1040 via bf16x2", "fp32", g, g_ref, margin)


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
def test_workspace_and_empty_batch(K, O, P, tier):
    """Exactly the queried bytes at a misaligned pointer succeed (the other tests); one byte short returns
    USF_E_WORKSPACE and writes nothing; B = 0 returns OK and writes nothing."""
    _, fp = flows(O, P, "cond200")
    cs = grad_stack(fp, tier)
    x, ctx = inputs("cond200", B=40)
    xin = rows_in(x, ctx)
    for off in (0, 3, 255):
        call_grad(K, cs, tier, xin, ws_off=off)
    call_grad(K, cs, tier, xin, short=1, expect=-3)
    call_grad(K, cs, tier, xin[:0])


def test_laplace_ties(K, O, P):
    """z == loc exactly at a few (row, column) pairs: the Laplace base gradient there is sign(0) = 0.  The ties are
    set from the forward chain's own z (usf_stack_run out_y on the same descriptor, fp32, deterministic)."""
    _, fp = flows(O, P, "C3")
    cs = grad_stack(fp, "fp32")
    x, _ = inputs("C3", B=64)
    xin = rows_in(x, None)
    _, z = call_run(K, cs, "fp32", xin, deterministic=True)
    loc = _keep(cs)[cs.desc.loc]
    saved = loc.clone()
    ties = torch.zeros(64, cs.D, dtype=torch.bool)
    try:
        for r, c in ((0, 0), (5, 17), (9, 400), (33, 783), (63, 256)):
            loc[c] = z[r, c]
            ties[r, c] = True
        _, z2 = call_run(K, cs, "fp32", xin, deterministic=True)
        assert torch.equal(z2, z)
        lp, g, _ = call_grad(K, cs, "fp32", xin, deterministic=True)
        _, g_ref, margin = ref_grad(cs, "fp32", xin, ties=ties.cuda())
        _, g_sign, _ = ref_grad(cs, "fp32", xin)
    finally:
        loc.copy_(saved)
    # the tie rows differ from the sign(+-1) reference by a full column of the Jacobian
    tie_rows = ties.any(1)
    assert float(row_err(g_sign, g_ref)[tie_rows].min()) > 100 * GRAD_TOL["fp32"]
    assert_grad_rows("C3 ties", "fp32", g, g_ref, margin)
    e = row_err(g, g_ref)
    assert bool((e[tie_rows & (margin.cpu() > MARGIN["fp32"])] <= GRAD_TOL["fp32"]).all())


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
def test_chunks(K, O, P, tier):
    """More than one internal chunk of 16384 rows in one call, NaN workspace: bit-identical to chunk-by-chunk calls, and
    the rows either side of every chunk boundary match the interpreter."""
    _, fp = flows(O, P, "cond200")
    cs = grad_stack(fp, tier)
    for B in (CHUNK + 1, 2 * CHUNK + 3):
        x, ctx = inputs("cond200", B=B, seed=B)
        xin = rows_in(x, ctx)
        lp, g, _ = call_grad(K, cs, tier, xin, deterministic=True)
        for r0 in range(0, B, CHUNK):
            lpc, gc, _ = call_grad(K, cs, tier, xin[r0:r0 + CHUNK], deterministic=True)
            assert torch.equal(lpc, lp[r0:r0 + CHUNK]) and torch.equal(gc, g[r0:r0 + CHUNK]), (B, r0)
        pick = torch.tensor(sorted({r for r in (0, CHUNK - 1, CHUNK, 2 * CHUNK - 1, 2 * CHUNK, B - 1) if r < B}))
        lp_ref, g_ref, margin = ref_grad(cs, tier, xin[pick.cuda()])
        assert float(lp_err(lp[pick.cuda()], lp_ref).max()) <= LP_TOL[tier]
        assert_grad_rows(f"cond200 B={B} boundary rows", tier, g[pick.cuda()], g_ref, margin, min_qualified=0.0)


@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
@pytest.mark.parametrize("name", ["C2", "C1", "add130", "cond200"])
def test_logprob_identity(K, O, P, name, tier):
    """Deterministic mode: the gradient call's log p is bit-identical to usf_stack_run's on the same descriptor (the
    launch chain: D > 64)."""
    _, fp = flows(O, P, name)
    cs = grad_stack(fp, tier)
    x, ctx = inputs(name)
    xin = rows_in(x, ctx)
    lp, _, _ = call_grad(K, cs, tier, xin, deterministic=True)
    lq, _ = call_run(K, cs, tier, xin, deterministic=True)
    assert torch.equal(lp, lq), float(lp_err(lp, lq).max())


# ------------------------------------------------------------------------------------------------------------------
# 4. the forward chain on the same interpreter
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["fp32", "tf32x3", "bf16x2"])
@pytest.mark.parametrize("name", NAMES)
def test_forward_chain_matches_interpreter(K, O, P, name, tier):
    """usf_stack_run's log p and latent z per row (fp32 with D + ctx <= 64: the one-kernel path)."""
    _, fp = flows(O, P, name)
    cs = fp._stack(True, "cuda", tier)
    if cs is None:
        assert name == "D1040" and tier != "fp32", fp._unsupported_reason
        return
    x, ctx = inputs(name)
    xin = rows_in(x, ctx)
    lp, z = call_run(K, cs, tier, xin)
    r = interpret(cs, tier, xin.double())
    el, ez = lp_err(lp, r.lp), row_err(z, r.z)
    print(f"[fwd] {name} {tier} single={cs.single_kernel}: log p {float(el.max()):.2e}, z row err {float(ez.max()):.2e}")
    assert float(el.max()) <= tol(LP_TOL, tier, name), (name, tier, float(el.max()))
    assert float(ez.max()) <= tol(Z_TOL, tier, name), (name, tier, float(ez.max()))


# ------------------------------------------------------------------------------------------------------------------
# 5. kernel error against packing error on the production shapes
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["fp32", "bf16x2"])
@pytest.mark.parametrize("name", ["C1", "C2"])
def test_error_split(K, O, P, name, tier):
    """The chain's error against the fp64 oracle splits into kernel error (chain vs interpreter of its packs) and
    packing error (interpreter vs oracle).  On the rows whose margin clears the tier's threshold in both fp64 passes,
    the chain-vs-oracle error must be explained by the packs: at most the packing error plus the kernel bound."""
    fo, fp = flows(O, P, name)
    cs = grad_stack(fp, tier)
    x, ctx = inputs(name)
    xin = rows_in(x, ctx)
    lp, g, _ = call_grad(K, cs, tier, xin)
    lp_i, g_i, margin = ref_grad(cs, tier, xin)
    xd = x.double().clone().requires_grad_(True)
    lo = fo.log_prob(xd) if ctx is None else fo.log_prob(xd, ctx.double())
    go, = torch.autograd.grad(lo.sum(), xd)
    ok = margin.cpu() > MARGIN[tier]
    e_kern, e_pack, e_tot = row_err(g, g_i), row_err(g_i, go), row_err(g, go)
    print(f"[split] {name} {tier}: kernel max {float(e_kern[ok].max()):.2e} median {float(e_kern.median()):.2e} | "
          f"packing max {float(e_pack[ok].max()):.2e} median {float(e_pack.median()):.2e} | "
          f"total max {float(e_tot[ok].max()):.2e} median {float(e_tot.median()):.2e} | "
          f"log p kernel {float(lp_err(lp, lp_i).max()):.2e} packing {float(lp_err(lp_i, lo.detach()).max()):.2e} "
          f"| all-rows total max {float(e_tot.max()):.2e} kernel {float(e_kern.max()):.2e} packing {float(e_pack.max()):.2e}")
    # every row beyond the kernel bound is explained: a packing flip (the interpreter itself is off the oracle) or a
    # unit of the packed pass within MARGIN of its kink
    far = e_tot > GRAD_TOL[tier]
    assert bool(((e_pack[far] > GRAD_TOL[tier]) | ~ok[far]).all()), (e_tot[far], e_pack[far], margin.cpu()[far])
