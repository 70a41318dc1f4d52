"""GPU parity, kernel level: every C-ABI layer kernel against the fp64 CPU oracle on the same seeded
inputs.  Tolerances: fp32 kernels max-norm relative error <= 2e-5 (well inside the 1e-4 log_prob
tier); the tcgen05 bf16 GEMM is compared against an exact fp32 product of the bf16-rounded operands."""
import math
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def relerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from nf4ad_b200 import _lib, ops as _ops
    assert _lib.lib().usf_device_ok() == 1, "expected an sm_100 device"
    return _ops


@pytest.mark.parametrize("B,N,K,relu", [(5, 7, 3, False), (1, 1, 1, True), (300, 130, 70, True),
                                        (257, 64, 129, False), (1000, 784, 784, False), (129, 1568, 256, True)])
def test_linear_fp32(ops, B, N, K, relu):
    g = torch.Generator().manual_seed(B * 1000 + N)
    x = torch.randn(B, K, generator=g)
    W = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    ref = x.double() @ W.double().t() + b.double()
    ref = ref.clamp_min(0) if relu else ref
    y = ops.linear(x.cuda(), W.cuda(), b.cuda(), relu)
    assert relerr(y, ref) < 2e-5
    # strided input (leading dimension > K)
    xp = torch.zeros(B, K + 5)
    xp[:, :K] = x
    y2 = ops.linear(xp.cuda()[:, :K], W.cuda(), b.cuda(), relu)
    assert relerr(y2, ref) < 2e-5


@pytest.mark.parametrize("D", [1, 5, 32, 100, 257])
def test_lu_pack_apply_solve(ops, O, D):
    torch.manual_seed(D)
    lu = O.transforms.LUTransform(D, 1.0).double()
    with torch.no_grad():
        lu.U_raw.diagonal().copy_((0.6 + torch.rand(D, dtype=torch.float64)) *
                                  torch.where(torch.rand(D) < 0.3, -1.0, 1.0))
        lu.L_raw.add_(torch.randn(D, D, dtype=torch.float64).triu(0))   # junk in the unused triangles
        lu.U_raw.add_(torch.randn(D, D, dtype=torch.float64).tril(-1))  # (and L's diagonal) must be ignored
    x = torch.randn(77, D, dtype=torch.float64)
    with torch.no_grad():
        y_ref = lu.forward(x)
        x_ref = lu.backward(y_ref)
    L, U, b = (t.detach().float().cuda() for t in (lu.L_raw, lu.U_raw, lu.bias))
    W = ops.lu_pack(L, U)
    assert relerr(W, lu.weight) < 2e-5
    y = ops.linear(x.float().cuda(), W, b)
    assert relerr(y, y_ref) < 2e-5
    xs = ops.lu_solve(y_ref.float().cuda(), L, U, b)
    assert relerr(xs, x_ref) < 1e-4
    # transposed solve: (LU)^T g = r
    r = torch.randn(33, D, dtype=torch.float64)
    g_ref = torch.linalg.solve(lu.weight.detach().t(), r.t()).t()
    g = ops.lu_solve(r.float().cuda(), L, U, None, transpose=True)
    assert relerr(g, g_ref) < 1e-4


@pytest.mark.parametrize("D,nvs", [(6, 1), (33, 3), (784, 2)])
def test_householder_scale(ops, O, D, nvs):
    torch.manual_seed(D + nvs)
    hh = O.transforms.HouseholderTransform(D, nvs).double()
    x = torch.randn(41, D, dtype=torch.float64)
    V = hh.vk_householder.detach().float().cuda()
    with torch.no_grad():
        assert relerr(ops.householder(x.float().cuda(), V, False), hh.forward(x)) < 2e-5
        assert relerr(ops.householder(x.float().cuda(), V, True), hh.backward(x)) < 2e-5
    s = (torch.rand(D, dtype=torch.float64) + 0.5) * torch.where(torch.rand(D) < 0.5, -1.0, 1.0)
    assert relerr(ops.scale(x.float().cuda(), s.float().cuda(), False), x * s) < 1e-6
    assert relerr(ops.scale(x.float().cuda(), s.float().cuda(), True), x / s) < 1e-6


# D = 2600: more columns than the base density kernel stages in shared memory (2048)
@pytest.mark.parametrize("D,affine", [(7, True), (64, True), (785, True), (20, False), (2600, True)])
def test_coupling_and_base(ops, D, affine):
    torch.manual_seed(D)
    B = 37
    x = torch.randn(B, D, dtype=torch.float64)
    s = torch.randn(B, D, dtype=torch.float64) * 2
    t = torch.randn(B, D, dtype=torch.float64)
    m = (torch.arange(D) % 2).double()
    ls = 5.0 * torch.tanh(s) if affine else torch.zeros_like(s)
    for act in (0, 1):
        if act == 0 or not affine:       # the additive form has no scale: the activation does not apply
            sc, inv_sc, lsc = torch.exp(ls), torch.exp(-ls), ls
        else:                            # softplus, with the reference's literal 1e-6 / 1e-12
            sp = torch.nn.functional.softplus(ls)
            sc, lsc = sp + 1e-6, torch.log(sp + 1e-12)
            inv_sc = 1.0 / (sc + 1e-12)
        for inverse in (False, True):
            ref = x * m + (1 - m) * ((x - t) * inv_sc if inverse else x * sc + t)
            ladj_ref = ((1 - m) * lsc).sum(1)
            y, ladj = ops.coupling(x.float().cuda(), s.float().cuda() if affine else None, t.float().cuda(),
                                   m.float().cuda(), 5.0, inverse, act)
            assert relerr(y, ref) < 1e-5, (act, inverse)
            assert float((ladj.double().cpu() - ladj_ref).abs().max()) < 1e-4 * max(1.0, float(ladj_ref.abs().max()))
    loc = torch.randn(D, dtype=torch.float64)
    for kind, dist in ((0, torch.distributions.Normal), (1, torch.distributions.Laplace)):
        for scale in (torch.rand(D, dtype=torch.float64) + 0.5, torch.tensor([1.7], dtype=torch.float64)):
            ref = dist(loc, scale.expand(D)).log_prob(x).sum(1)
            out = ops.base_logprob(kind, x.float().cuda(), loc.float().cuda(), scale.float().cuda())
            assert relerr(out, ref) < 1e-5


@pytest.mark.parametrize("B,N,K,relu,f32out", [(128, 16, 16, False, True), (128, 256, 64, False, True),
                                               (300, 208, 104, True, False), (1000, 784, 784, False, False),
                                               (4096, 1568, 256, True, False), (77, 48, 392, False, True),
                                               (20000, 256, 392, True, False), (130, 64, 64, False, False),
                                               (513, 48, 128, False, False)])
def test_tcgen05_linear_bf16(ops, B, N, K, relu, f32out):
    """tcgen05 GEMM (TMA 128B swizzle, TMEM accumulators) vs exact fp32 product of the same bf16 operands, for ragged
    row counts and tiles narrower than 64 columns.  The output has a leading dimension wider than N inside a NaN
    sentinel: every element of [B, N] is written and nothing outside it."""
    from nf4ad_b200 import _lib
    from nf4ad_b200._lib import lib, ptr, stream
    g = torch.Generator().manual_seed(B + N + K)
    ldx, ldw = (K + 7) // 8 * 8, (K + 7) // 8 * 8
    x = torch.zeros(B, ldx)
    x[:, :K] = torch.randn(B, K, generator=g)
    W = torch.zeros(N, ldw)
    W[:, :K] = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    xb, Wb = x.cuda().bfloat16(), W.cuda().bfloat16()
    ref = xb.float().double().cpu()[:, :K] @ Wb.float().double().cpu()[:, :K].t() + b.double()
    ref = ref.clamp_min(0) if relu else ref
    out = torch.full((B + 3, N + 16), float("nan"), device="cuda", dtype=torch.float32 if f32out else torch.bfloat16)
    _lib.check(lib().usf_linear_bf16(ptr(xb), ldx, ptr(Wb), ldw, ptr(b.cuda()), int(relu), ptr(out), N + 16,
                                     0 if f32out else 1, B, N, K, stream()), "usf_linear_bf16")
    torch.cuda.synchronize()
    flag = C.c_int(0)
    _lib.check(lib().usf_debug_tc_timeout(C.byref(flag), 1))
    assert flag.value == 0, "a bounded mbarrier wait expired inside the tcgen05 GEMM"
    assert bool(torch.isnan(out[B:].float()).all()) and bool(torch.isnan(out[:, N:].float()).all())
    y = out[:B, :N]
    assert torch.isfinite(y.float()).all()
    tol = 1e-5 if f32out else 6e-3
    assert relerr(y.float(), ref) < tol


@pytest.mark.parametrize("B,N,relu,ld", [(8, 16, False, 0), (64, 784, True, 0), (257, 100, True, 0), (4096, 256, False, 0),
                                         (4096, 1568, True, 0), (130, 99, True, 0), (131, 99, True, 104), (70, 5, False, 8),
                                         (1000, 784, False, 800)])
def test_to_bf16_operand_pass(ops, B, N, relu, ld):
    """usf_to_bf16: bf16 row-major copy, bf16 transposed copy (both zero padded to a multiple of 8 columns) and
    fp32 column sums of the (ReLU-gated) input, in one pass -- bit-exact against torch's round-to-nearest-even.
    16-byte aligned rows take the vectorised kernel (64 x 64 tiles; `ld` > 0: a strided view whose width is not a multiple
    of 4), anything else the element-wise one."""
    g = torch.Generator().manual_seed(B + N)
    if ld:
        x = torch.randn(B, ld, generator=g).cuda()[:, :N]
        mask = torch.randn(B, ld, generator=g).cuda()[:, :N] if relu else None
    else:
        x = torch.randn(B, N, generator=g).cuda()
        mask = torch.randn(B, N, generator=g).cuda() if relu else None
    rows, tr, cs = ops.to_bf16(x, relu_mask=mask, want_rows=True, want_transposed=True, want_colsum=True)
    v = torch.where(mask > 0, x, torch.zeros_like(x)) if relu else x
    ref = v.to(torch.bfloat16)
    assert rows.shape == (B, (N + 7) // 8 * 8) and tr.shape == (N, (B + 7) // 8 * 8)
    assert torch.equal(rows[:, :N], ref) and torch.equal(tr[:, :B], ref.t())
    assert float(rows[:, N:].float().abs().sum()) == 0.0 and float(tr[:, B:].float().abs().sum()) == 0.0
    assert relerr(cs, v.double().sum(0)) < 1e-5


def test_linear_t3_autograd_function():
    """LinearT3Fn: forward, dgrad, wgrad and the bias gradient on the 3xTF32 GEMM against float64."""
    from nf4ad_b200 import ops
    g = torch.Generator().manual_seed(11)
    for (B, K, N, relu) in ((512, 64, 1568, False), (1000, 80, 48, True), (256, 784, 256, True)):
        x = torch.randn(B, K, generator=g).cuda().requires_grad_(True)
        W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda().requires_grad_(True)
        b = torch.randn(N, generator=g).cuda().requires_grad_(True)
        dy = torch.randn(B, N, generator=g).cuda()
        y = ops.LinearT3Fn.apply(x, W, b, relu)
        y.backward(dy)
        xd, Wd, bd = (t.detach().double().requires_grad_(True) for t in (x, W, b))
        pre = xd @ Wd.T + bd
        gate = (y.detach() > 0).double() if relu else 1.0          # the kernel's own gate (ties at rounding of zero)
        yd = pre * gate
        yd.backward(dy.double())
        for got, ref, name in ((y, yd, "y"), (x.grad, xd.grad, "dx"), (W.grad, Wd.grad, "dW"), (b.grad, bd.grad, "db")):
            err = float((got.detach().double() - ref.detach()).abs().max() / ref.detach().abs().max().clamp_min(1e-30))
            assert err < 2e-5, (B, K, N, relu, name, err)


@pytest.mark.parametrize("B,N,K", [(64, 256, 784), (4096, 784, 784), (256, 1568, 256)])
def test_linear_tc_autograd_function(ops, B, N, K):
    """LinearTCFn (bf16 tensor-core forward / dgrad / wgrad) against fp64 autograd of the same layer."""
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, K, generator=g).cuda().requires_grad_()
    W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda().requires_grad_()
    b = torch.randn(N, generator=g).cuda().requires_grad_()
    dy = torch.randn(B, N, generator=g).cuda()
    y = ops.LinearTCFn.apply(x, W, b, True)
    y.backward(dy)
    xr, Wr, br = (t.detach().double().cpu().requires_grad_() for t in (x, W, b))
    # same ReLU gate as the GPU result: pre-activations within bf16 rounding of zero may legitimately gate differently
    gate = (y.detach().cpu() > 0).double()
    yr = (xr @ Wr.t() + br) * gate
    yr.backward(dy.double().cpu())
    assert relerr(y, yr) < 2e-2
    for got, ref in ((x.grad, xr.grad), (W.grad, Wr.grad), (b.grad, br.grad)):
        assert relerr(got, ref) < 3e-2


@pytest.mark.parametrize("B,N,K,relu", [(300, 256, 392, True), (4096, 800, 784, False), (129, 208, 70, False)])
def test_tcgen05_linear_tf32x3(ops, B, N, K, relu):
    """3xTF32 GEMM (usf_linear_tf32x3): fp32 operands as hi + lo, three kind::tf32 MMAs per K step.  Against fp64:
    max-norm relative error <= 2e-5 (the fp32 SIMT GEMM sits at ~1e-6; a single-pass tf32 GEMM at ~1e-3)."""
    from nf4ad_b200._lib import lib, ptr, stream, check
    g = torch.Generator().manual_seed(B + N + K)
    ld = (K + 3) // 4 * 4
    x = torch.zeros(B, ld); x[:, :K] = torch.randn(B, K, generator=g); x = x.cuda()
    W = torch.zeros(N, ld); W[:, :K] = torch.randn(N, K, generator=g) / K ** 0.5; W = W.cuda()
    b = torch.randn(N, generator=g).cuda()
    xlo, Wlo = torch.empty_like(x), torch.empty_like(W)
    check(lib().usf_split_lo(ptr(x), ld, ptr(xlo), ld, B, ld, stream()))
    check(lib().usf_split_lo(ptr(W), ld, ptr(Wlo), ld, N, ld, stream()))
    y, ylo = torch.empty(B, N, device="cuda"), torch.empty(B, N, device="cuda")
    check(lib().usf_linear_tf32x3(ptr(x), ptr(xlo), ld, ptr(W), ptr(Wlo), ld, ptr(b), int(relu), ptr(y), ptr(ylo), N, B, N, K,
                                  stream()))
    torch.cuda.synchronize()
    flag = C.c_int(0)
    check(lib().usf_debug_tc_timeout(C.byref(flag), 1))
    assert flag.value == 0
    ref = x[:, :K].double().cpu() @ W[:, :K].double().cpu().t() + b.double().cpu()
    if relu:
        ref = ref.clamp_min(0)
    assert int(((y.view(torch.int32) & 8191) != 0).sum()) == 0          # hi part is tf32-exact
    assert relerr(y.double() + ylo.double(), ref) < 2e-5


def test_vae_latent_tail_kernels():
    """usf_vae_reparam / usf_recon_nll and their backward kernels against the reference's formulas
    (nf4ad/vaeflow.py:176-179, 203-224) in float64 autograd."""
    from nf4ad_b200 import vae
    g = torch.Generator().manual_seed(21)
    for (B, L, img) in ((16, 128, (1, 28, 28)), (3, 7, (5,)), (64, 256, (3, 32, 32))):
        mu = torch.randn(B, L, generator=g).cuda().requires_grad_()
        lv = (0.5 * torch.randn(B, L, generator=g)).cuda().requires_grad_()
        eps = torch.randn(B, L, generator=g).cuda()
        x = torch.randn(B, *img, generator=g).cuda().requires_grad_()
        xr = torch.randn(B, *img, generator=g).cuda().requires_grad_()
        wz = torch.randn(B, L, generator=g).cuda()
        wq, wn = torch.randn(B, generator=g).cuda(), torch.randn(B, generator=g).cuda()
        z, log_q = vae.reparameterize(mu, lv, eps)
        nll = vae.recon_nll(x, xr, 0.1)
        ((z * wz).sum() + (log_q * wq).sum() + (nll * wn).sum()).backward()
        mud, lvd, xd, xrd = (t.detach().double().requires_grad_() for t in (mu, lv, x, xr))
        std = torch.exp(0.5 * lvd)
        zd = mud + eps.double() * std
        lqd = torch.distributions.Normal(mud, std).log_prob(zd).view(B, -1).sum(1)
        D = x[0].numel()
        nlld = 0.5 * ((xd - xrd) ** 2).view(B, -1).sum(1) / 0.01 + 0.5 * D * math.log(2 * math.pi * 0.01)
        ((zd * wz.double()).sum() + (lqd * wq.double()).sum() + (nlld * wn.double()).sum()).backward()
        for got, ref, name in ((z, zd, "z"), (log_q, lqd, "log_q"), (nll, nlld, "nll"), (mu.grad, mud.grad, "dmu"),
                               (lv.grad, lvd.grad, "dlogvar"), (xr.grad, xrd.grad, "dx_recon"), (x.grad, xd.grad, "dx")):
            assert relerr(got, ref) < 2e-5, (B, L, name, relerr(got, ref))
    # log q evaluated through the reparameterised z has no gradient path to mu (z - mu = eps std): dmu == dz exactly
    mu = torch.randn(4, 8).cuda().requires_grad_()
    lv = torch.zeros(4, 8).cuda().requires_grad_()
    z, log_q = vae.reparameterize(mu, lv, torch.randn(4, 8).cuda())
    log_q.sum().backward()
    assert float(mu.grad.abs().max()) == 0.0 and torch.allclose(lv.grad, torch.full_like(lv.grad, -0.5))


def test_fused_adam_matches_torch_adam():
    """usf_adam_step through `FusedAdam` against torch.optim.Adam / AdamW on the same parameters and gradients: ragged
    sizes (more than one 32-tensor launch, unaligned views), weight decay in both forms, ten steps."""
    from nf4ad_b200.optim import FusedAdam
    g = torch.Generator().manual_seed(5)
    sizes = [1, 3, 17, 784 * 784, 8191, 8192, 8193, 256 * 784] + [7 * (i + 1) for i in range(40)]
    for decoupled, wd in ((False, 0.0), (False, 0.01), (True, 0.05)):
        ours = [torch.randn(n, generator=g).cuda().requires_grad_() for n in sizes]
        base = torch.randn(101, generator=g).cuda()
        ours.append(base[1:].detach().requires_grad_())           # 4-byte aligned only: scalar path
        theirs = [p.detach().clone().requires_grad_() for p in ours]
        a = FusedAdam(ours, lr=3e-3, betas=(0.9, 0.99), eps=1e-8, weight_decay=wd, decoupled=decoupled)
        cls = torch.optim.AdamW if decoupled else torch.optim.Adam
        b = cls(theirs, lr=3e-3, betas=(0.9, 0.99), eps=1e-8, weight_decay=wd)
        for it in range(10):
            for p, q in zip(ours, theirs):
                gr = torch.randn(p.shape, generator=g).cuda() * (1.0 + it)
                p.grad, q.grad = gr.clone(), gr.clone()
            a.step()
            b.step()
        for p, q in zip(ours, theirs):
            assert relerr(p, q) < 2e-6, (decoupled, wd, p.numel(), relerr(p, q))
    # the clipping coefficient folded into the update == gradients scaled beforehand
    p1 = torch.randn(1000, generator=g).cuda().requires_grad_()
    p2 = p1.detach().clone().requires_grad_()
    o1, o2 = FusedAdam([p1], lr=1e-2), FusedAdam([p2], lr=1e-2)
    o1.clip_coef = torch.tensor(0.25, device="cuda")
    gr = torch.randn(1000, generator=g).cuda()
    p1.grad, p2.grad = gr.clone(), gr * 0.25
    o1.step()
    o2.step()
    assert relerr(p1, p2) < 1e-6
