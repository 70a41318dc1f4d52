"""GPU parity of the training backward kernels: every backward entry point of the C ABI, called directly, against fp64
torch autograd of the forward formula (the oracle's own transform modules where they exist, else the formula of
include/usflow_b200.h).

Harness rules, so that a subtly wrong kernel fails instead of passing:
  * every operand lives inside a wider buffer: leading dimension wider than the row and one extra row below.  The
    padding of inputs is NaN (a kernel that reads past a row or past the last row produces NaN); the padding of outputs
    holds a fixed sentinel that must be bit-unchanged afterwards;
  * `=` outputs start as NaN, so every element must be written; `+=` outputs start as random values and are checked
    against prefill + reference;
  * inputs are scaled so that every term of a gradient is of the same order as the others, and masks are random.
Tolerance: max-norm relative error <= 2e-5 against fp64, the convention of test_gpu_kernels.py."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

NAN = float("nan")
SENTINEL = -12345.5          # exactly representable: bit comparisons are meaningful
TOL = 2e-5


@pytest.fixture(scope="module")
def K():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from nf4ad_b200 import _lib
    assert _lib.lib().usf_device_ok() == 1, "expected an sm_100 device"
    return _lib


def relerr(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def assert_close(got, ref, what, tol=TOL):
    """Max-norm relative error; an all-zero reference is compared absolutely."""
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.numel() == 0:
        return
    g, r = got.detach().double().cpu(), ref.detach().double().cpu()
    assert bool(torch.isfinite(g).all()), (what, "non-finite output: an element was not written")
    err = float((g - r).abs().max()) if float(r.abs().max()) == 0.0 else relerr(g, r)
    assert err <= tol, (what, err)


class Buf:
    """A (rows, cols) fp32 operand inside a wider device buffer: leading dimension cols + pad, one extra row below, and
    `off` floats before the first element (off = 1 misaligns the rows for the vector loads).  `fill` goes everywhere
    outside the operand, `inner` (or `fill`) inside it."""

    def __init__(self, rows, cols, pad=3, fill=SENTINEL, inner=None, off=0, ld=None):
        self.rows, self.cols, self.off = rows, cols, off
        self.ld = ld if ld is not None else cols + pad
        self.buf = torch.full(((rows + 1) * self.ld + off,), fill, dtype=torch.float32, device="cuda")
        self.grid = self.buf[off:].view(rows + 1, self.ld)
        self.outside = torch.ones(rows + 1, self.ld, dtype=torch.bool, device="cuda")
        self.outside[:rows, :cols] = False
        if inner is not None:
            self.view.copy_(inner.reshape(rows, cols).to(torch.float32))
        self.before = self.buf.clone()

    @property
    def view(self):
        return self.grid[:self.rows, :self.cols]

    @property
    def ptr(self):
        return C.c_void_p(self.buf.data_ptr() + 4 * self.off)   # non-NULL also when the operand is empty

    def value(self):
        return self.view.detach().double().cpu()

    def assert_outside_unchanged(self, what):
        now, was = self.buf.view(torch.int32), self.before.view(torch.int32)
        head = bool((now[:self.off] == was[:self.off]).all())
        grid_now, grid_was = now[self.off:].view(self.rows + 1, self.ld), was[self.off:].view(self.rows + 1, self.ld)
        body = bool((grid_now[self.outside] == grid_was[self.outside]).all())
        assert head and body, (what, "wrote outside the operand")


def as2d(t):
    return t if t.dim() == 2 else t.reshape(1, -1)


def inp(t, pad=3, off=0):
    """Input operand: NaN padding."""
    t = as2d(t)
    return Buf(t.shape[0], t.shape[1], pad=pad, fill=NAN, inner=t, off=off)


def vec_in(t):
    return inp(t.reshape(1, -1))


def out_eq(rows, cols, pad=3, off=0):
    """`=` output: NaN inside, sentinel outside."""
    b = Buf(rows, cols, pad=pad, fill=SENTINEL, off=off)
    b.view.fill_(NAN)
    b.before = b.buf.clone()
    return b


def out_acc(prefill, pad=3, off=0):
    """`+=` output: random prefill inside, sentinel outside."""
    p = as2d(prefill)
    return Buf(p.shape[0], p.shape[1], pad=pad, fill=SENTINEL, inner=p, off=off)


def prefill_like(ref, g, scale=0.5):
    """Random values of about half the reference's size: an output that overwrites instead of adding is off by ~50%."""
    mag = float(ref.abs().max()) if ref.numel() else 1.0
    return (torch.randn(ref.shape, generator=g, dtype=torch.float64) * scale * max(mag, 1e-3)).float().double()


def sync_check(K, rc, what):
    K.check(rc, what)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------------
# usf_gemm: C[M,N] (+)= opA(A) opB(B)^T
# ------------------------------------------------------------------------------------------------------------------
def _gemm_case(K, M, N, Kd, at, bt, acc, pad=3, off=0, seed=0):
    g = torch.Generator().manual_seed(seed)
    A = torch.randn((Kd, M) if at else (M, Kd), generator=g, dtype=torch.float64).float().double()
    Bm = torch.randn((Kd, N) if bt else (N, Kd), generator=g, dtype=torch.float64).float().double()
    Aop, Bop = (A.t() if at else A), (Bm.t() if bt else Bm)
    ref = Aop @ Bop.t()
    a, b = inp(A, pad, off), inp(Bm, pad, off)
    if acc:
        pre = prefill_like(ref, g)
        c = out_acc(pre, pad, off)
        ref = ref + pre
    else:
        c = out_eq(M, N, pad, off)
    sync_check(K, K.lib().usf_gemm(a.ptr, a.ld, at, b.ptr, b.ld, bt, c.ptr, c.ld, acc, M, N, Kd, K.stream()), "usf_gemm")
    c.assert_outside_unchanged("C")
    return c.value(), ref


# (256, 256, 1024): 4 output tiles, K >= 64 -> split-K with atomics (the output is cleared first unless accumulate);
# (1280, 1280, 96): 100 tiles > 74 -> one CTA per tile walks K
@pytest.mark.parametrize("M,N,Kd", [(256, 256, 1024), (1280, 1280, 96)])
@pytest.mark.parametrize("at,bt", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("acc", [0, 1])
def test_gemm_transposes_and_split(K, M, N, Kd, at, bt, acc):
    got, ref = _gemm_case(K, M, N, Kd, at, bt, acc, seed=M + 2 * at + bt + 4 * acc)
    assert_close(got, ref, "C")


@pytest.mark.parametrize("M,N,Kd,pad,off", [
    (256, 256, 1024, 0, 0),     # split path with ldc == N: the plain memset clears C
    (1, 1, 1, 3, 0), (129, 130, 17, 3, 0), (129, 130, 300, 5, 0),
    (70, 33, 200, 4, 1), (300, 260, 40, 4, 1),      # every pointer one float past 16-byte alignment: scalar loads
])
@pytest.mark.parametrize("at,bt", [(0, 1), (1, 0)])
@pytest.mark.parametrize("acc", [0, 1])
def test_gemm_ragged_strided_unaligned(K, M, N, Kd, pad, off, at, bt, acc):
    got, ref = _gemm_case(K, M, N, Kd, at, bt, acc, pad=pad, off=off, seed=M * 7 + N + Kd + acc)
    assert_close(got, ref, "C")


@pytest.mark.parametrize("acc", [0, 1])
def test_gemm_empty_reduction_and_empty_output(K, acc):
    g = torch.Generator().manual_seed(3)
    dummy = inp(torch.randn(4, 4, generator=g))
    # K = 0: C = 0, or C unchanged when accumulating
    pre = torch.randn(37, 45, generator=g).double()
    c = out_acc(pre) if acc else out_eq(37, 45)
    sync_check(K, K.lib().usf_gemm(dummy.ptr, 4, 0, dummy.ptr, 4, 1, c.ptr, c.ld, acc, 37, 45, 0, K.stream()), "usf_gemm")
    c.assert_outside_unchanged("C")
    expect = pre if acc else torch.zeros(37, 45, dtype=torch.float64)
    assert torch.equal(c.value(), expect)
    # M = 0 or N = 0: nothing is written
    for M, N in ((0, 45), (37, 0)):
        c = Buf(37, 45, fill=SENTINEL)
        sync_check(K, K.lib().usf_gemm(dummy.ptr, 4, 0, dummy.ptr, 4, 1, c.ptr, c.ld, acc, M, N, 4, K.stream()),
                   "usf_gemm")
        assert torch.equal(c.buf.view(torch.int32), c.before.view(torch.int32)), (M, N)


# ------------------------------------------------------------------------------------------------------------------
# usf_linear_bwd: dx = g W, dW (+)= g^T x, db (+)= colsum(g), g = dy gated by y_relu > 0
# ------------------------------------------------------------------------------------------------------------------
def _linear_bwd_case(K, B, N, Kd, relu, acc, drop=None, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, Kd, generator=g, dtype=torch.float64).float().double().requires_grad_()
    W = (torch.randn(N, Kd, generator=g, dtype=torch.float64) / Kd ** 0.5).float().double().requires_grad_()
    b = torch.randn(N, generator=g, dtype=torch.float64).float().double().requires_grad_()
    dy = torch.randn(B, N, generator=g, dtype=torch.float64).float().double()
    pre = x @ W.t() + b
    y = torch.relu(pre) if relu else pre
    (y * dy).sum().backward()
    # the kernel's gate is y_relu > 0: the fp64 output cast to fp32 has exact zeros exactly where pre <= 0
    y_relu = torch.relu(pre.detach()).float()
    ops = {"dx": x.grad, "dW": W.grad, "db": b.grad}
    dyb, xb, Wb = inp(dy), inp(x.detach()), inp(W.detach())
    yrb = inp(y_relu) if relu else None
    scratch = torch.full((max(B * N, 1),), NAN, device="cuda") if relu else None
    outs, refs = {}, {}
    for name, ref in ops.items():
        if name == drop:
            continue
        if name == "dx" or not acc:
            outs[name] = out_eq(*as2d(ref).shape)
            refs[name] = ref
        else:
            pre_v = prefill_like(ref, g)
            outs[name] = out_acc(pre_v)
            refs[name] = ref + pre_v
    p = lambda n: outs[n].ptr if n in outs else None
    ld = lambda n: outs[n].ld if n in outs else 0
    sync_check(K, K.lib().usf_linear_bwd(dyb.ptr, dyb.ld, xb.ptr, xb.ld, Wb.ptr, Wb.ld, yrb.ptr if relu else None,
                                         yrb.ld if relu else 0, p("dx"), ld("dx"), p("dW"), ld("dW"), p("db"), acc,
                                         C.c_void_p(scratch.data_ptr()) if relu else None, B, N, Kd, K.stream()),
               "usf_linear_bwd")
    for name, o in outs.items():
        o.assert_outside_unchanged(name)
        assert_close(o.value().reshape(refs[name].shape), refs[name], name)


# wgrad GEMM (M = N, N = K, reduction over B): (1000, 64, 130) 2 tiles -> split-K; (257, 1160, 1030) 90 tiles -> not
# split (its dgrad GEMM, 27 tiles, is); (50, 200, 70) B < 64 -> no split anywhere
@pytest.mark.parametrize("B,N,Kd", [(1000, 64, 130), (257, 1160, 1030), (50, 200, 70), (1, 1, 1), (129, 130, 17)])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("acc", [0, 1])
def test_linear_bwd(K, B, N, Kd, relu, acc):
    _linear_bwd_case(K, B, N, Kd, relu, acc, seed=B + N + Kd + 2 * relu + acc)


@pytest.mark.parametrize("drop", ["dx", "dW", "db"])
@pytest.mark.parametrize("relu", [False, True])
def test_linear_bwd_null_outputs(K, drop, relu):
    _linear_bwd_case(K, 300, 96, 80, relu, 0, drop=drop, seed=11 + relu)
    _linear_bwd_case(K, 300, 96, 80, relu, 1, drop=drop, seed=12 + relu)


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("acc", [0, 1])
@pytest.mark.parametrize("null_rows", [False, True])
def test_linear_bwd_empty_batch(K, relu, acc, null_rows):
    """B = 0: dW = 0 and db = 0 (accumulate == 0) -- not whatever the caller's buffers held -- and dx untouched.
    null_rows: the row operands are NULL, as torch's data pointer of an empty tensor is."""
    g = torch.Generator().manual_seed(5)
    N, Kd = 48, 70
    dummy = inp(torch.randn(2, max(N, Kd), generator=g))
    rows = None if null_rows else dummy.ptr
    Wb = inp(torch.randn(N, Kd, generator=g))
    dx = Buf(4, Kd, fill=SENTINEL)
    pre_W, pre_b = torch.randn(N, Kd, generator=g).double(), torch.randn(N, generator=g).double()
    dW = out_acc(pre_W) if acc else out_eq(N, Kd)
    db = out_acc(pre_b) if acc else out_eq(1, N)
    sync_check(K, K.lib().usf_linear_bwd(rows, dummy.ld, rows, dummy.ld, Wb.ptr, Wb.ld, rows if relu else None, dummy.ld,
                                         dx.ptr, dx.ld, dW.ptr, dW.ld, db.ptr, acc, rows if relu else None, 0, N, Kd,
                                         K.stream()), "usf_linear_bwd")
    assert torch.equal(dx.buf.view(torch.int32), dx.before.view(torch.int32))
    dW.assert_outside_unchanged("dW")
    db.assert_outside_unchanged("db")
    assert torch.equal(dW.value(), pre_W if acc else torch.zeros(N, Kd, dtype=torch.float64))
    assert torch.equal(db.value().reshape(-1), pre_b if acc else torch.zeros(N, dtype=torch.float64))


def test_linear_fn_empty_batch_zero_grads(K):
    """ops.LinearFn on an empty batch: W.grad and b.grad are exactly zero, even when the allocator hands the backward
    pass a block that held NaN."""
    from nf4ad_b200 import ops
    N, Kd = 40, 24
    for relu in (False, True):
        x = torch.randn(0, Kd, device="cuda", requires_grad=True)
        W = torch.randn(N, Kd, device="cuda", requires_grad=True)
        b = torch.randn(N, device="cuda", requires_grad=True)
        y = ops.LinearFn.apply(x, W, b, relu)
        assert y.shape == (0, N)
        loss = y.sum()
        # NaN-filled blocks of dW's and db's sizes, freed again: the many of them take up every free block of those
        # sizes the allocator held, so the torch.empty of the backward pass is handed NaN, not fresh zeros
        junk = [torch.full((N, Kd), NAN, device="cuda") for _ in range(64)]
        junk += [torch.full((N,), NAN, device="cuda") for _ in range(64)]
        del junk
        loss.backward()
        assert W.grad is not None and b.grad is not None
        assert float(W.grad.abs().max()) == 0.0 and not bool(W.grad.isnan().any())
        assert float(b.grad.abs().max()) == 0.0 and not bool(b.grad.isnan().any())
        assert x.grad.shape == (0, Kd)


# ------------------------------------------------------------------------------------------------------------------
# usf_colsum: out[c] (+)= coef * sum_b a[b, c]
# ------------------------------------------------------------------------------------------------------------------
# B = 70000: more than 64 row slices of 256 rows, so every CTA of the capped grid loops
@pytest.mark.parametrize("B,N,coef", [(1000, 70, -0.75), (70000, 33, 1.5), (1, 1, 2.0), (0, 20, 1.0)])
@pytest.mark.parametrize("acc", [0, 1])
def test_colsum(K, B, N, coef, acc):
    g = torch.Generator().manual_seed(B + N + acc)
    a = (torch.randn(B, N, generator=g) + 0.3).double()
    ref = coef * a.sum(0)
    ab = inp(a) if B else inp(torch.randn(2, N, generator=g))
    if acc:
        pre = prefill_like(ref, g) if B else torch.randn(N, generator=g).double()
        o = out_acc(pre)
        ref = ref + pre
    else:
        o = out_eq(1, N)
    sync_check(K, K.lib().usf_colsum(ab.ptr, ab.ld, coef, acc, o.ptr, B, N, K.stream()), "usf_colsum")
    o.assert_outside_unchanged("out")
    if B == 0:
        assert torch.equal(o.value().reshape(-1), ref)
    else:
        assert_close(o.value().reshape(-1), ref, "colsum")


# ------------------------------------------------------------------------------------------------------------------
# usf_lu_pack_bwd: dL_raw += strict_lower(dW U^T), dU_raw += upper(L^T dW), dU_raw_ii += dlogdet / U_ii
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [1, 5, 33, 130, 784])
@pytest.mark.parametrize("dlogdet", [0.0, 1.3])
@pytest.mark.parametrize("with_dW", [True, False])
def test_lu_pack_bwd(K, O, D, dlogdet, with_dW):
    torch.manual_seed(D)
    g = torch.Generator().manual_seed(D + 1)
    lu = O.transforms.LUTransform(D, 1.0).double()
    with torch.no_grad():
        lu.L_raw.add_(torch.randn(D, D, generator=g, dtype=torch.float64) / D ** 0.5)
        lu.U_raw.add_(torch.randn(D, D, generator=g, dtype=torch.float64) / D ** 0.5)
        lu.U_raw.diagonal().copy_((0.6 + torch.rand(D, generator=g, dtype=torch.float64)) *
                                  torch.where(torch.rand(D, generator=g) < 0.3, -1.0, 1.0))
        lu.L_raw.add_(torch.randn(D, D, generator=g, dtype=torch.float64).triu(0) * 3)   # junk in the unused triangles
        lu.U_raw.add_(torch.randn(D, D, generator=g, dtype=torch.float64).tril(-1) * 3)  # and L's diagonal: ignored
        lu.L_raw.copy_(lu.L_raw.float())
        lu.U_raw.copy_(lu.U_raw.float())
    dW = torch.randn(D, D, generator=g, dtype=torch.float64).float().double()
    loss = dlogdet * lu.log_abs_det_jacobian(None, None)
    if with_dW:
        loss = loss + (lu.weight * dW).sum()
    if with_dW or dlogdet != 0.0:
        loss.backward()
    zero = torch.zeros(D, D, dtype=torch.float64)
    gL = lu.L_raw.grad if lu.L_raw.grad is not None else zero
    gU = lu.U_raw.grad if lu.U_raw.grad is not None else zero
    # leading dimension is D for every matrix of this entry point: pad = 0, the sentinel / NaN row below remains
    Lb, Ub, dWb = inp(lu.L_raw.detach(), pad=0), inp(lu.U_raw.detach(), pad=0), inp(dW, pad=0)
    pre_L = prefill_like(gL if with_dW else gU, g)
    pre_U = prefill_like(gU, g)
    dL, dU = out_acc(pre_L, pad=0), out_acc(pre_U, pad=0)
    scratch = torch.full((3 * D * D,), NAN, device="cuda")
    sync_check(K, K.lib().usf_lu_pack_bwd(dWb.ptr if with_dW else None, Lb.ptr, Ub.ptr, dlogdet, D, dL.ptr, dU.ptr,
                                          C.c_void_p(scratch.data_ptr()), K.stream()), "usf_lu_pack_bwd")
    dL.assert_outside_unchanged("dL_raw")
    dU.assert_outside_unchanged("dU_raw")
    gotL, gotU = dL.value(), dU.value()
    # outside the strict lower (dL_raw) / upper (dU_raw) triangles the prefill stays bit for bit
    assert torch.equal(gotL.triu(0), pre_L.triu(0)) and torch.equal(gotU.tril(-1), pre_U.tril(-1))
    if not with_dW and dlogdet == 0.0:
        assert torch.equal(gotL, pre_L) and torch.equal(gotU, pre_U)
        return
    if with_dW:
        assert_close(gotL.tril(-1) - pre_L.tril(-1), gL, "dL_raw")
    else:
        assert torch.equal(gotL, pre_L)
    assert_close(gotU, pre_U + gU, "dU_raw")


# ------------------------------------------------------------------------------------------------------------------
# usf_householder_bwd: dx and dV (+=) through nvs reflections, given the layer input
# ------------------------------------------------------------------------------------------------------------------
def _householder_case(K, O, B, D, nvs, reverse, seed):
    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed + 1)
    hh = O.transforms.HouseholderTransform(D, nvs).double()
    with torch.no_grad():
        hh.vk_householder.copy_(hh.vk_householder.float())
    V = hh.vk_householder
    # x and dy carry a component along a reflection vector, so that (x.v) and (dy.v) -- and with them every term of
    # dv = -c dy - e x + f v -- are of the same order instead of O(1/sqrt(D)) apart
    x = torch.randn(B, D, generator=g, dtype=torch.float64)
    dy = torch.randn(B, D, generator=g, dtype=torch.float64)
    if nvs:
        vhat = V.detach() / V.detach().norm(dim=1, keepdim=True)
        x = x + torch.randn(B, 1, generator=g, dtype=torch.float64) * vhat[0] * D ** 0.5
        dy = dy + torch.randn(B, 1, generator=g, dtype=torch.float64) * vhat[-1] * D ** 0.5
    x = x.float().double().requires_grad_()
    dy = dy.float().double()
    y = hh.backward(x) if reverse else hh.forward(x)
    (y * dy).sum().backward()
    ref_dx = x.grad
    ref_dV = V.grad if V.grad is not None else torch.zeros(nvs, D, dtype=torch.float64)
    dyb, xb = inp(dy), inp(x.detach())
    Vb = inp(V.detach(), pad=0) if nvs else inp(torch.zeros(1, D), pad=0)
    dx = out_eq(B, D)
    pre_V = prefill_like(ref_dV, g) if nvs else torch.zeros(0, D, dtype=torch.float64)
    dV = out_acc(pre_V, pad=0) if nvs else Buf(1, D, pad=0, fill=SENTINEL)
    scratch = torch.full((nvs * B * D,), NAN, device="cuda") if nvs > 1 else None      # as ops.HouseholderFn sizes it
    sync_check(K, K.lib().usf_householder_bwd(dyb.ptr, dyb.ld, xb.ptr, xb.ld, Vb.ptr if nvs else None, nvs, int(reverse),
                                              dx.ptr, dx.ld, dV.ptr, C.c_void_p(scratch.data_ptr()) if nvs > 1 else None,
                                              B, D, K.stream()), "usf_householder_bwd")
    dx.assert_outside_unchanged("dx")
    dV.assert_outside_unchanged("dV")
    assert_close(dx.value(), ref_dx, "dx")
    if nvs == 0:
        assert torch.equal(dV.buf.view(torch.int32), dV.before.view(torch.int32))
        return
    got_dV = dV.value()
    if D == 1:
        # one coordinate: every reflection is -1 whatever v is, dV = 0 analytically.  The kernel's per-row terms
        # (-c dy, -e x, f v: each ~2|x dy / v|) cancel in fp32, so the sum is bounded against their magnitude.
        scale = float((4 * (x.detach() * dy).abs().sum(0) / V.detach().abs().min()).max())
        err = float((got_dV - pre_V).abs().max())
        assert err <= TOL * scale, ("dV", err, scale)
    else:
        assert_close(got_dV, pre_V + ref_dV, "dV")


# B = 5: fewer rows than one CTA's 8 warps; B = 5000: more rows than 2 CTAs per SM x 8 warps, each warp loops.
# nvs >= 3 runs the middle reflections in place on the gradient scratch buffer.
@pytest.mark.parametrize("D", [1, 33, 784])
@pytest.mark.parametrize("nvs", [0, 1, 2, 3, 5])
@pytest.mark.parametrize("reverse", [0, 1])
@pytest.mark.parametrize("B", [5, 5000])
def test_householder_bwd(K, O, D, nvs, reverse, B):
    _householder_case(K, O, B, D, nvs, reverse, seed=D * 10 + nvs + 100 * reverse + B)


@pytest.mark.parametrize("reverse", [0, 1])
def test_householder_bwd_large_dim(K, O, reverse):
    """D = 13000: the CTA's dv accumulator (4 D bytes) needs the > 48 KB dynamic shared-memory opt-in."""
    _householder_case(K, O, 64, 13000, 3, reverse, seed=13000 + reverse)


# ------------------------------------------------------------------------------------------------------------------
# usf_scale_bwd: forward y = x * s (xy = x), inverse y = x / s (xy = the OUTPUT y)
# ------------------------------------------------------------------------------------------------------------------
# B = 140000: the row grid (256 slices of 512 rows) is capped, every CTA loops
@pytest.mark.parametrize("B,D", [(300, 70), (33, 784), (140000, 3)])
@pytest.mark.parametrize("inverse", [0, 1])
@pytest.mark.parametrize("with_dscale", [True, False])
def test_scale_bwd(K, O, B, D, inverse, with_dscale):
    g = torch.Generator().manual_seed(B + D + inverse)
    st = O.transforms.ScaleTransform((D,)).double()
    with torch.no_grad():
        st.scale.copy_(((0.5 + torch.rand(D, generator=g)) * torch.where(torch.rand(D, generator=g) < 0.4, -1.0, 1.0)))
    x = (torch.randn(B, D, generator=g) + 0.3).double().requires_grad_()
    dy = (torch.randn(B, D, generator=g) + 0.3).double()
    y = st.backward(x) if inverse else st.forward(x)
    (y * dy).sum().backward()
    xy = y.detach().float() if inverse else x.detach().float()
    dyb, xyb, sb = inp(dy), inp(xy), vec_in(st.scale.detach())
    dx = out_eq(B, D)
    pre = prefill_like(st.scale.grad, g)
    ds = out_acc(pre) if with_dscale else None
    sync_check(K, K.lib().usf_scale_bwd(dyb.ptr, dyb.ld, xyb.ptr, xyb.ld, sb.ptr, inverse, dx.ptr, dx.ld,
                                        ds.ptr if ds else None, B, D, K.stream()), "usf_scale_bwd")
    dx.assert_outside_unchanged("dx")
    assert_close(dx.value(), x.grad, "dx")
    if ds is not None:
        ds.assert_outside_unchanged("dscale")
        assert_close(ds.value().reshape(-1), pre.reshape(-1) + st.scale.grad, "dscale")


# ------------------------------------------------------------------------------------------------------------------
# usf_base_logprob_bwd: dz = dout * d logp / dz, dloc += ..., dscale[d or 0] += ...
# ------------------------------------------------------------------------------------------------------------------
def _base_case(K, kind, B, D, numel, drop, seed):
    g = torch.Generator().manual_seed(seed)
    dist = (torch.distributions.Normal, torch.distributions.Laplace)[kind]
    loc = torch.randn(D, generator=g).double().requires_grad_()
    sc = (0.5 + torch.rand(numel, generator=g)).double().requires_grad_()
    z = (loc.detach() + sc.detach() * torch.randn(B, D, generator=g, dtype=torch.float64)).float().double()
    tie = torch.rand(B, D, generator=g) < 0.05
    z = torch.where(tie, loc.detach().expand(B, D), z).requires_grad_()   # z == loc: Laplace subgradient 0, as torch
    dout = (torch.randn(B, generator=g) + 0.5).double()
    lp = dist(loc, sc.expand(D)).log_prob(z).sum(1)
    (lp * dout).sum().backward()
    doutb, zb, locb, scb = vec_in(dout), inp(z.detach()), vec_in(loc.detach()), vec_in(sc.detach())
    dz = None if drop == "dz" else out_eq(B, D)
    pre_l, pre_s = prefill_like(loc.grad, g), prefill_like(sc.grad, g)
    dl = None if drop == "dloc" else out_acc(pre_l)
    ds = None if drop == "dscale" else out_acc(pre_s)
    sync_check(K, K.lib().usf_base_logprob_bwd(kind, doutb.ptr, zb.ptr, zb.ld, locb.ptr, scb.ptr, numel,
                                               dz.ptr if dz else None, dz.ld if dz else 0, dl.ptr if dl else None,
                                               ds.ptr if ds else None, B, D, K.stream()), "usf_base_logprob_bwd")
    if dz is not None:
        dz.assert_outside_unchanged("dz")
        assert_close(dz.value(), z.grad, "dz")
    if dl is not None:
        dl.assert_outside_unchanged("dloc")
        assert_close(dl.value().reshape(-1), pre_l + loc.grad, "dloc")
    if ds is not None:
        ds.assert_outside_unchanged("dscale")
        assert_close(ds.value().reshape(-1), pre_s + sc.grad, "dscale")


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("per_dim", [True, False])
@pytest.mark.parametrize("drop", [None, "dz", "dloc", "dscale"])
def test_base_logprob_bwd(K, kind, per_dim, drop):
    D = 70
    _base_case(K, kind, 300, D, D if per_dim else 1, drop, seed=kind * 7 + per_dim * 3 + len(drop or ""))


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("per_dim", [True, False])
def test_base_logprob_bwd_many_rows(K, kind, per_dim):
    """B = 140000: the row grid is capped at 256 slices, every CTA loops."""
    _base_case(K, kind, 140000, 5, 5 if per_dim else 1, None, seed=140000 + kind + 2 * per_dim)


# ------------------------------------------------------------------------------------------------------------------
# usf_coupling_bwd: dx, ds, dt of the masked coupling in the direction that ran, with the log-det term
# ------------------------------------------------------------------------------------------------------------------
class _GivenConditioner(torch.nn.Module):
    """A conditioner that ignores its input and returns given leaves: the coupling's own VJP, with s and t as inputs."""

    def __init__(self, out):
        super().__init__()
        self.out = out

    def forward(self, xm, context=None):
        return self.out


_COUPLING_CASES = [(act, inverse, affine, packed) for act in (0, 1) for inverse in (0, 1) for affine in (True, False)
                   for packed in (False, True) if affine or not packed]


@pytest.mark.parametrize("act,inverse,affine,packed", _COUPLING_CASES)
def test_coupling_bwd(K, O, act, inverse, affine, packed):
    """The reference is the restated MaskedAffineCoupling (with its literal 1e-6 / 1e-12) for the affine form and the
    oracle's MaskedCoupling for the additive one.  packed: s and t are the two halves of one (B, 2D) conditioner output
    and ds / dt the two halves of one (B, 2D) gradient (CouplingPackedFn), lds = ldt = ldds = lddt = 2D."""
    B, D = 67, 45
    seed = 1000 + 8 * act + 4 * inverse + 2 * affine + packed
    g = torch.Generator().manual_seed(seed)
    mask = (torch.rand(D, generator=g) < 0.5).double()
    mask[0], mask[1] = 0.0, 1.0
    name = ("exp", "softplus")[act]
    for clamp in (1.0, 5.0):
        for coef in (1.0, -1.0, 0.5):
            for with_dladj in (False, True):
                x = torch.randn(B, D, generator=g).double().requires_grad_()
                s = torch.randn(B, D, generator=g) * 0.8
                s[torch.rand(B, D, generator=g) < 0.05] = 20.0          # tanh saturates (to +-1 exactly in fp32)
                s[torch.rand(B, D, generator=g) < 0.05] = -20.0
                s = s.double().requires_grad_()
                t = torch.randn(B, D, generator=g).double().requires_grad_()
                dy = torch.randn(B, D, generator=g).double()
                dladj = (2.0 * torch.randn(B, generator=g)).double()
                if affine:
                    layer = O.MaskedAffineCoupling(mask, _GivenConditioner((s, t)), scale_activation=name, clamp=clamp)
                else:
                    layer = O.MaskedCoupling(mask, _GivenConditioner(t))
                layer = layer.double()
                y = layer.backward(x) if inverse else layer.forward(x)
                loss = (y * dy).sum()
                if with_dladj and affine:
                    loss = loss + (coef * layer.log_abs_det_jacobian(x, y) * dladj).sum()
                loss.backward()
                dyb, xb, mb = inp(dy), inp(x.detach()), vec_in(mask)
                dlb = vec_in(dladj) if with_dladj else None
                if packed:
                    stb = Buf(B, 2 * D, pad=0, fill=NAN, inner=torch.cat([s.detach(), t.detach()], 1))
                    s_ptr, t_ptr = stb.ptr, C.c_void_p(stb.buf.data_ptr() + 4 * D)
                    lds = ldt = 2 * D
                    dst = out_eq(B, 2 * D, pad=0)
                    ds_ptr, dt_ptr = dst.ptr, C.c_void_p(dst.buf.data_ptr() + 4 * D)
                    ldds = lddt = 2 * D
                else:
                    sb, tb = (inp(s.detach()) if affine else None), inp(t.detach())
                    s_ptr, lds, t_ptr, ldt = (sb.ptr if affine else None), (sb.ld if affine else 0), tb.ptr, tb.ld
                    dsb, dtb = (out_eq(B, D) if affine else None), out_eq(B, D)
                    ds_ptr, ldds = (dsb.ptr, dsb.ld) if affine else (None, 0)
                    dt_ptr, lddt = dtb.ptr, dtb.ld
                dx = out_eq(B, D)
                sync_check(K, K.lib().usf_coupling_bwd(dyb.ptr, dyb.ld, dlb.ptr if dlb else None, coef, xb.ptr, xb.ld,
                                                       s_ptr, lds, t_ptr, ldt, mb.ptr, clamp, inverse, act, dx.ptr, dx.ld,
                                                       ds_ptr, ldds, dt_ptr, lddt, B, D, K.stream()), "usf_coupling_bwd")
                case = (name, inverse, affine, packed, clamp, coef, with_dladj)
                dx.assert_outside_unchanged(("dx",) + case)
                assert_close(dx.value(), x.grad, ("dx",) + case)
                if packed:
                    dst.assert_outside_unchanged(("dst",) + case)
                    got_ds, got_dt = dst.value()[:, :D], dst.value()[:, D:]
                else:
                    dtb.assert_outside_unchanged(("dt",) + case)
                    got_dt = dtb.value()
                    if affine:
                        dsb.assert_outside_unchanged(("ds",) + case)
                        got_ds = dsb.value()
                assert_close(got_dt, t.grad, ("dt",) + case)
                if affine:
                    assert_close(got_ds, s.grad, ("ds",) + case)


# ------------------------------------------------------------------------------------------------------------------
# usf_to_tf32x3: (hi, lo) operand pairs of the 3xTF32 training GEMMs
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,relu,ld", [(8, 16, False, 0), (64, 784, True, 0), (257, 100, True, 0), (4096, 256, False, 0),
                                         (4096, 1568, True, 0), (130, 99, True, 0), (131, 99, True, 104), (70, 5, False, 8),
                                         (1000, 784, False, 800)])
def test_to_tf32x3_operand_pass(K, B, N, relu, ld):
    """Row and transposed (hi, lo) pairs and column sums of the (ReLU-gated) input, checked by their properties: hi is
    tf32 (low 13 mantissa bits zero), hi + lo == v exactly, |lo| <= 2^-11 |hi|, the transposed pair is the row pair
    transposed bit for bit, the pad columns are zero."""
    g = torch.Generator().manual_seed(B + N)
    xin = torch.randn(B, ld or N, generator=g)
    mask_in = torch.randn(B, ld or N, generator=g)
    xb = Buf(B, N, ld=ld or N, fill=NAN, inner=xin[:, :N])
    mb = Buf(B, N, ld=ld or N, fill=NAN, inner=mask_in[:, :N]) if relu else None
    v = torch.where(mask_in[:, :N] > 0, xin[:, :N], torch.zeros(B, N)) if relu else xin[:, :N]
    ldr, ldt = (N + 3) // 4 * 4, (B + 3) // 4 * 4
    rh, rl = out_eq(B, ldr, pad=0), out_eq(B, ldr, pad=0)
    th, tl = out_eq(N, ldt, pad=0), out_eq(N, ldt, pad=0)
    pre = torch.randn(N, generator=g).double()
    cs = out_acc(pre)
    sync_check(K, K.lib().usf_to_tf32x3(xb.ptr, xb.ld, mb.ptr if relu else None, mb.ld if relu else 0, rh.ptr, rl.ptr, ldr,
                                        th.ptr, tl.ptr, ldt, cs.ptr, B, N, K.stream()), "usf_to_tf32x3")
    for b_, n_ in ((rh, "rows_hi"), (rl, "rows_lo"), (th, "t_hi"), (tl, "t_lo"), (cs, "colsum")):
        b_.assert_outside_unchanged(n_)
    RH, RL, TH, TL = (b_.view.cpu() for b_ in (rh, rl, th, tl))
    assert float(RH[:, N:].abs().sum()) == 0.0 and float(RL[:, N:].abs().sum()) == 0.0
    assert float(TH[:, B:].abs().sum()) == 0.0 and float(TL[:, B:].abs().sum()) == 0.0
    hi, lo = RH[:, :N], RL[:, :N]
    assert int((hi.view(torch.int32) & 0x1FFF).ne(0).sum()) == 0
    assert torch.equal(hi.double() + lo.double(), v.double())
    assert bool((lo.abs() <= hi.abs() * 2.0 ** -11).all())
    assert torch.equal(TH[:, :B].view(torch.int32), hi.t().contiguous().view(torch.int32))
    assert torch.equal(TL[:, :B].view(torch.int32), lo.t().contiguous().view(torch.int32))
    assert_close(cs.value().reshape(-1), pre + v.double().sum(0), "colsum", tol=1e-5)
