"""Stack compiler: turns a `Flow`'s layer list into the packed descriptor array of `usf_stack_run`.

A flow built by `USFlow` / `NonUSFlow` (`/root/reference/src/nf4ad/flows.py:78-114`) is, in either
direction, an alternation   affine run, coupling, affine run, coupling, ..., affine run   where an "affine
run" is a maximal sequence of LU / Householder / Scale / Sequential / BlockAffine / Inverse layers.  Every
run is a single dense map `x -> A x + c`; the compiler materialises (A, c) ONCE per weight version by
pushing the rows of `[0; I]` through the run's own layer kernels (usf_linear / usf_lu_solve /
usf_householder / usf_scale -- so the inverse of an LU layer is produced by the triangular-solve
kernel), then packs it with the coupling masks folded in as a column permutation: after each affine map
the activation row is laid out `[conditioning coords | pad | transformed coords]`, so mask-select costs
nothing and the conditioner GEMMs touch only the coordinates they need (mask-pruned FLOPs).

The per-batch work is then one GEMM launch chain (`usf_stack_run`): G-GEMM, conditioner GEMMs, and a
last GEMM whose epilogue performs the coupling update + log-det reduction (or the base log-density).
"""
import ctypes as C
import math
import os

import torch

from . import _lib, ops
from ._lib import BlockDesc, BlockGradDesc, LinearDesc, StackDesc, StackGradDesc, check, lib, ptr, stream
from .transforms import context_dim, mlp_layers

_LOG_2PI = math.log(2.0 * math.pi)


def _round_up(a, b):
    return (a + b - 1) // b * b


class Unsupported(Exception):
    """The layer list is not a stack the fused path understands (the layer-wise path is used instead)."""


def _is_coupling(layer):
    return hasattr(layer, "mask") and hasattr(layer, "conditioner") and isinstance(
        getattr(layer, "conditioner"), torch.nn.Module)


def _classify(layers):
    """-> (runs, couplings) with len(runs) == len(couplings) + 1, in generative order."""
    runs, couplings, cur = [], [], []
    for layer in layers:
        if _is_coupling(layer):
            runs.append(cur)
            cur = []
            couplings.append(layer)
        elif getattr(layer, "is_affine", False):
            cur.append(layer)
        else:
            raise Unsupported(f"layer {type(layer).__name__} is neither an affine layer nor a masked coupling")
    runs.append(cur)
    return runs, couplings


def base_params(base, D, device):
    """(kind, loc(D), scale(D)) of a supported base distribution, else None."""
    inner = base
    while isinstance(inner, torch.distributions.Independent):
        inner = inner.base_dist
    name = type(inner).__name__
    if isinstance(inner, torch.distributions.Normal) or name == "Normal":
        kind = 0
    elif isinstance(inner, torch.distributions.Laplace) or name == "Laplace":
        kind = 1
    else:
        return None
    loc, scale = getattr(inner, "loc", None), getattr(inner, "scale", None)
    if loc is None or scale is None:
        return None
    loc = torch.as_tensor(loc, device=device, dtype=torch.float32).reshape(-1)
    scale = torch.as_tensor(scale, device=device).to(torch.float32).reshape(-1)
    if loc.numel() == 1:
        loc = loc.expand(D)
    if scale.numel() == 1:
        scale = scale.expand(D)
    if loc.numel() != D or scale.numel() != D:
        return None
    return kind, loc.contiguous(), scale.contiguous()


class CompiledStack:
    """Device-resident packed weights + the ctypes descriptor tree for one (direction, precision); `grad_desc`: the
    transposed matrices of the reverse chain (`run_grad`), built from the same packs on first use."""

    def __init__(self, layers, base, D, device, inverse, precision):
        self.D, self.inverse, self.precision = D, bool(inverse), precision
        self.device = device
        self._keep = []          # every tensor the descriptors point to
        self._packs = {}         # descriptor address -> the packed weight tensor behind it (W, or bf16x2 [hi ; lo])
        self._grad_desc = None
        self._mlp_widths = {}    # block -> unpadded widths of its conditioner layers
        bf16 = precision == _lib.USF_PREC_BF16
        self._t3 = precision == _lib.USF_PREC_TF32X3      # fp32 weights travel as [W ; W - tf32(W)] (2N rows)
        self._b2 = precision == _lib.USF_PREC_BF16X2      # bf16 weights travel as [bf16(W) ; bf16(W - bf16(W))] (2N rows)
        runs, couplings = _classify(layers)
        n = len(couplings)
        # conditional flows (USFlows soft training): every conditioner takes `cd` context columns, which then travel
        # through the chain as extra conditioning columns of the activation row
        cds = {context_dim(c.conditioner) for c in couplings}
        if len(cds) > 1:
            raise Unsupported("couplings disagree on the context width")
        cd = self.ctx_dim = cds.pop() if cds else 0
        for c in couplings:                # before any packing work: is every coupling one the fused kernels run?
            if getattr(c, "scale_activation", "exp") != "exp":
                raise Unsupported("scale_activation != 'exp'")
            lin = mlp_layers(c.conditioner)
            if lin is None:
                raise Unsupported("conditioner is not a Linear/ReLU chain")
            if len(lin) > _lib.USF_MAX_MLP:
                raise Unsupported("conditioner deeper than USF_MAX_MLP")
            if lin[0].in_features != D + cd:
                raise Unsupported("conditioner input width != D (+ context)")
        Dx = D + cd                        # columns of an input row / of the natural layout: [x (D) | context (cd)]

        with torch.no_grad():
            # ---- per-coupling coordinate layout --------------------------------------------------
            lay = []
            for cpl in couplings:
                m = cpl.mask.reshape(-1).to(device=device, dtype=torch.float32)
                if m.numel() != D or not bool(((m == 0) | (m == 1)).all()):
                    raise Unsupported("mask is not a binary vector of length D")
                idx_a = torch.nonzero(m == 1).reshape(-1).to(torch.int32)
                idx_b = torch.nonzero(m == 0).reshape(-1).to(torch.int32)
                Da, Db = idx_a.numel(), idx_b.numel()
                if Db == 0:
                    raise Unsupported("coupling transforms no coordinate")
                # conditioning part = [a coords | context columns]: contiguous, read by the first conditioner layer
                idx_a = torch.cat([idx_a, torch.arange(D, Dx, dtype=torch.int32, device=device)])
                Da = Da + cd
                b_off = _round_up(Da, 16)      # 32-byte aligned b-part: the epilogues use 256-bit row accesses
                width = _round_up(b_off + Db, 16)
                cols = torch.full((width,), -1, dtype=torch.int32, device=device)
                cols[:Da] = idx_a
                cols[b_off:b_off + Db] = idx_b
                lay.append(dict(idx_a=idx_a, idx_b=idx_b, Da=Da, Db=Db, b_off=b_off, width=width, cols=cols))

            # ---- execution order -------------------------------------------------------------------
            # inverse: runs reversed, each inverted; block j pairs run n-j with coupling n-1-j
            if self.inverse:
                order = [(runs[n - j], couplings[n - 1 - j], lay[n - 1 - j]) for j in range(n)]
                last_run = runs[0]
            else:
                order = [(runs[j], couplings[j], lay[j]) for j in range(n)]
                last_run = runs[n]

            eye_aug = torch.zeros(D + 1, D, device=device, dtype=torch.float32)
            eye_aug[1:] = torch.eye(D, device=device, dtype=torch.float32)

            def run_matrix(run):
                """rows: f(0) = c, f(e_i) = A[:, i] + c   for the run applied in this direction; the context columns
                pass through every affine run unchanged (identity block)."""
                v = eye_aug
                seq = reversed(run) if self.inverse else run
                for layer in seq:
                    v = layer.backward(v) if self.inverse else layer.forward(v)
                if cd == 0:
                    return v.contiguous()
                M = torch.zeros(Dx + 1, Dx, device=device, dtype=torch.float32)
                M[:D + 1, :D] = v
                M[D + 1:, :D] = v[0]          # row i is f(e_i) = A e_i + c: a context unit vector maps x-coordinates to c
                M[D + 1:, D:] = torch.eye(cd, device=device, dtype=torch.float32)
                return M

            natural = torch.arange(Dx, dtype=torch.int32, device=device)
            in_cols = natural                        # column layout of the current activation
            self.blocks = (BlockDesc * max(n, 1))()
            logdet = 0.0
            for j, (run, cpl, L) in enumerate(order):
                blk = self.blocks[j]
                Mt = run_matrix(run)
                self._fill_affine(blk.G, Mt, in_cols, L["cols"], bf16)
                blk.b_off, blk.Da, blk.Db = L["b_off"], L["Da"], L["Db"]
                blk.clamp = float(getattr(cpl, "clamp", 5.0))
                self._fill_conditioner(blk, cpl, L, D, bf16)
                in_cols = L["cols"]
            Mt = run_matrix(last_run)
            out_w = _round_up(D, 16)
            out_cols = torch.full((out_w,), -1, dtype=torch.int32, device=device)
            out_cols[:D] = natural[:D]
            self.G_final = LinearDesc()
            self._fill_affine(self.G_final, Mt, in_cols, out_cols, bf16)

            # ---- data-independent terms ------------------------------------------------------------
            probe = torch.zeros(1, D, device=device, dtype=torch.float32)
            for run in runs:
                for layer in run:
                    logdet = logdet + float(layer.log_abs_det_jacobian(probe, probe))
            self.logdet_const = logdet      # sum of log|det| of all affine layers (generative direction)
            self.base_const = None          # the base log-density's normalising constant (None: no supported base)

            st = StackDesc()
            st.D, st.n_blocks, st.ctx_dim = D, n, cd
            st.blocks = C.cast(self.blocks, C.POINTER(BlockDesc))
            st.G_final = self.G_final
            st.inverse = 1 if self.inverse else 0
            st.base_kind = -1
            st.const_term = 0.0
            bp = base_params(base, D, device) if (base is not None and self.inverse) else None
            if bp is not None:
                kind, loc, scale = bp
                inv_scale = (1.0 / scale).contiguous()
                self._keep += [loc, inv_scale]
                st.base_kind, st.loc, st.inv_scale = kind, loc.data_ptr(), inv_scale.data_ptr()
                if kind == 0:
                    base_const = -float(scale.log().sum()) - 0.5 * D * _LOG_2PI
                else:
                    base_const = -float((2.0 * scale).log().sum())
                self.base_const = base_const
                st.const_term = base_const - logdet
            self.desc = st

    # -------------------------------------------------------------------------------------------
    def _fill_linear(self, desc, W32, Wb, bias, N, K, ldw):
        if getattr(self, "_b2", False):
            if N > 1024:
                raise Unsupported("bf16x2 path keeps the per-column vectors resident: N <= 1024")
            lo = (W32 - Wb.float()).to(torch.bfloat16)          # exact difference in fp32, rounded once
            Wb, W32 = torch.cat([Wb, lo], dim=0).contiguous(), None
        if getattr(self, "_t3", False) and W32 is not None:
            if N > 1024:
                raise Unsupported("3xTF32 path keeps the per-column vectors resident: N <= 1024")
            hi = ((W32.view(torch.int32) + 0x1000) & -8192).view(torch.float32)   # rounded to tf32 (exact under the
            W32 = torch.cat([hi, W32 - hi], dim=0).contiguous()                   # tensor core's truncating read)
        self._keep += [t for t in (W32, Wb, bias) if t is not None]
        self._packs[C.addressof(desc)] = W32 if W32 is not None else Wb
        desc.W = W32.data_ptr() if W32 is not None else None
        desc.Wb = Wb.data_ptr() if Wb is not None else None
        desc.bias = bias.data_ptr()
        desc.N, desc.K, desc.ldw = N, K, ldw

    def _fill_affine(self, desc, Mt, in_cols, out_cols, bf16):
        """W[j, i] = A[out_cols[j], in_cols[i]], bias[j] = c[out_cols[j]]  (index -1 -> 0)."""
        N, K = out_cols.numel(), in_cols.numel()
        ldw = _round_up(K, 8)
        src_rows = torch.where(in_cols >= 0, in_cols + 1, in_cols).contiguous()
        W32, Wb = ops.pack_matrix(Mt, out_cols, src_rows, N, K, ldw, sub_row0=True, transpose_src=True,
                                  want_f32=not bf16, want_bf16=bf16 or self._b2)
        bias, _ = ops.pack_matrix(Mt[:1], None, out_cols, 1, N, N)
        self._fill_linear(desc, W32, Wb, bias.reshape(-1), N, K, ldw)

    def _fill_conditioner(self, blk, cpl, L, D, bf16):
        linears = mlp_layers(cpl.conditioner)
        cd = self.ctx_dim
        out_f = linears[-1].out_features
        additive = bool(getattr(cpl, "additive", False))
        if out_f == 2 * D and not additive:
            affine = True
        elif out_f == D or (additive and out_f in (D, 2 * D)):
            affine = False
        else:
            raise Unsupported("conditioner output width is neither D nor 2D")
        self._verify_mlp(cpl.conditioner, linears, D, cd)
        Da, Db, idx_a, idx_b = L["Da"], L["Db"], L["idx_a"], L["idx_b"]
        # the module's own first layer reads cat([context, x]) (pyro ConditionalDenseNN): activation column j of the
        # conditioning part [a | ctx] is weight column  cd + a_j  /  (j - |a|)
        first_cols = torch.where(idx_a < D, idx_a + cd, idx_a - D).to(torch.int32).contiguous()
        dev = self.device
        # tile geometry of the last layer: tiles of Cc coordinates, packed per tile as [s(Cc) | t(Cc)] (additive: [t(Cc)])
        # (Tried: tiles of 128 coordinates plus one ragged last tile -- Db = 392: 3 x 128 + 16 = 800 [s|t] columns instead of
        # 4 x 112 = 896.  The last layer of the fused kernel is bound by its coupling epilogue, not by its MMAs, and the
        # longer 128-coordinate tiles plus the hand-over of a fourth, tiny tile cost 1.3 us per launch: dropped.)
        ragged = False
        if bf16:
            cap = 128      # coords per tile: the epilogues prefetch <= 4 chunks of 16 per warp half
            nt = -(-Db // cap)
            Cc = _round_up(-(-Db // nt), 16)
        elif self._t3 or self._b2:
            cap = 128      # coords per tile: the epilogues prefetch <= 4 chunks of 16 per warp half
            nt = -(-Db // cap)
            Cc = _round_up(-(-Db // nt), 16)
        else:
            Cc = 64 if affine else 128
            nt = -(-Db // Cc)
        blk.C, blk.affine, blk.n_mlp = Cc, 1 if affine else 0, len(linears)
        t_off = D if (out_f == 2 * D) else 0        # row offset of the shift parameters in the last Linear
        self._mlp_widths[len(self._mlp_widths)] = [l.out_features for l in linears]    # block order (flops_per_row)
        tiles = []
        for ti in range(nt):
            Ct = Cc if not (ragged and ti == nt - 1) else _round_up(Db - (nt - 1) * Cc, 16)
            coord = ti * Cc + torch.arange(Ct, dtype=torch.int32, device=dev)
            valid = coord < Db
            src_b = torch.where(valid, idx_b[torch.clamp(coord, max=Db - 1).long()], torch.full_like(coord, -1))
            shifted = torch.where(valid, src_b + t_off, src_b)
            tiles.append(torch.cat([src_b, shifted]) if affine else shifted)
        rows_last = torch.cat(tiles)
        rows_last = rows_last.contiguous()

        for li, lin in enumerate(linears):
            first, last = li == 0, li == len(linears) - 1
            Wsrc = lin.weight.detach().to(device=dev, dtype=torch.float32)
            bsrc = lin.bias.detach().to(device=dev, dtype=torch.float32) if lin.bias is not None else \
                torch.zeros(lin.out_features, device=dev)
            col_idx = first_cols if first else None
            K = Da if first else lin.in_features
            if last:
                row_idx, N = rows_last, rows_last.numel()
            else:
                N = _round_up(lin.out_features, 16)
                row_idx = torch.full((N,), -1, dtype=torch.int32, device=dev)
                row_idx[:lin.out_features] = torch.arange(lin.out_features, dtype=torch.int32, device=dev)
            if K == 0:
                # no conditioning coordinate (D == 1): the conditioner sees zeros -> constant params
                K, col_idx = 1, torch.full((1,), -1, dtype=torch.int32, device=dev)
            ldw = _round_up(K, 8)
            W32, Wb = ops.pack_matrix(Wsrc, row_idx, col_idx, N, K, ldw, want_f32=not bf16, want_bf16=bf16 or self._b2)
            bias, _ = ops.pack_matrix(bsrc.reshape(-1, 1), row_idx, None, N, 1, 1)
            self._fill_linear(blk.mlp[li], W32, Wb, bias.reshape(-1), N, K, ldw)

    @staticmethod
    def _verify_mlp(cond, linears, D, cd=0):
        """The Linear chain must reproduce the module (guards against a custom forward)."""
        p = linears[0].weight
        probe = torch.linspace(-1.0, 1.0, 2 * D, device=p.device, dtype=p.dtype).reshape(2, D)
        if cd:
            ctx = torch.linspace(0.1, 0.9, 2 * cd, device=p.device, dtype=p.dtype).reshape(2, cd)
            ref = cond(probe, ctx)
        else:
            ref = cond(probe)
        if isinstance(ref, (tuple, list)):
            ref = torch.cat(list(ref), dim=-1)
        h = torch.cat([ctx, probe], dim=-1) if cd else probe
        for i, lin in enumerate(linears):
            h = torch.nn.functional.linear(h, lin.weight, lin.bias)
            if i + 1 < len(linears):
                h = torch.relu(h)
        if ref.shape != h.shape or not torch.allclose(ref, h, rtol=1e-4, atol=1e-5):
            raise Unsupported("conditioner is not equivalent to its Linear/ReLU chain")

    # -------------------------------------------------------------------------------------------
    def flops_per_row(self):
        """FLOPs one row costs in this launch chain, per kernel kind, as {kind: (executed, useful)}: `executed` counts the
        padded GEMM shapes the kernels really multiply (N, K rounded up to the tile granularity, the half-empty last
        [s|t] tile), `useful` the same GEMMs without padding.  (bench.py: roofline per kernel kind.)"""
        out = {"affine_gemm": [0, 0], "conditioner+coupling": [0, 0], "final_gemm+base": [0, 0]}
        D = self.D
        for j in range(self.desc.n_blocks):
            blk = self.blocks[j]
            out["affine_gemm"][0] += 2 * blk.G.N * blk.G.K
            out["affine_gemm"][1] += 2 * (D + self.ctx_dim) * (D + self.ctx_dim)
            o = 2 if blk.affine else 1
            for l in range(blk.n_mlp):
                lin = blk.mlp[l]
                out["conditioner+coupling"][0] += 2 * lin.N * lin.K
                n_useful = o * blk.Db if l == blk.n_mlp - 1 else self._mlp_widths[j][l]
                k_useful = blk.Da if l == 0 else self._mlp_widths[j][l - 1]
                out["conditioner+coupling"][1] += 2 * n_useful * k_useful
        out["final_gemm+base"][0] += 2 * self.G_final.N * self.G_final.K
        out["final_gemm+base"][1] += 2 * D * D
        return {k: tuple(v) for k, v in out.items()}

    @property
    def single_kernel(self):
        """True when usf_stack_run serves this stack with the one whole-stack kernel (small event shapes)."""
        return bool(lib().usf_stack_is_single_kernel(C.byref(self.desc), self.precision))

    @property
    def grad_single_kernel(self):
        """True when `run_grad` is served by the one-kernel gradient path (small event shapes at fp32)."""
        return bool(lib().usf_stack_grad_is_single_kernel(C.byref(self.desc), C.byref(self.grad_desc), self.precision))

    def run(self, x, want_logprob=False, want_y=False, want_ladj=False, deterministic=False):
        """`deterministic`: per-row sums without atomics (usf_set_deterministic): bit-identical results run to run.
        x: (B, D) fp32 CUDA -- or bf16 rows for the bf16 tier (usf_stack_run_bf16in: bit-identical to fp32 rows that
        round to them).  Returns (logprob | None, y | None, ladj | None, n_launches)."""
        if want_logprob and self.desc.base_kind < 0:
            raise _lib.USFError("this stack was compiled without a supported base distribution")
        bf16_rows = x.dtype == torch.bfloat16 and self.precision == _lib.USF_PREC_BF16
        return self._call("usf_stack_run_bf16in" if bf16_rows else "usf_stack_run", x, want_logprob, want_y, want_ladj,
                          deterministic)

    def run_terms(self, x):
        """log p(x) and its terms (usf_stack_log_prob_terms, always in the deterministic form) of rows x:(B, D + ctx_dim).
        Returns (logprob (B,), terms (n_blocks + 1, B), z (B, D), n_launches): terms[j] is block j's coupling term in
        execution order (block j inverts coupling n_blocks - 1 - j of the layer list), terms[n_blocks] the data-dependent
        part of the base log-density; logprob = desc.const_term + their sum, with const_term = base_const - logdet_const."""
        if self.desc.base_kind < 0:
            raise _lib.USFError("this stack was compiled without a supported base distribution")
        lp, z, terms, n = self._call("usf_stack_log_prob_terms", x, True, True, True, True)
        return lp, terms, z, n

    def _call(self, entry, x, want_lp, want_rows, want_ladj, deterministic):
        """One library call of `entry` on the rows x:(B, D + ctx_dim), `deterministic` mode set for it: the fp32 outputs
        it writes are a (B,) log p, (B, D) rows (y, or the gradient of usf_stack_log_prob_grad, which has no ladj) and a
        (B,) ladj -- or, for usf_stack_log_prob_terms, the (n_blocks + 1, B) terms in its place.
        -> (lp | None, rows | None, ladj | terms | None, n_launches)."""
        grad = entry == "usf_stack_log_prob_grad"
        terms = entry == "usf_stack_log_prob_terms"
        bf16_rows = entry == "usf_stack_run_bf16in"
        _lib.require_cuda(x)
        if x.dim() != 2 or x.shape[1] != self.D + self.ctx_dim:
            raise ValueError(f"expected rows of {self.D} coordinates (+ {self.ctx_dim} context columns), got shape {tuple(x.shape)}")
        if bf16_rows:
            if x.stride(1) != 1 or (x.shape[0] > 1 and x.stride(0) < x.shape[1]):
                x = x.contiguous()
            ldx = x.stride(0) if x.shape[0] > 1 else max(x.shape[1], 1)
        else:
            x, ldx = ops._rows(x)
        B, dev = x.shape[0], x.device
        lp = torch.empty(B, device=dev, dtype=torch.float32) if want_lp else None
        rows = torch.empty(B, self.D, device=dev, dtype=torch.float32) if want_rows else None
        ladj = torch.empty(*((self.desc.n_blocks + 1,) if terms else ()), B, device=dev, dtype=torch.float32) \
            if want_ladj else None
        if B == 0:
            return lp, rows, ladj, 0
        descs = (C.byref(self.desc), C.byref(self.grad_desc)) if grad else (C.byref(self.desc),)
        query = {"usf_stack_log_prob_grad": "usf_stack_grad_workspace_bytes",
                 "usf_stack_log_prob_terms": "usf_stack_terms_workspace_bytes"}.get(entry, "usf_stack_workspace_bytes")
        if grad:
            outs = (ptr(lp), ptr(rows), self.D)
        elif terms:
            outs = (ptr(lp), ptr(ladj), B, ptr(rows), self.D)
        else:
            outs = (ptr(lp), ptr(rows), self.D, ptr(ladj))
        tier = () if bf16_rows else (self.precision,)          # (usf_stack_run_bf16in runs the bf16 tier)
        L = lib()
        prev = L.usf_set_deterministic(int(bool(deterministic)))
        try:
            nbytes = getattr(L, query)(*descs, B, self.precision)
            if nbytes == 0:
                raise _lib.USFError(f"{query} failed: " + L.usf_last_error().decode())
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            n = C.c_int(0)
            check(getattr(L, entry)(*descs, ptr(x), ldx, B, *outs, ptr(ws), nbytes, *tier, C.byref(n), stream()), entry)
        finally:
            L.usf_set_deterministic(prev)
        return lp, rows, ladj, n.value

    @property
    def grad_desc(self):
        """The `usf_stack_grad_desc` of `run_grad`, built on first use from this stack's own forward packs: for a matrix
        W (N, K valid columns), W^T[:K] = W[:, :K]^T (bf16x2: the hi and the lo half each), rows K .. round_up(K, 16)
        zero, no bias.  Raises Unsupported where the gradient chain does not run."""
        if self._grad_desc is not None:
            return self._grad_desc
        if not self.inverse or self.precision not in (_lib.USF_PREC_FP32, _lib.USF_PREC_BF16X2):
            raise Unsupported("the input-gradient chain runs the inverse direction at fp32 or bf16x2")
        n = self.desc.n_blocks
        self.grad_blocks = (BlockGradDesc * max(n, 1))()
        gd = StackGradDesc()
        gd.n_blocks = n
        gd.blocks = C.cast(self.grad_blocks, C.POINTER(BlockGradDesc))
        pairs = [(gd.G_final, self.G_final)]          # (transposed, forward) descriptors
        for j in range(n):
            blk, gb = self.blocks[j], self.grad_blocks[j]
            pairs += [(gb.G, blk.G)] + [(gb.mlp[l], blk.mlp[l]) for l in range(blk.n_mlp)]
        if self._b2 and any(_round_up(F.K, 16) > 1024 for _, F in pairs):
            raise Unsupported("bf16x2 path keeps the per-column vectors resident: N <= 1024")
        for T, F in pairs:
            Kp = _round_up(F.K, 16)
            halves = self._packs[C.addressof(F)].view(-1, F.N, F.ldw)[:, :, :F.K]     # fp32 W, or bf16x2 hi and lo
            Wt = halves.new_zeros(halves.shape[0], Kp, F.N)
            Wt[:, :F.K] = halves.transpose(1, 2)
            Wt = Wt.reshape(-1, F.N)
            self._keep.append(Wt)
            T.W, T.Wb = (None, Wt.data_ptr()) if self._b2 else (Wt.data_ptr(), None)
            T.bias = None
            T.N, T.K, T.ldw = Kp, F.N, F.N
        self._grad_desc = gd
        return gd

    def run_grad(self, x, deterministic=False):
        """log p(x) and d log p(x) / dx of rows x:(B, D + ctx_dim): one kernel where `grad_single_kernel`, else the
        reverse launch chain (`grad_desc`).
        Returns (logprob (B,), grad (B, D) fp32, n_launches)."""
        lp, g, _, n = self._call("usf_stack_log_prob_grad", x, True, True, False, deterministic)
        return lp, g, n
