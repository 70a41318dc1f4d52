/*
 * usflow_b200.h -- C ABI of the B200-native USFlows density path.
 *
 * This is the drop-in boundary: a plain-C shared library (libusflow_b200.so,
 * sm_100a only) that the Python mirror of the USFlows module API
 * (nf4ad_b200/, import names `src.usflows.*`) binds with ctypes.  There are no
 * torch types in any signature: raw device pointers, int64 sizes / leading
 * dimensions (in elements), a cudaStream_t passed as void*.
 *
 * Conventions
 *   - every matrix is row-major; `(B, D)` activations are fp32 with leading
 *     dimension `ld*` (elements); bf16 buffers are `uint16_t*`.
 *   - the CALLER allocates every output and workspace; the library never
 *     allocates device memory, frees, or keeps a pointer past the call.
 *   - all entry points return 0 on success, or a negative USF_E_* code;
 *     `usf_last_error()` gives the thread-local message.
 *   - every call only enqueues work on `stream` (no host sync), so the chain is
 *     CUDA-graph capturable; re-entrant across streams/threads.  The only state
 *     the library keeps is per-thread caches of things derived from ADDRESSES and
 *     shapes, never from buffer contents: encoded TMA tensor maps, and (for
 *     usf_stack_run, unless USF_GRAPHS=0) instantiated CUDA graphs of launch
 *     chains that were requested twice with identical arguments.
 *   - there is NO CPU fallback: without a CUDA device the compute entry points
 *     return USF_E_CUDA.
 *
 * "Reference interface" citations are file:line in /root/reference (nf4ad) or,
 * where the arithmetic lives in the un-vendored USFlows package, the nf4ad call
 * site that fixes the contract (see SURVEY.md section 8a/8b).
 */
#ifndef USFLOW_B200_H
#define USFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USF_VERSION 100 /* 0.1.0 */

#define USF_OK 0
#define USF_E_ARG (-1)       /* bad argument (null pointer, negative size, unsupported combination) */
#define USF_E_CUDA (-2)      /* CUDA runtime / launch error (message has cudaGetErrorString) */
#define USF_E_WORKSPACE (-3) /* caller workspace too small */
#define USF_E_UNSUPPORTED (-4)

typedef void* usf_stream_t; /* cudaStream_t */

int usf_version(void);
const char* usf_last_error(void);
/* 1 if a CUDA device with compute capability 10.x is usable by this process, else 0. */
int usf_device_ok(void);
/* A new non-blocking stream on the current device (and its release).  The host side forks the weight-space work of a
 * training step (one chain per affine run, `Flow._compose_affine_runs`) onto ~20 streams that must be DISTINCT: a
 * framework-level stream pool that hands the same stream out twice would order two chains after each other.  (The
 * host side keeps ONE such set per device for the whole process, `_lib.pooled_stream`: flows and trainers come and go.)
 * priority: 0 = default, negative = more urgent (clamped to the device's range): the batch-sized chain of the step runs
 * above the weight-space chains, and those in the order the batch will need them. */
int usf_stream_create(int priority, usf_stream_t* out);
int usf_stream_destroy(usf_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Layer kernels (fp32).  One entry point per bijector of the BaseTransform   */
/* protocol `forward / backward / log_abs_det_jacobian`                       */
/* (/root/reference/src/nf4ad/transforms.py:66-140).                          */
/* ------------------------------------------------------------------------- */

/* LUTransform parameter packing: W = (tril(L_raw,-1)+I) * triu(U_raw)  (D x D),
 * logabsdet[0] = sum_i log|U_ii|  (data-independent log-det folded into a constant).
 * Replaces USFlows LUTransform weight build; call site nf4ad/flows.py:85,110. */
int usf_lu_pack(const float* L_raw, const float* U_raw, int64_t D, float* W, float* logabsdet,
                float* scratch /* 2*D*D floats */, usf_stream_t stream);

/* y = x W^T + bias : LUTransform.forward / any dense affine map / nn.Linear.
 * relu != 0 applies max(0, .) (conditioner hidden layers, tests/conftest.py:114-118).
 * x:(B,K) ldx, W:(N,K) ldw, y:(B,N) ldy. */
int usf_linear(const float* x, int64_t ldx, const float* W, int64_t ldw, const float* bias, int relu,
               float* y, int64_t ldy, int64_t B, int64_t N, int64_t K, usf_stream_t stream);

/* x = U^{-1} L^{-1} (y - bias): LUTransform.backward as a blocked triangular solve
 * (forward substitution with unit-lower L, back substitution with U).  In place
 * (x == y) is allowed.  bias may be NULL.  transpose != 0 solves with (L U)^T instead
 * (the input-gradient of the same layer).  nf4ad/flows.py:85 -> Flow.log_prob inverse direction. */
int usf_lu_solve(const float* y, int64_t ldy, const float* L_raw, const float* U_raw, const float* bias,
                 int transpose, float* x, int64_t ldx, int64_t B, int64_t D,
                 float* scratch /* usf_lu_solve_scratch_floats(D) floats, or NULL for the slow generic kernel */,
                 usf_stream_t stream);

/* A = (L U)^{-1}, dense row-major D x D, from the raw factors (L = unit lower triangle of L_raw, U = upper triangle of
 * U_raw): what mixed-precision training applies to the batch by a GEMM instead of solving per row
 * (`LUTransform.backward`, nf4ad/flows.py:85,110 call sites).  The two triangular inverses run in one launch (identity
 * right-hand sides, half the work of a solve each), the product on the fp32 GEMM -- or, with A == NULL, left to the
 * caller: U^{-1} is then at scratch[0 .. D^2), L^{-1} at scratch[D^2 .. 2 D^2) (row-major).
 * scratch: usf_lu_inverse_scratch_floats(D) floats (0 = D not supported: use usf_lu_solve on the identity). */
int64_t usf_lu_inverse_scratch_floats(int64_t D);
int usf_lu_inverse(const float* L_raw, const float* U_raw, int64_t D, float* A, float* scratch, usf_stream_t stream);
int64_t usf_lu_solve_scratch_floats(int64_t D);

/* Product of nvs Householder reflections H_v = I - 2 v v^T/|v|^2, applied in storage
 * order (reverse != 0: last first = the inverse map).  V:(nvs,D).  nf4ad/flows.py:90. */
int usf_householder(const float* x, int64_t ldx, const float* V, int64_t nvs, int reverse, float* y,
                    int64_t ldy, int64_t B, int64_t D, usf_stream_t stream);

/* y = x * scale (inverse != 0: x / scale).  ScaleTransform, nf4ad/flows.py:113. */
int usf_scale(const float* x, int64_t ldx, const float* scale, int inverse, float* y, int64_t ldy,
              int64_t B, int64_t D, usf_stream_t stream);

/* out[0] = sum_i log|v_i| : the constant log-det of Scale / diag(U). */
int usf_sum_log_abs(const float* v, int64_t n, int64_t stride, float* out, usf_stream_t stream);

/* Masked coupling epilogue given conditioner outputs s,t:(B,D) (s == NULL: additive,
 * USFlows MaskedCoupling).  log_s = clamp*tanh(s).
 *   inverse == 0: y = m*x + (1-m)*(x*exp(log_s) + t)      nf4ad/transforms.py:66-90
 *   inverse != 0: y = m*x + (1-m)*((x - t)*exp(-log_s))   nf4ad/transforms.py:92-113
 * ladj (optional, (B,)): ladj[b] += ladj_coef * sum_d (1-m_d) log_s[b,d]   (:115-140)
 * scale_activation 0 = "exp" (above); 1 = "softplus" (:83-85,107-108,131-132): scale = softplus(log_s) + 1e-6,
 * the inverse divides by scale + 1e-12 and the log-det term is log(softplus(log_s) + 1e-12) (the reference's own
 * 1e-6 / 1e-12 inconsistency is reproduced).  In place (y == x) allowed. */
int usf_coupling(const float* x, int64_t ldx, const float* s, int64_t lds, const float* t, int64_t ldt,
                 const float* mask, float clamp, int inverse, int scale_activation, float* y, int64_t ldy,
                 float* ladj, float ladj_coef, int64_t B, int64_t D, usf_stream_t stream);

/* Base log-density summed over the event dim (Independent(base,1).log_prob):
 *   kind 0 Normal : -0.5*((z-loc)/scale)^2 - log scale - 0.5 log 2pi
 *   kind 1 Laplace: -|z-loc|/scale - log(2 scale)
 * loc:(D), scale:(scale_numel in {1,D}).  out[b] = sum_d(...) + (add ? add_coef*add[b] : 0).
 * tests/conftest.py:105-108, experiments/fashion/fashion.yaml:55-60. */
int usf_base_logprob(int kind, const float* z, int64_t ldz, const float* loc, const float* scale,
                     int64_t scale_numel, const float* add, float add_coef, float* out, int64_t B,
                     int64_t D, usf_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Training backward of the layer kernels (autograd of                        */
/* `loss = -log_prob.mean(); loss.backward()`, adbench_wrapper.py:383-386).   */
/* ------------------------------------------------------------------------- */

/* Backward of y = x W^T + b (optionally through relu, given y):
 *   dx = dy W (dx may be NULL), dW (+)= dy^T x, db (+)= colsum(dy).  accumulate != 0 adds.
 * B == 0 (dy, x, y_relu may then be NULL) still writes dW = 0 and db = 0 when accumulate == 0. */
int usf_linear_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* W,
                   int64_t ldw, const float* y_relu, int64_t ldyr, float* dx, int64_t lddx, float* dW,
                   int64_t lddw, float* db, int accumulate, float* scratch, int64_t B, int64_t N,
                   int64_t K, usf_stream_t stream);
/* bytes of `scratch` needed by usf_linear_bwd (masked dy copy when y_relu != NULL). */
size_t usf_linear_bwd_scratch_bytes(int64_t B, int64_t N);

/* Chain rule from W = L*U to the raw factors: dL_raw += strict_lower(dW U^T),
 * dU_raw += upper(L^T dW); dU_raw_ii += dlogdet / U_ii. */
int usf_lu_pack_bwd(const float* dW, const float* L_raw, const float* U_raw, float dlogdet, int64_t D,
                    float* dL_raw, float* dU_raw, float* scratch /* 3*D*D floats */,
                    usf_stream_t stream);

/* Backward of usf_scale.  `xy` is the layer INPUT x (inverse == 0) or OUTPUT y (inverse != 0);
 * dx = dy*scale (or dy/scale), dscale[d] += sum_b ... (atomic accumulate, may be NULL). */
int usf_scale_bwd(const float* dy, int64_t lddy, const float* xy, int64_t ldxy, const float* scale,
                  int inverse, float* dx, int64_t lddx, float* dscale, int64_t B, int64_t D,
                  usf_stream_t stream);

/* Operand preparation of the tensor-core (bf16) training GEMMs: one pass over the fp32 (B x N) matrix x, optionally
 * gated by a ReLU output (v = relu_mask[r,c] > 0 ? x[r,c] : 0), writes any of: `rows` (B x ldr bf16, pad columns
 * zero), `transposed` (N x ldt bf16, pad columns zero: the weight-gradient GEMM reduces over the batch) and
 * `colsum` (fp32, += column sums of v: the bias gradient; the caller zeroes it).  NULL outputs are skipped. */
int usf_to_bf16(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, uint16_t* rows, int64_t ldr,
                uint16_t* transposed, int64_t ldt, float* colsum, int64_t B, int64_t N, usf_stream_t stream);

/* The same operand pass for the 3xTF32 training GEMMs: fp32 (hi, lo) pairs (hi rounded to tf32, lo = value - hi) in
 * row-major (B x ldr) and transposed (N x ldt) form, pads zero; leading dimensions multiples of 4. */
int usf_to_tf32x3(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, float* rows_hi, float* rows_lo,
                  int64_t ldr, float* t_hi, float* t_lo, int64_t ldt, float* colsum, int64_t B, int64_t N,
                  usf_stream_t stream);

/* out[c] (+)= coef * sum_b a[b,c]  (bias gradients). */
int usf_colsum(const float* a, int64_t lda, float coef, int accumulate, float* out, int64_t B, int64_t N,
               usf_stream_t stream);

/* Plain fp32 GEMM C[M,N] (+)= opA(A) * opB(B)^T used by the backward pass:
 * a_trans == 0: A[m*lda+k], 1: A[k*lda+m];  b_trans == 0: B[n*ldb+k], 1: B[k*ldb+n]. */
int usf_gemm(const float* A, int64_t lda, int a_trans, const float* B, int64_t ldb, int b_trans, float* C,
             int64_t ldc, int accumulate, int64_t M, int64_t N, int64_t K, usf_stream_t stream);

/* Backward of usf_coupling in the direction that was run (needs the layer INPUT x, s, t):
 * produces dx, ds (NULL if additive), dt from dy and dladj (scalar per row, may be NULL). */
int usf_coupling_bwd(const float* dy, int64_t lddy, const float* dladj, float ladj_coef, const float* x,
                     int64_t ldx, const float* s, int64_t lds, const float* t, int64_t ldt,
                     const float* mask, float clamp, int inverse, int scale_activation, float* dx,
                     int64_t lddx, float* ds, int64_t ldds, float* dt, int64_t lddt, int64_t B, int64_t D,
                     usf_stream_t stream);

/* Backward of usf_householder: dx and dV (+=) from dy, given the layer input x. scratch: B*D floats * (nvs+1). */
int usf_householder_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* V,
                        int64_t nvs, int reverse, float* dx, int64_t lddx, float* dV, float* scratch,
                        int64_t B, int64_t D, usf_stream_t stream);

/* Backward of usf_base_logprob w.r.t. z (dz = dout[b] * d logp/dz) and the per-dim sums needed for
 * loc / scale gradients: dloc[d] += ..., dscale[d or 0] += ... (either may be NULL). */
int usf_base_logprob_bwd(int kind, const float* dout, const float* z, int64_t ldz, const float* loc,
                         const float* scale, int64_t scale_numel, float* dz, int64_t lddz, float* dloc,
                         float* dscale, int64_t B, int64_t D, usf_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Weight packing for the fused stack (runs once per weight version).         */
/* ------------------------------------------------------------------------- */

/* Generic gather/pack:  out[r, c] = src[row_idx[r], col_idx[c]] - (sub_row0 ? src[0, col_idx[c]] : 0)
 * (transpose_src != 0: out[r, c] = src[col_idx[c], row_idx[r]] - (sub_row0 ? src[0, row_idx[r]] : 0));
 * any index < 0 -> 0; idx == NULL -> identity.  Writes fp32 `out` (may be NULL) and/or bf16
 * `out_bf16` (may be NULL), both with leading dimension ldo; columns [n_cols, ldo) are zeroed. */
int usf_pack_matrix(const float* src, int64_t lds, const int32_t* row_idx, const int32_t* col_idx,
                    int sub_row0, int transpose_src, int64_t n_rows, int64_t n_cols, float* out,
                    uint16_t* out_bf16, int64_t ldo, usf_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Fused stack: Flow.log_prob / Flow.backward / Flow.forward(sample) as ONE    */
/* call over a packed layer-descriptor array                                   */
/* (USFlows Flow.log_prob = TransformedDistribution.log_prob; callers          */
/*  adbench_wrapper.py:383,424, vaeflow.py:201,240).                           */
/* ------------------------------------------------------------------------- */

#define USF_PREC_FP32 0 /* SIMT FFMA GEMMs, fp32 activations: log_prob rel. err <= 1e-4 tier */
#define USF_PREC_BF16 1 /* tcgen05 bf16 GEMMs (fp32 accumulate in TMEM), bf16 activations: <= 1e-2 tier */
#define USF_PREC_TF32X3 2 /* tcgen05 3xTF32 GEMMs (fp32 operands as hi + lo parts), fp32 activations: the <= 1e-4 tier on
                             tensor cores.  usf_linear_desc.W then holds 2N rows: the N fp32 rows followed by their N
                             low-part rows (W - tf32(W)); tile geometry (C) as for USF_PREC_BF16; every N <= 1024 */
#define USF_PREC_BF16X2 3 /* tcgen05 bf16 GEMMs on (hi, lo) bf16 operand pairs, 3 MMAs per K step (16 mantissa bits per
                             operand): the <= 1e-4 tier at a third of the bf16 rate -- twice the 3xTF32 rate on half its
                             operand bytes.  usf_linear_desc.Wb then holds 2N rows: the N bf16 rows followed by their N
                             low-part rows bf16(W - hi); activations travel as two bf16 buffers; every N <= 1024 */

#define USF_MAX_MLP 8

typedef struct {
  const float* W;      /* (N, ldw) fp32, K-major rows (used by USF_PREC_FP32) */
  const uint16_t* Wb;  /* same matrix in bf16 (used by USF_PREC_BF16), may be NULL */
  const float* bias;   /* (N) */
  int32_t N, K, ldw;
} usf_linear_desc;

typedef struct {
  usf_linear_desc G;   /* dense affine map applied BEFORE the coupling: u = G x + g; output columns are
                          [a-part (Da) | zero pad | b-part (Db) starting at column b_off (multiple of 16)] */
  int32_t b_off;       /* first column of the transformed (b) coordinates in the activation row */
  int32_t n_mlp;       /* conditioner Linear layers; all but the last are followed by ReLU */
  usf_linear_desc mlp[USF_MAX_MLP]; /* first: K = Da (conditioning coords); last: rows packed per tile [s(C)|t(C)] or [t(C)] */
  int32_t Da, Db;      /* |mask==1| conditioning coords, |mask==0| transformed coords; Da + Db = D */
  int32_t C;           /* coords per output tile of the last layer */
  int32_t affine;      /* 1: (s,t) affine coupling (nf4ad MaskedAffineCoupling); 0: additive (USFlows MaskedCoupling) */
  float clamp;         /* log_s = clamp * tanh(s) */
} usf_block_desc;

typedef struct {
  int32_t D;
  int32_t n_blocks;
  const usf_block_desc* blocks; /* HOST pointer to n_blocks descriptors, in execution order */
  usf_linear_desc G_final;      /* last affine map (outputs in natural coordinate order) */
  int32_t inverse;              /* 1: data -> latent direction (couplings inverted; log_prob/backward); 0: generative */
  int32_t base_kind;            /* -1: none (transform only), 0: Normal, 1: Laplace */
  const float* loc;             /* (D) */
  const float* inv_scale;       /* (D) 1/scale */
  float const_term;             /* sum of all data-independent terms (affine log-dets, -sum log scale, -D/2 log 2pi ...) */
  int32_t ctx_dim;              /* context columns appended to every input row (x:(B, D + ctx_dim)): a conditional flow's
                                   per-sample context (USFlows soft training: the noise level) travels through the chain as
                                   extra conditioning columns [a | ctx | pad | b]; 0 = unconditional */
} usf_stack_desc;

/* Workspace bytes needed to push up to B rows through the stack at the given precision. */
size_t usf_stack_workspace_bytes(const usf_stack_desc* st, int64_t B, int precision);

/* Runs the whole stack on x:(B, D + ctx_dim) fp32.
 *   out_logprob (B) : log p(x) (requires st->inverse==1 and base_kind >= 0); may be NULL
 *   out_y (B,D) ldy : transformed points (latent z if inverse, data x if generative); may be NULL
 *   out_ladj (B)    : accumulated log|det| of the applied direction (optional)
 * gpu_launches (optional host int) receives the number of kernels enqueued. */
int usf_stack_run(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob,
                  float* out_y, int64_t ldy, float* out_ladj, void* workspace, size_t workspace_bytes,
                  int precision, int* gpu_launches, usf_stream_t stream);

/* Deterministic mode of the calling thread's later usf_stack_workspace_bytes / usf_stack_run calls (returns the previous
 * setting).  Off (default): the per-row log-det / log-density terms of the tiles and warps that share a row are added
 * with fp32 atomics, whose order -- and so the last ulp of log_prob -- varies from run to run.  On: every such partial
 * sum is stored in its own slot of the workspace and one more kernel at the end of the chain adds the slots in a fixed
 * order (bit-identical results run to run, as the reference's are; a few MB of extra workspace, one extra launch, and
 * the fp32 tier's small-batch split-K GEMM form is not used).  The one-kernel path for small event shapes is always
 * deterministic. */
int usf_set_deterministic(int on);

/* 1 if usf_stack_run serves this stack at this precision with ONE whole-stack kernel (small event shapes: D + ctx_dim
 * <= 64, every layer width <= 128, fp32 weights; rows stay in shared memory across all layers, deterministic row sums),
 * 0 if it runs the launch chain. */
int usf_stack_is_single_kernel(const usf_stack_desc* st, int precision);

/* usf_stack_run (precision USF_PREC_BF16) on rows that are bf16 already: x_bf16:(B,D) with ldx in bf16 elements.  The bf16
 * tier rounds its fp32 input to bf16 (round-to-nearest-even) as its first device step, so rows narrowed the same way
 * beforehand -- usf_host_f32_to_bf16 on the host, halving the PCIe copy of a scoring call -- give bit-identical results. */
int usf_stack_run_bf16in(const usf_stack_desc* st, const uint16_t* x_bf16, int64_t ldx, int64_t B, float* out_logprob,
                         float* out_y, int64_t ldy, float* out_ladj, void* workspace, size_t workspace_bytes,
                         int* gpu_launches, usf_stream_t stream);

/* ---- input gradient of log p: log p(x) and d log p(x) / dx per row in one call ---------------------------------------
 * The reverse (vector-Jacobian) chain of an inverse-direction stack, with the weights treated as constants.  It needs
 * every matrix of the chain transposed: for a forward layer W (N x K) a `usf_linear_desc` T with T.N = round_up(K, 16)
 * rows holding W^T (zero in the padded rows), T.K = N, T.ldw = N, bias unused (NULL).  T.W (fp32) is read by
 * USF_PREC_FP32, T.Wb (2 T.N bf16 rows: hi, then lo = bf16(W^T - hi) computed from fp32) by USF_PREC_BF16X2. */
typedef struct {
  usf_linear_desc G;                  /* G_j^T */
  usf_linear_desc mlp[USF_MAX_MLP];   /* conditioner layer l transposed */
} usf_block_grad_desc;

typedef struct {
  int32_t n_blocks;                     /* == usf_stack_desc.n_blocks */
  const usf_block_grad_desc* blocks;    /* HOST pointer to n_blocks descriptors, in the stack's execution order */
  usf_linear_desc G_final;              /* G_final^T */
} usf_stack_grad_desc;

/* Workspace bytes usf_stack_log_prob_grad needs for up to B rows (0 on a bad descriptor).  Rows are processed in chunks
 * of at most 16384, so the size stops growing there. */
size_t usf_stack_grad_workspace_bytes(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int64_t B, int precision);

/* log p(x) (out_logprob, (B)) and g = d log p(x) / dx (out_grad, (B, D) with leading dimension ldg) of an inverse-direction
 * stack with a base density, x:(B, D + ctx_dim).  precision: USF_PREC_FP32 (SIMT chain) or USF_PREC_BF16X2.  A forward
 * chain that keeps every block's output row and hidden activations is followed by the reverse chain on the same GEMM
 * kernels.  No atomics touch the gradient (bit-identical run to run); out_logprob follows usf_set_deterministic as in
 * usf_stack_run and equals its result bit for bit in deterministic mode at the same precision on the launch chain.  The
 * context gradient is not formed.  gpu_launches (optional) receives the number of kernels enqueued. */
int usf_stack_log_prob_grad(const usf_stack_desc* st, const usf_stack_grad_desc* gd, const float* x, int64_t ldx, int64_t B,
                            float* out_logprob, float* out_grad, int64_t ldg, void* workspace, size_t workspace_bytes,
                            int precision, int* gpu_launches, usf_stream_t stream);

/* HOST function (no CUDA call): dst[r, c] = bf16(src[r, c]), round-to-nearest-even, NaN -> 0x7FFF -- the bit pattern the
 * device conversion produces.  src/dst are host pointers (pinned or not), leading dimensions in elements; `threads`
 * host threads of a persistent pool (<= 0: all hardware threads).  Calls are serialised. */
int usf_host_f32_to_bf16(const float* src, int64_t lds, uint16_t* dst, int64_t ldd, int64_t rows, int64_t cols,
                         int threads);

/* HOST function: the same threaded pass without narrowing -- stages pageable fp32 rows into a pinned buffer, so that the
 * PCIe copy of a caller's numpy array is asynchronous and pipelined (fp32 / tf32x3 tiers). */
int usf_host_copy_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t rows, int64_t cols, int threads);

/* ---- VAE-flow latent tail (nf4ad/vaeflow.py) -- the steps either side of flow_prior.log_prob --------------------------
 * usf_vae_reparam: z = mu + eps * exp(logvar / 2) (vaeflow.py:176-179) and, in the same pass, the posterior log-density
 *   log_q[b] = sum_c log N(z | mu, std) = sum_c (-eps^2/2 - logvar/2) - L/2 log 2pi   (vaeflow.py:214-219); log_q may be NULL.
 * usf_vae_reparam_bwd: dlogvar = dz * eps * std / 2 - dlog_q[b] / 2 (either upstream gradient may be NULL); dmu = dz.
 * usf_recon_nll: out[b] = sum (x - x_recon)^2 / (2 sigma2) + D/2 log(2 pi sigma2) over contiguous rows (vaeflow.py:208-211,
 *   255-259); usf_recon_nll_bwd: dx_recon = -dout[b] (x - x_recon) / sigma2, dx = -dx_recon (either may be NULL). */
int usf_vae_reparam(const float* mu, int64_t ldm, const float* logvar, int64_t ldv, const float* eps, int64_t lde, float* z,
                    int64_t ldz, float* log_q, int64_t B, int64_t L, usf_stream_t stream);
int usf_vae_reparam_bwd(const float* dz, int64_t lddz, const float* dlog_q, const float* eps, int64_t lde,
                        const float* logvar, int64_t ldv, float* dlogvar, int64_t lddv, int64_t B, int64_t L,
                        usf_stream_t stream);
int usf_recon_nll(const float* x, const float* x_recon, int64_t B, int64_t D, float sigma2, float* out, usf_stream_t stream);
int usf_recon_nll_bwd(const float* x, const float* x_recon, const float* dout, int64_t B, int64_t D, float sigma2,
                      float* dx_recon, float* dx, usf_stream_t stream);

/* ---- optimizer step of the training loop (adbench_wrapper.py:369,391: the Adam optimizer) -------------------------------
 * One launch per 32 parameter tensors: m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t)
 * + eps), the reference optimizer's arithmetic (weight_decay: L2 into g, or decoupled = 1 for AdamW's p *= 1 - lr wd).  `tensors` is
 * a HOST array of DEVICE pointers (contiguous fp32); step_dev is a device float holding t (already incremented), so a
 * captured step advances; grad_scale_dev (optional device float) multiplies every gradient (clipping coefficient). */
typedef struct {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
} usf_adam_tensor;
int usf_adam_step(const usf_adam_tensor* tensors, int n_tensors, const float* step_dev, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int decoupled, const float* grad_scale_dev, usf_stream_t stream);

/* SophiaG step (`src.usflows.sophia.SophiaG`, named by experiments/gmm/gaussian_mixture_standart_base.yaml:45), same tensor
 * table (`v` = the diagonal Hessian estimate h):  every hess_every-th step h = b2 h + (1-b2) g^2;  p *= 1 - lr wd;
 * m = b1 m + (1-b1) g;  p -= lr sign(m) min(|m| / (rho batch_size h + 1e-15), 1). */
int usf_sophia_step(const usf_adam_tensor* tensors, int n_tensors, const float* step_dev, float lr, float beta1, float beta2,
                    float rho, float batch_size, float weight_decay, int hess_every, const float* grad_scale_dev,
                    usf_stream_t stream);

/* Measurement only (thread-local): between usf_profile_begin and usf_profile_end every kernel that
 * usf_stack_run enqueues is bracketed by CUDA events on the launching stream.  usf_profile_end
 * synchronises and returns per-launch device milliseconds and a tag per launch
 * (0 input pack, 1 affine GEMM, 2 conditioner hidden GEMM, 3 last conditioner GEMM + coupling
 * epilogue, 4 final GEMM + base density, 5 fused conditioner chain + coupling, 6 the whole stack in one
 * kernel (small event shapes)).  ms/tags must hold
 * max_launches entries. */
int usf_profile_begin(int max_launches);
int usf_profile_end(float* ms, int* tags, int* n_out);

/* Debug: counters of the calling thread's usf_stack_run calls -- stats4 = {graph replays, successful captures,
 * failed captures, eager first sightings}; last_failure receives the reason of the last failed capture. */
int usf_debug_graph_stats(long long* stats4, char* last_failure, int failure_bytes);

/* Debug: reads (and optionally clears) the flag raised when a bounded mbarrier wait of the tcgen05
 * GEMM expired (a pipeline protocol bug); synchronises the device. */
int usf_debug_tc_timeout(int* flag, int reset);

/* 3xTF32: fp32-grade accuracy on the tensor cores.  Every fp32 operand travels as hi + lo, where hi is what the tensor
 * core sees when it reads fp32 as tf32 (low 13 mantissa bits dropped) and lo = value - hi; usf_split_lo computes lo
 * for a (rows x cols) matrix.  usf_linear_tf32x3: y = act(x W^T + bias) with three tcgen05.mma.kind::tf32 per K step
 * (x_hi W_hi + x_hi W_lo + x_lo W_hi); x, x_lo: (B, ldx), W, W_lo: (N, ldw) (ld multiples of 4, N multiple of 16 and
 * <= 1024); y fp32 and optionally its low part y_lo (NULL to skip), both with leading dimension ldy. */
int usf_split_lo(const float* x, int64_t ldx, float* lo, int64_t ldl, int64_t rows, int64_t cols, usf_stream_t stream);
int usf_linear_tf32x3(const float* x, const float* x_lo, int64_t ldx, const float* W, const float* W_lo, int64_t ldw,
                      const float* bias, int relu, float* y, float* y_lo, int64_t ldy, int64_t B, int64_t N, int64_t K,
                      usf_stream_t stream);

/* Standalone bf16 tensor-core GEMM y = act(x W^T + bias) (testing / conditioner layers):
 * x:(B,K) bf16 ldx, W:(N,K) bf16 ldw (ld multiples of 8, N multiple of 16), y:(B,N) bf16 or fp32. */
int usf_linear_bf16(const uint16_t* x, int64_t ldx, const uint16_t* W, int64_t ldw, const float* bias, int relu,
                    void* y, int64_t ldy, int y_is_bf16, int64_t B, int64_t N, int64_t K, usf_stream_t stream);

/* Name of the dominant GEMM kernel of the given precision (for profiler filters). */
const char* usf_gemm_kernel_name(int precision);

#ifdef __cplusplus
}
#endif
#endif /* USFLOW_B200_H */
