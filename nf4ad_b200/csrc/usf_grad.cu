// Input gradient of log p (usf_stack_log_prob_grad): the forward launch chain of usf_stack_run with every block's output
// row and hidden activations kept in per-block slots, followed by the reverse (vector-Jacobian) chain on the same GEMM
// kernels.  The reverse GEMMs are plain products with the transposed packed weights (usf_stack_grad_desc); the steps
// between them -- base-density gradient, coupling VJP, ReLU gate, pass-through residual -- are small element-wise
// kernels over the saved rows.  Nothing on the gradient is summed with atomics.  Small event shapes at fp32 take the
// one-kernel path of usf_small.cu instead (usf_small_stack_grad_kernel), as usf_stack_run takes usf_small_stack_kernel.
#include <vector>

#include "usf_common.cuh"

namespace usf {
namespace {

// rows per pass: bounds the saved state (C2 at bf16x2: ~65 KB per row with the reverse buffers, ~1.1 GB per chunk)
// while every GEMM of the chain still has >= 64 row tiles of 256 to spread over the 74 SM pairs
constexpr int64_t kGradChunkRows = 16384;

__device__ __forceinline__ float ld_op(const void* hi, const void* lo, int64_t i) {
  if (lo == nullptr) return reinterpret_cast<const float*>(hi)[i];
  return __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(hi)[i] << 16) +
         __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(lo)[i] << 16);
}

__device__ __forceinline__ void st_op(void* hi, void* lo, int64_t i, float v) {
  if (lo == nullptr) {
    reinterpret_cast<float*>(hi)[i] = v;
    return;
  }
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  reinterpret_cast<uint16_t*>(hi)[i] = __bfloat16_as_ushort(h);
  reinterpret_cast<uint16_t*>(lo)[i] = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(h)));
}

inline unsigned grid_of(int64_t total) {
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  return (unsigned)(blocks > 0 ? blocks : 1);
}

// d log p / dz of the base density for columns < D (0 in the pad columns up to `width`):
// Normal -(z - loc) inv_scale^2, Laplace -sign(z - loc) inv_scale (sign(0) = 0).
__global__ void usf_grad_base_kernel(const float* __restrict__ z, int64_t ldz, int kind, const float* __restrict__ loc,
                                     const float* __restrict__ inv_scale, int64_t D, int64_t width, Buf out, int64_t R) {
  const int64_t total = R * width;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width, c = i - r * width;
    float g = 0.f;
    if (c < D) {
      const float d = z[r * ldz + c] - loc[c];
      const float is = inv_scale[c];
      g = kind == 0 ? -d * is * is : (d > 0.f ? -is : (d < 0.f ? is : 0.f));
    }
    st_op(out.hi, out.lo, r * out.ld + c, g);
  }
}

// Coupling VJP of block j (inverse direction: x'_b = (u_b - t) e^{-ls}, ls = clamp tanh(s); additive: x'_b = u_b - t).
// st: the recomputed last conditioner layer, packed per tile as [s(C) | t(C)] ([t(C)] additive); y: the block's saved
// output row (b-part at b_off); g: dL/dx'_b on entry at b_off, dL/du_b on exit.  Writes the [ds | dt] tile operand of
// the conditioner dgrad in the same packed layout (zero for the padded coordinates >= Db).  One thread per coordinate.
__global__ void usf_grad_coupling_kernel(const float* __restrict__ st, int64_t ldst, Buf y, int b_off, float* g, int64_t ldg,
                                         Buf gst, int Db, int C, int n_tiles, int affine, float clamp, int64_t R) {
  const int64_t per_row = (int64_t)n_tiles * C;
  const int64_t total = R * per_row;
  const int W = affine ? 2 * C : C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per_row;
    const int q = (int)(i - r * per_row);
    const int tile = q / C, w = q - tile * C;
    const int64_t cs = (int64_t)tile * W + w, ct = cs + (affine ? C : 0);
    float ds = 0.f, dt = 0.f;
    if (q < Db) {
      const int64_t ig = r * ldg + b_off + q;
      const float gb = g[ig];
      if (affine) {
        const float th = tanhf(st[r * ldst + cs]);
        const float e = expf(-clamp * th);
        const float xb = ld_op(y.hi, y.lo, r * y.ld + b_off + q);
        ds = (-gb * xb - 1.f) * clamp * (1.f - th * th);     // the -1: the coupling's -sum(ls) log-det term
        dt = -gb * e;
        g[ig] = gb * e;
      } else {
        dt = -gb;
      }
    }
    if (affine) st_op(gst.hi, gst.lo, r * gst.ld + cs, ds);
    st_op(gst.hi, gst.lo, r * gst.ld + ct, dt);
  }
}

// ReLU gate of a conditioner dgrad: out = h > 0 ? gh : 0 (relu'(0) = 0), h the saved hidden activation.
__global__ void usf_grad_relu_kernel(const float* __restrict__ gh, int64_t ldgh, Buf h, int64_t N, Buf out, int64_t R) {
  const int64_t total = R * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / N, c = i - r * N;
    const float v = ld_op(h.hi, h.lo, r * h.ld + c) > 0.f ? gh[r * ldgh + c] : 0.f;
    st_op(out.hi, out.lo, r * out.ld + c, v);
  }
}

// dL/du of the whole row: the conditioning columns [0, Ka) add the conditioner's input gradient ga to their
// pass-through gradient; the rest of the row (pad, b-part) is taken as is.  out may alias g (fp32 tier).
__global__ void usf_grad_residual_kernel(const float* g, int64_t ldg, const float* __restrict__ ga, int64_t ldga, int64_t Ka,
                                         int64_t width, Buf out, int64_t R) {
  const int64_t total = R * width;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width, c = i - r * width;
    float v = g[r * ldg + c];
    if (c < Ka) v += ga[r * ldga + c];
    st_op(out.hi, out.lo, r * out.ld + c, v);
  }
}

struct GradPlan {
  int64_t ld_act, ld_hid, ld_st, ld_gh, ld_z;
  int n_hidden;   // saved hidden activations over all blocks
  int det_slots;
  size_t total;
};

int plan_grad(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int64_t rows, int precision, GradPlan* p) {
  USF_CHECK_ARG(st != nullptr && gd != nullptr && st->D > 0 && st->n_blocks >= 0 && st->ctx_dim >= 0,
                "stack grad: bad descriptor");
  USF_CHECK_ARG(st->n_blocks == 0 || (st->blocks != nullptr && gd->blocks != nullptr), "stack grad: blocks pointer is null");
  USF_CHECK_ARG(gd->n_blocks == st->n_blocks, "stack grad: %d transposed blocks for %d blocks", gd->n_blocks, st->n_blocks);
  USF_CHECK_ARG(st->inverse && st->base_kind >= 0, "stack grad: needs the inverse direction and a base distribution");
  USF_CHECK_ARG(precision == USF_PREC_FP32 || precision == USF_PREC_BF16X2,
                "stack grad: precision %d (only USF_PREC_FP32 and USF_PREC_BF16X2)", precision);
  const bool b2 = precision == USF_PREC_BF16X2;
  int64_t wmax = st->D + st->ctx_dim, hmax = 16, smax = 16;
  p->n_hidden = 0;
  p->det_slots = 0;
  for (int b = 0; b < st->n_blocks; ++b) {
    const usf_block_desc& blk = st->blocks[b];
    const usf_block_grad_desc& gb = gd->blocks[b];
    USF_CHECK_ARG(blk.n_mlp >= 1 && blk.n_mlp <= USF_MAX_MLP, "stack grad: block %d has %d conditioner layers", b, blk.n_mlp);
    USF_CHECK_ARG(gb.G.K == blk.G.N && gb.G.N >= blk.G.K, "stack grad: block %d: G^T does not match G", b);
    if (blk.G.N > wmax) wmax = blk.G.N;
    if (gb.G.N > wmax) wmax = gb.G.N;
    for (int l = 0; l < blk.n_mlp; ++l) {
      const usf_linear_desc& T = gb.mlp[l];
      USF_CHECK_ARG(T.K == blk.mlp[l].N && T.N >= blk.mlp[l].K && (b2 ? T.Wb != nullptr : T.W != nullptr),
                    "stack grad: block %d layer %d: transposed weights do not match", b, l);
      if (l + 1 < blk.n_mlp) {
        if (blk.mlp[l].N > hmax) hmax = blk.mlp[l].N;
        ++p->n_hidden;
      } else if (blk.mlp[l].N > smax) {
        smax = blk.mlp[l].N;
      }
      if (T.N > hmax) hmax = T.N;
    }
    USF_CHECK_ARG(b2 ? gb.G.Wb != nullptr : gb.G.W != nullptr, "stack grad: block %d: G^T weights missing", b);
  }
  USF_CHECK_ARG(gd->G_final.K == st->G_final.N && gd->G_final.N >= st->G_final.K &&
                    (b2 ? gd->G_final.Wb != nullptr : gd->G_final.W != nullptr), "stack grad: G_final^T does not match");
  if (st->G_final.K > wmax) wmax = st->G_final.K;
  if (gd->G_final.N > wmax) wmax = gd->G_final.N;
  if (st->G_final.N > wmax) wmax = st->G_final.N;
  if (st->G_final.N > smax) smax = st->G_final.N;      // the [ds | dt] operand buffer carries dL/dz first
  if (deterministic_mode())   // the slots of usf_stack_run's chain: the same log p, bit for bit
    for (int b = 0; b <= st->n_blocks; ++b) p->det_slots += det_slots(st, b, precision);
  p->ld_act = round_up(wmax, 16);
  p->ld_hid = round_up(hmax, 16);
  p->ld_st = round_up(smax, 16);
  p->ld_gh = p->ld_hid;
  p->ld_z = round_up(st->D, 16);
  const size_t esz = b2 ? 2 : 4, twins = b2 ? 2 : 1;
  const size_t act = align256((size_t)rows * p->ld_act * esz), hid = align256((size_t)rows * p->ld_hid * esz);
  size_t t = twins * ((size_t)(st->n_blocks + 1) * act + (size_t)p->n_hidden * hid);           // saved forward state
  t += align256((size_t)rows * p->ld_z * 4);                                                    // z
  t += 2 * align256((size_t)rows * p->ld_act * 4);                                              // dL/dx row ping-pong
  t += align256((size_t)rows * p->ld_st * 4) + twins * align256((size_t)rows * p->ld_st * esz); // [s|t] and [ds|dt]
  t += align256((size_t)rows * p->ld_gh * 4) + twins * align256((size_t)rows * p->ld_gh * esz); // hidden dgrads
  if (b2) t += twins * act;                                                                     // dL/du operand
  t += align256((size_t)p->det_slots * (size_t)rows * 4);
  p->total = t + 256;
  return USF_OK;
}

}  // namespace
}  // namespace usf

using namespace usf;

extern "C" size_t usf_stack_grad_workspace_bytes(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int64_t B,
                                                 int precision) {
  GradPlan p;
  const int64_t rows = B < kGradChunkRows ? (B > 0 ? B : 1) : kGradChunkRows;
  if (plan_grad(st, gd, rows, precision, &p) != USF_OK) return 0;
  if (small_grad_supported(st, gd, precision)) return small_grad_workspace_bytes(st, gd);
  return p.total;
}

extern "C" int usf_stack_grad_is_single_kernel(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int precision) {
  GradPlan p;
  if (plan_grad(st, gd, 1, precision, &p) != USF_OK) return 0;
  return small_grad_supported(st, gd, precision) ? 1 : 0;
}

extern "C" int usf_stack_log_prob_grad(const usf_stack_desc* st, const usf_stack_grad_desc* gd, const float* x, int64_t ldx,
                                       int64_t B, float* out_logprob, float* out_grad, int64_t ldg, void* workspace,
                                       size_t workspace_bytes, int precision, int* gpu_launches, usf_stream_t stream) {
  USF_CHECK_ARG(x != nullptr && B >= 0 && out_logprob != nullptr && out_grad != nullptr, "usf_stack_log_prob_grad: bad arguments");
  if (gpu_launches) *gpu_launches = 0;
  GradPlan p;
  const int64_t rows_max = B < kGradChunkRows ? (B > 0 ? B : 1) : kGradChunkRows;
  int rc = plan_grad(st, gd, rows_max, precision, &p);
  if (rc) return rc;
  const int64_t d_in = (int64_t)st->D + st->ctx_dim;
  USF_CHECK_ARG(ldx >= d_in && ldg >= st->D, "usf_stack_log_prob_grad: leading dimension too small");
  if (B == 0) return USF_OK;
  if (small_grad_supported(st, gd, precision)) {
    if ((rc = small_grad_run(st, gd, x, ldx, B, out_logprob, out_grad, ldg, workspace, workspace_bytes, as_stream(stream))))
      return rc;
    if (gpu_launches) *gpu_launches = 1;
    return USF_OK;
  }
  if (workspace == nullptr || workspace_bytes < p.total) {
    set_error("usf_stack_log_prob_grad: workspace too small (%zu < %zu bytes)", workspace_bytes, p.total);
    return USF_E_WORKSPACE;
  }
  cudaStream_t s = as_stream(stream);
  const bool b2 = precision == USF_PREC_BF16X2;
  const size_t esz = b2 ? 2 : 4;
  const int nb = st->n_blocks;
  const int64_t R = rows_max;

  Arena ws(workspace);
  auto op_buf = [&](int64_t ld) {   // a GEMM operand: fp32, or a (hi, lo) bf16 pair
    Buf o;
    o.ld = ld;
    o.hi = ws.take((size_t)R * ld * esz);
    o.lo = b2 ? ws.take((size_t)R * ld * esz) : nullptr;
    return o;
  };
  auto f32_buf = [&](int64_t ld) { return reinterpret_cast<float*>(ws.take((size_t)R * ld * 4)); };
  std::vector<Buf> act(nb + 1);             // act[0]: the input row; act[j + 1]: block j's output row (u, b-part coupled)
  for (int j = 0; j <= nb; ++j) act[j] = op_buf(p.ld_act);
  std::vector<Buf> hid(p.n_hidden);         // hidden activations, block-major
  for (int i = 0; i < p.n_hidden; ++i) hid[i] = op_buf(p.ld_hid);
  float* z = f32_buf(p.ld_z);
  float* gy[2] = {f32_buf(p.ld_act), f32_buf(p.ld_act)};
  float* stb = f32_buf(p.ld_st);
  Buf gst = op_buf(p.ld_st);
  float* gh = f32_buf(p.ld_gh);
  Buf gho = op_buf(p.ld_gh);
  Buf guo = b2 ? op_buf(p.ld_act) : Buf{nullptr, nullptr, p.ld_act};
  // the forward pass: usf_stack_run's chain, with every block's output row and hidden activation kept in its own slot
  ChainIO io{};
  io.act = act.data();
  io.n_act = nb + 1;
  io.hid = hid.data();
  io.n_hid = p.n_hidden;
  io.density = true;
  io.out = z;
  io.ldo = p.ld_z;
  io.acc_init = st->const_term;
  io.det = p.det_slots > 0 ? reinterpret_cast<float*>(ws.take((size_t)p.det_slots * (size_t)R * 4)) : nullptr;
  io.det_n = p.det_slots;

  int launches = 0;
  // A (rows, L.K) x L^T, N columns, into the fp32 product `ep`
  auto gemm = [&](const Buf& A, const usf_linear_desc& L, int64_t N, const EpiParams& ep, int64_t rows) -> int {
    ++launches;
    return chain_gemm(precision, A, L, rows, N, 0, ep, nullptr, nullptr, nullptr, 0, s);
  };
  auto plain = [&](float* out, int64_t ldo, int n_valid) {   // fp32 product, no bias
    EpiParams ep{};
    ep.mode = EPI_BIAS;
    ep.out = out;
    ep.ldo = ldo;
    ep.n_valid = n_valid;
    return ep;
  };

  for (int64_t r0 = 0; r0 < B; r0 += kGradChunkRows) {
    const int64_t rows = (B - r0) < kGradChunkRows ? (B - r0) : kGradChunkRows;
    io.row_acc = out_logprob + r0;
    if ((rc = run_chain(st, x + r0 * ldx, ldx, false, rows, precision, io, &launches, s))) return rc;

    // ---- reverse: dL/dz, then back through G_final^T and every block
    float* go = out_grad + r0 * ldg;
    {
      const Buf gz = gst;             // (free until the first coupling VJP)
      usf_grad_base_kernel<<<grid_of(rows * st->G_final.N), 256, 0, s>>>(z, p.ld_z, st->base_kind, st->loc, st->inv_scale,
                                                                           st->D, st->G_final.N, gz, rows);
      USF_LAUNCH_CHECK("usf_grad_base_kernel");
      ++launches;
      const usf_linear_desc& T = gd->G_final;
      if (nb == 0) rc = gemm(gz, T, b2 ? T.N : st->D, plain(go, ldg, st->D), rows);
      else rc = gemm(gz, T, T.N, plain(gy[0], p.ld_act, 0), rows);
      if (rc) return rc;
    }
    int g = 0, hi_idx = p.n_hidden;
    for (int j = nb - 1; j >= 0; --j) {
      const usf_block_desc& blk = st->blocks[j];
      const usf_block_grad_desc& gb = gd->blocks[j];
      hi_idx -= blk.n_mlp - 1;
      const int nl = blk.n_mlp;
      const usf_linear_desc& Ll = blk.mlp[nl - 1];
      // recompute [s | t] of the last conditioner layer
      const Buf in_last = nl >= 2 ? hid[hi_idx + nl - 2] : act[j + 1];
      EpiParams ep = plain(stb, p.ld_st, 0);
      ep.bias = Ll.bias;
      if ((rc = gemm(in_last, Ll, Ll.N, ep, rows))) return rc;
      const int W = blk.affine ? 2 * blk.C : blk.C;
      usf_grad_coupling_kernel<<<grid_of(rows * (Ll.N / W) * blk.C), 256, 0, s>>>(
          stb, p.ld_st, act[j + 1], blk.b_off, gy[g], p.ld_act, gst, blk.Db, blk.C, Ll.N / W, blk.affine, blk.clamp, rows);
      USF_LAUNCH_CHECK("usf_grad_coupling_kernel");
      ++launches;
      // conditioner dgrads, ReLU-gated by the saved hidden activations
      Buf a = gst;
      for (int l = nl - 1; l >= 0; --l) {
        const usf_linear_desc& T = gb.mlp[l];
        if ((rc = gemm(a, T, T.N, plain(gh, p.ld_gh, 0), rows))) return rc;
        if (l > 0) {
          const int64_t n = blk.mlp[l - 1].N;
          usf_grad_relu_kernel<<<grid_of(rows * n), 256, 0, s>>>(gh, p.ld_gh, hid[hi_idx + l - 1], n, gho, rows);
          USF_LAUNCH_CHECK("usf_grad_relu_kernel");
          ++launches;
          a = gho;
        }
      }
      // dL/du = pass-through + conditioner input gradient on [a | ctx]; the dL/du_b part was written by the VJP
      const Buf gu = b2 ? guo : Buf{gy[g], nullptr, p.ld_act};
      usf_grad_residual_kernel<<<grid_of(rows * blk.G.N), 256, 0, s>>>(gy[g], p.ld_act, gh, p.ld_gh, blk.mlp[0].K, blk.G.N,
                                                                        gu, rows);
      USF_LAUNCH_CHECK("usf_grad_residual_kernel");
      ++launches;
      // dL/dx_j = dL/du G_j: into the other gradient row, or (block 0) the caller's output, context columns dropped
      const usf_linear_desc& T = gb.G;
      if (j == 0) rc = gemm(gu, T, b2 ? T.N : st->D, plain(go, ldg, st->D), rows);
      else rc = gemm(gu, T, T.N, plain(gy[g ^ 1], p.ld_act, 0), rows);
      if (rc) return rc;
      g ^= 1;
    }
  }
  if (gpu_launches) *gpu_launches = launches;
  return USF_OK;
}
