// Whole-stack kernel for small event shapes (D + context <= 64, layer widths <= 128): ONE launch runs the complete
// launch chain of usf_stack_run -- every affine map, conditioner layer, coupling update and the base log-density --
// for a tile of 64 rows that never leaves shared memory.
//
// Why: the ADBench / GMM shapes (BASELINE.json C4 D = 6..64, C1 D = 2; the reference's own test fixtures, D = 20 / 32)
// are launch-latency bound as a chain: 8-43 kernels of a few microseconds each for 28..260 bytes per row (round 1:
// 0.4 % of the HBM roofline at D = 6).  Their weights are a few KB to a few hundred KB and sit in L2; per row tile each
// layer's packed fp32 weights are staged into shared memory once and used by all 64 rows.
//
//   * arithmetic: fp32 FFMA, precise tanhf / expf -- the <= 1e-4 tier; every precision request is served by it when the
//     stack is eligible (the tensor cores have nothing to win at these widths);
//   * deterministic: a row's log-det / log-density terms are summed by one half-warp in a fixed order -- no atomics;
//   * 256 threads = 16 row groups x 16 column lanes; a thread owns a 4 x 8 register tile (rows 4 ty..+3, columns
//     tx + 16 j), operands are read as float4 along K from padded rows (conflict-free quarter-warp accesses);
//   * latency: the next layer's packed weights (and the next tile's input rows) travel into the second half of a
//     double-buffered staging area with cp.async while the current layer computes -- one __syncthreads per layer, no
//     global-memory latency on the layer-to-layer critical path; only the output columns a coupling really uses
//     (round_up(Db, 16) of s and of t out of the packed 64 + 64) are staged and multiplied;
//   * shared memory is sized from the widest layer of the stack (a few KB for D = 6 -> two CTAs per SM; ~200 KB for
//     128-wide hidden layers).
//
// Layout conventions are those of the packed descriptors (include/usflow_b200.h): activation row
// [a-part | pad | b-part at b_off], last conditioner layer packed as ONE tile [s(64) | t(64)] (affine) or [t(128)]
// (additive), final map in natural column order.
#include <algorithm>

#include "usf_common.cuh"

namespace usf {
namespace {

constexpr int SS_ROWS = 64;
constexpr int SS_THREADS = 256;
constexpr int SS_MAX_OPS = 96;
constexpr int SS_MAX_GRAD_OPS = 256;   // forward + reverse ops of the gradient kernel (kernel parameters < 32 KB)
constexpr int SS_MAXW = 128;

// SS_CVJP / SS_RPROD: reverse-pass ops of the gradient kernel (usf_small_stack_grad_kernel)
enum SsKind : int { SS_AFFINE = 0, SS_HIDDEN = 1, SS_COUPLING = 2, SS_FINAL = 3, SS_CVJP = 4, SS_RPROD = 5 };
// row buffers a reverse op names (SsOp src / dst / aux): the block's saved output row, the two activation rows (the
// gradient rows of the reverse pass), the caller's out_grad, hidden slot l at SB_HID + l
enum SsBuf : int { SB_NONE = -1, SB_SAVE = 0, SB_G0 = 1, SB_G1 = 2, SB_OUT = 3, SB_HID = 4 };

struct SsOp {
  const float* W;      // (N, ldw) fp32, K-major rows (ldw a multiple of 8, pad columns zero: usf_pack_matrix)
  const float* bias;   // (N)
  int N, K, ldw;       // N: columns this kernel computes (a coupling: 2 x Db16 (affine) / Db16 (additive))
  int kind;
  int first;           // conditioner layer whose input is the activation row (columns [0, K)) instead of the hidden buffer
  int b_off, Db, affine;
  int t_row;           // affine coupling: first packed row of the shift parameters (64)
  int woff;            // resident mode: offset (floats) of this layer's staged weights
  int boff;            // ... and of its bias from there
  float clamp;
  // gradient kernel only
  int8_t rev;          // reverse-pass op: its rows are the buffers src / dst / aux, not the forward ping-pong
  int8_t src, dst, aux;
  int8_t slot;         // block whose saved output row the op writes (forward) or reads (reverse)
  int8_t resid;        // SS_RPROD: add the product into dst columns < ncols (pass-through residual) instead of storing
  int8_t narrow;       // stage with 4-byte copies, zero columns >= K (transposed packs: ldw = forward N, any value)
  int8_t stage;        // resident mode: 0 = reads the staged weights of an earlier op (woff / boff)
  int16_t ncols;
  int16_t ksplit, kcol2;   // staged columns [0, ksplit) then [kcol2, kcol2 + K - ksplit) (0: [0, K))
};

template <int MAXOPS>
struct SsArgsT {
  int n_ops;
  int d_in;            // input columns (D + context)
  int D;
  int lda;             // shared-memory row stride of the activation buffers (floats)
  int ldh;             // ... of the hidden buffers
  int ldxs;            // ... of the input staging buffers
  int wbuf_floats;     // capacity of ONE weight staging buffer (resident mode: of the whole weight area)
  int resident;        // every layer's weights fit in shared memory together: staged once per CTA, not once per row tile
  int inverse;
  int base_kind;       // -1: none
  int x_vec;           // input rows can be fetched in 16-byte pieces
  int64_t B;
  const float* x;
  int64_t ldx;
  float* out_lp;
  float* out_y;
  int64_t ldy;
  float* out_ladj;
  float acc_init;
  const float* loc;
  const float* inv_scale;
  // gradient kernel only
  float* out_grad;
  int64_t ldgo;
  float* save;         // saved block output rows in the workspace, n_blocks x 64 x lda floats per CTA; nullptr: in smem
  int n_blocks;
  int nhs;             // hidden slots (2 for the scoring kernel)
  SsOp ops[MAXOPS];
};
using SsArgs = SsArgsT<SS_MAX_OPS>;
using SsGradArgs = SsArgsT<SS_MAX_GRAD_OPS>;
// the terms instance (usf_stack_log_prob_terms): row j < n_blocks of out_terms receives what block j adds to log p, row
// n_blocks the base log-density sum
struct SsTermsArgs : SsArgs {
  float* out_terms;
  int64_t ldt;
};

__device__ __forceinline__ float half_warp_sum(float v) {
  // the 16 column lanes of one row group are 16 consecutive lanes of a warp
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v;
}
__device__ __forceinline__ uint32_t s_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Requests one layer's weights + bias into a staging buffer (asynchronously; rows beyond N are zeroed with plain stores).
// A coupling layer only brings the rows it uses: [0, Db16) of s and [t_row, t_row + Db16) of t, packed back to back.
// A transposed pack of the gradient kernel may take its columns from two ranges (ksplit) or need 4-byte copies (narrow).
__device__ __forceinline__ void stage_op(const SsOp& op, float* wbuf, float* bbuf, int tid) {
  const int K4 = (op.K + 3) & ~3, ldw = K4 + 4, N = op.N, N16 = (N + 15) & ~15, kq = K4 >> 2;
  const int half = op.kind == SS_COUPLING && op.affine ? (N >> 1) : N;   // rows of the first (or only) source range
  if (op.narrow) {
    for (int i = tid; i < N16 * K4; i += SS_THREADS) {
      const int n = i / K4, k = i - n * K4;
      float* dst = wbuf + n * ldw + k;
      if (n < N && k < op.K) cp_async4(dst, op.W + (size_t)n * op.ldw + k);
      else *dst = 0.f;
    }
  } else {
    for (int i = tid; i < N16 * kq; i += SS_THREADS) {
      const int n = i / kq, k = (i - n * kq) << 2;
      float* dst = wbuf + n * ldw + k;
      if (n < N) {
        const int src_row = n < half ? n : op.t_row + (n - half);
        const int src_col = op.ksplit != 0 && k >= op.ksplit ? op.kcol2 + (k - op.ksplit) : k;
        cp_async16(dst, op.W + (size_t)src_row * op.ldw + src_col);
      } else {
        *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  for (int i = tid; i < N16; i += SS_THREADS) {
    if (i < N && op.bias != nullptr) cp_async4(bbuf + i, op.bias + (i < half ? i : op.t_row + (i - half)));
    else bbuf[i] = 0.f;
  }
}

// Requests the input rows of one tile into a staging buffer (columns [d_in, d4) and rows beyond the batch are zeroed).
template <class A>
__device__ __forceinline__ void stage_x(const A& args, int64_t tile, float* xbuf, int tid) {
  const int64_t row0 = tile * SS_ROWS;
  const int nrows = (int)((args.B - row0) < SS_ROWS ? (args.B - row0) : SS_ROWS);
  const int d4 = (args.d_in + 3) & ~3;
  if (args.x_vec) {
    const int q = d4 >> 2;
    for (int i = tid; i < SS_ROWS * q; i += SS_THREADS) {
      const int r = i / q, c = (i - r * q) << 2;
      float* dst = xbuf + r * args.ldxs + c;
      if (r < nrows) cp_async16(dst, args.x + (row0 + r) * args.ldx + c);
      else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
    for (int i = tid; i < SS_ROWS * d4; i += SS_THREADS) {
      const int r = i / d4, c = i - r * d4;
      float* dst = xbuf + r * args.ldxs + c;
      if (r < nrows && c < args.d_in) cp_async4(dst, args.x + (row0 + r) * args.ldx + c);
      else *dst = 0.f;
    }
  }
}

struct SsLayerCtx {
  const float* in; int ldi;
  const float* wbuf; const float* bbuf; int ldw, K4, jn;
  float* actc;        // current activation buffer (coupling: updated in place)
  float* act_out;     // the other activation buffer (affine map output)
  float* hid_out;     // hidden buffer this layer writes
  int lda, ldh;
  float* racc; const float* locs; const float* iscs;
  int64_t row0; int nrows, tx, ty;
  // gradient kernel: aux row (the gradient row of a coupling VJP, the ReLU gate of a dgrad, dL/dz of the final map)
  // and the block's saved output row
  float* aux; int ldaux;
  float* save;
};

// TERMS: a value the row's log p accumulator just took, stored into row `term` of out_terms
template <class A>
__device__ __forceinline__ void store_term(const A& args, const SsLayerCtx& cx, int term, int r, float v) {
  if (r < cx.nrows) args.out_terms[(int64_t)term * args.ldt + cx.row0 + r] = v;
}

// One layer on this thread's 4 x (16 JN) register tile: GEMM against the staged weights, then the layer's epilogue.
// GRAD: the gradient kernel's instance -- the same GEMM and forward epilogues, which also keep what the reverse pass
// reads (block output rows, dL/dz), plus the reverse epilogues.  TERMS: the terms instance -- the same arithmetic, and
// every term added to a row's log p also stored on its own (store_term).
template <int JN, bool GRAD, bool TERMS = false, class A>
__device__ __forceinline__ void ss_layer(const A& args, const SsOp& op, const SsLayerCtx& cx) {
  const int jn = cx.jn, tx = cx.tx, ty = cx.ty, lda = cx.lda;
  const float* bbuf = cx.bbuf;
  float acc[4][JN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < JN; ++j) acc[i][j] = 0.f;
  const float* arow = cx.in + (ty * 4) * cx.ldi;
  const float* wrow = cx.wbuf + tx * cx.ldw;
  for (int k = 0; k < cx.K4; k += 4) {
    float4 a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(arow + i * cx.ldi + k);
#pragma unroll
    for (int j = 0; j < JN; ++j) {
      if (JN <= 2 || j < jn) {
        const float4 w = *reinterpret_cast<const float4*>(wrow + j * 16 * cx.ldw + k);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          acc[i][j] = fmaf(a[i].x, w.x, acc[i][j]);
          acc[i][j] = fmaf(a[i].y, w.y, acc[i][j]);
          acc[i][j] = fmaf(a[i].z, w.z, acc[i][j]);
          acc[i][j] = fmaf(a[i].w, w.w, acc[i][j]);
        }
      }
    }
  }

  if (op.kind == SS_AFFINE || op.kind == SS_HIDDEN) {
    float* out = op.kind == SS_AFFINE ? cx.act_out : cx.hid_out;
    const int ldo = op.kind == SS_AFFINE ? lda : cx.ldh;
#pragma unroll
    for (int j = 0; j < JN; ++j) {
      if (j < jn) {
        const int n = tx + 16 * j;
        const float b = bbuf[n];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v = acc[i][j] + b;
          if (op.kind == SS_HIDDEN) v = fmaxf(v, 0.f);
          out[(ty * 4 + i) * ldo + n] = v;
          if (GRAD && op.kind == SS_AFFINE && !op.rev) cx.save[(ty * 4 + i) * lda + n] = v;
        }
      }
    }
  } else if (GRAD && op.kind == SS_CVJP) {
    // coupling VJP of the inverse map x'_b = (u_b - t) e^{-ls}, ls = clamp tanh(s) (additive: x'_b = u_b - t); the
    // accumulators are the recomputed s columns (affine; an additive op has K = 0).  aux: dL/dx'_b on entry, dL/du_b on
    // exit; writes [ds | dt] (affine, Db16 columns each) or [dt] into the destination row, zero for coordinates >= Db.
    constexpr int JH = JN > 4 ? 4 : JN;
#pragma unroll
    for (int j = 0; j < JH; ++j) {
      if (j < jn) {
        const int c = tx + 16 * j;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = ty * 4 + i;
          float ds = 0.f, dt = 0.f;
          if (c < op.Db) {
            float* gp = cx.aux + r * cx.ldaux + op.b_off + c;
            const float g = *gp;
            if (op.affine) {
              const float th = tanhf(acc[i][j] + bbuf[c]);
              const float e = expf(-(op.clamp * th));
              const float xb = cx.save[r * lda + op.b_off + c];
              ds = (-g * xb - 1.f) * op.clamp * (1.f - th * th);   // the -1: the coupling's -sum(ls) log-det term
              dt = -g * e;
              *gp = g * e;
            } else {
              dt = -g;
            }
          }
          if (op.affine) {
            cx.hid_out[r * cx.ldh + c] = ds;
            cx.hid_out[r * cx.ldh + 16 * jn + c] = dt;
          } else {
            cx.hid_out[r * cx.ldh + c] = dt;
          }
        }
      }
    }
  } else if (GRAD && op.kind == SS_RPROD) {
    // g_in = g_out W (the staged transposed pack): into the caller's out_grad (columns < D), added to the gradient row
    // (pass-through residual on the conditioning columns), or stored -- ReLU-gated by the hidden slot in aux
#pragma unroll
    for (int j = 0; j < JN; ++j) {
      if (j < jn) {
        const int n = tx + 16 * j;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = ty * 4 + i;
          float v = acc[i][j];
          if (op.dst == SB_OUT) {
            if (n < args.D && r < cx.nrows) args.out_grad[(cx.row0 + r) * args.ldgo + n] = v;
          } else if (op.resid) {
            if (n < op.ncols) cx.hid_out[r * cx.ldh + n] += v;
          } else {
            if (op.aux != SB_NONE) v = cx.aux[r * cx.ldaux + n] > 0.f ? v : 0.f;   // relu'(0) = 0
            cx.hid_out[r * cx.ldh + n] = v;
          }
        }
      }
    }
  } else if (op.kind == SS_COUPLING) {
    // staged columns: [s of coordinates 0..Db16) | t of the same] (affine) or [t] (additive); this thread's
    // coordinates are c = tx + 16 j
    float* u_base = cx.actc + op.b_off;
    float lsum[4] = {0.f, 0.f, 0.f, 0.f};
    const int jh = op.affine ? (jn >> 1) : jn;    // column groups of one parameter
    constexpr int JH = JN > 4 ? 4 : JN;           // (at most 64 coordinates = 4 groups)
#pragma unroll
    for (int j = 0; j < JH; ++j) {
      if (j < jh) {
        const int c = tx + 16 * j;
        if (c < op.Db) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float* up = u_base + (ty * 4 + i) * lda + c;
            const float u = *up;
            if (op.affine) {
              // the shift of coordinate group j is accumulator group j + jh (jh = 1 .. 4); indices kept in range
              const float tj = jh == 1 ? acc[i][(j + 1) % JN]
                                       : (jh == 2 ? acc[i][(j + 2) % JN] : (jh == 3 ? acc[i][(j + 3) % JN] : acc[i][(j + 4) % JN]));
              const float t = tj + bbuf[jh * 16 + c];
              // __fmul_rn / __fadd_rn: never contracted into an FMA, so both kernels instantiating this body round
              // the log-det sum alike (their log p must agree bit for bit)
              const float ls = __fmul_rn(op.clamp, tanhf(acc[i][j] + bbuf[c]));
              lsum[i] = __fadd_rn(lsum[i], ls);
              *up = args.inverse ? (u - t) * expf(-ls) : fmaf(u, expf(ls), t);
            } else {
              const float t = acc[i][j] + bbuf[c];
              *up = args.inverse ? u - t : u + t;
            }
            if (GRAD) cx.save[(ty * 4 + i) * lda + op.b_off + c] = *up;
          }
        }
      }
    }
    if (op.affine) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float s = half_warp_sum(lsum[i]);
        if (tx == 0) cx.racc[ty * 4 + i] += args.inverse ? -s : s;   // one writer per row, fixed order: deterministic
        if constexpr (TERMS)
          if (tx == 0) store_term(args, cx, op.slot, ty * 4 + i, args.inverse ? -s : s);
      }
    } else if constexpr (TERMS) {
      if (tx == 0)
        for (int i = 0; i < 4; ++i) store_term(args, cx, op.slot, ty * 4 + i, 0.f);   // an additive block adds nothing
    }
  } else {  // SS_FINAL: natural column order, optional store, optional base log-density
    float lsum[4] = {0.f, 0.f, 0.f, 0.f};
    constexpr int JF = JN > 4 ? 4 : JN;           // D <= 64
#pragma unroll
    for (int j = 0; j < JF; ++j) {
      if (j < jn) {
        const int n = tx + 16 * j;
        if (n < args.D) {
          const float b = bbuf[n], lc = cx.locs[n], is = cx.iscs[n];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = ty * 4 + i;
            const float z = acc[i][j] + b;
            if (args.out_y != nullptr && r < cx.nrows) args.out_y[(cx.row0 + r) * args.ldy + n] = z;
            const float d = __fmul_rn(z - lc, is);   // (rounded as the coupling's log-det sum above)
            lsum[i] = __fadd_rn(lsum[i], args.base_kind == 0 ? __fmul_rn(__fmul_rn(-0.5f, d), d) : -fabsf(d));
            if (GRAD) {   // dL/dz: Normal -(z - loc) / scale^2, Laplace -sign(z - loc) / scale with sign(0) = 0
              const float dz = z - lc;
              cx.aux[r * cx.ldaux + n] = args.base_kind == 0 ? -dz * is * is : (dz > 0.f ? -is : (dz < 0.f ? is : 0.f));
            }
          }
        } else if (GRAD) {
#pragma unroll
          for (int i = 0; i < 4; ++i) cx.aux[(ty * 4 + i) * cx.ldaux + n] = 0.f;
        }
      }
    }
    if (args.base_kind >= 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float s = half_warp_sum(lsum[i]);
        if (tx == 0) cx.racc[ty * 4 + i] += s;
        if constexpr (TERMS)
          if (tx == 0) store_term(args, cx, args.n_blocks, ty * 4 + i, s);
      }
    }
  }
}

// The whole-stack tile loop of both kernels.  The gradient kernel (GRAD) runs the same forward ops with the same code --
// its log p is usf_small_stack_kernel's bit for bit -- and then its reverse ops on the tile, last block first, before
// the next tile.  Shared memory: the scoring kernel's buffers (nhs hidden slots instead of 2), then, GRAD only and when
// they fit, the saved block output rows (else args.save, this CTA's part).
template <bool GRAD, bool TERMS = false, class A>
__device__ __forceinline__ void ss_body(const A& args) {
  extern __shared__ float4 smem4[];
  float* smem = reinterpret_cast<float*>(smem4);
  const int lda = args.lda, ldh = args.ldh;
  float* const act0 = smem;
  float* const act1 = act0 + SS_ROWS * lda;
  float* const hid0 = act1 + SS_ROWS * lda;
  float* const hid1 = hid0 + SS_ROWS * ldh;
  float* const xb0 = hid0 + args.nhs * SS_ROWS * ldh;
  float* const xb1 = xb0 + SS_ROWS * args.ldxs;
  float* const wb0 = xb1 + SS_ROWS * args.ldxs;
  float* const wb1 = wb0 + (args.resident ? 0 : args.wbuf_floats);
  float* const bb0 = wb0 + (args.resident ? 1 : 2) * args.wbuf_floats;
  float* const bb1 = bb0 + SS_MAXW;
  float* const racc = bb1 + SS_MAXW;
  float* const locs = racc + SS_ROWS;
  float* const iscs = locs + 64;
  float* const saved = args.save != nullptr ? args.save + (size_t)blockIdx.x * args.n_blocks * SS_ROWS * lda
                                            : iscs + 64;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t n_tiles = (args.B + SS_ROWS - 1) / SS_ROWS;
  if ((int64_t)blockIdx.x >= n_tiles) return;
  // the rows a reverse op names
  auto rbuf = [&](int id, int slot, int& ld) -> float* {
    ld = lda;
    switch (id) {
      case SB_NONE: case SB_OUT: return nullptr;
      case SB_SAVE: return saved + slot * SS_ROWS * lda;
      case SB_G0: return act0;
      case SB_G1: return act1;
      default: ld = ldh; return hid0 + (id - SB_HID) * SS_ROWS * ldh;
    }
  };

  if (tid < 64) {
    locs[tid] = (args.base_kind >= 0 && tid < args.D) ? args.loc[tid] : 0.f;
    iscs[tid] = (args.base_kind >= 0 && tid < args.D) ? args.inv_scale[tid] : 0.f;
  }
  // in flight before the first layer: this CTA's first input tile and the first layer's weights -- or, when they all
  // fit, EVERY layer's weights, which then stay for all the row tiles of this CTA
  stage_x(args, blockIdx.x, xb0, tid);
  if (args.resident) {
    for (int oi = 0; oi < args.n_ops; ++oi) {
      const SsOp& op = args.ops[oi];
      if (op.stage) stage_op(op, wb0 + op.woff, wb0 + op.woff + op.boff, tid);
    }
  } else {
    stage_op(args.ops[0], wb0, bb0, tid);
  }
  cp_async_commit();

  int sbuf = 0;   // staging buffer holding the CURRENT layer's weights
  int xsel = 0;   // staging buffer holding the CURRENT tile's input rows
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row0 = tile * SS_ROWS;
    const int nrows = (int)((args.B - row0) < SS_ROWS ? (args.B - row0) : SS_ROWS);
    if (tid < SS_ROWS) racc[tid] = args.acc_init;   // (its previous values were stored by these same threads)
    int cur = 0, hp = 0;
    for (int oi = 0; oi < args.n_ops; ++oi) {
      const SsOp& op = args.ops[oi];
      cp_async_wait_all();
      __syncthreads();   // this layer's weights (and, for the first layer, the tile's rows) have landed; the previous
                         // layer's output is complete and its weights are no longer read
      {
        // next in line: the next layer of this tile, or the first layer + the input rows of this CTA's next tile
        const bool last_op = oi + 1 == args.n_ops;
        const int64_t next_tile = tile + gridDim.x;
        if (!last_op) {
          if (!args.resident) stage_op(args.ops[oi + 1], sbuf ? wb0 : wb1, sbuf ? bb0 : bb1, tid);
        } else if (next_tile < n_tiles) {
          if (!args.resident) stage_op(args.ops[0], sbuf ? wb0 : wb1, sbuf ? bb0 : bb1, tid);
          stage_x(args, next_tile, xsel ? xb0 : xb1, tid);
        }
        cp_async_commit();
      }
      float* const actc = cur ? act1 : act0;
      const int N = op.N, K4 = (op.K + 3) & ~3, ldw = K4 + 4, N16 = (N + 15) & ~15;
      const float* wbuf = args.resident ? wb0 + op.woff : (sbuf ? wb1 : wb0);
      const float* bbuf = args.resident ? wbuf + op.boff : (sbuf ? bb1 : bb0);
      // the layer itself, compiled for 1 / 2 / 4 / 8 column groups of 16 (a 6-wide layer must not pay for the 128-wide
      // register tile: with one body predicated over 8 groups the tiny stacks were instruction-bound)
      const int jn = N16 >> 4;
      int lds;
      float* const save = GRAD ? rbuf(SB_SAVE, op.slot, lds) : nullptr;
      if (GRAD && op.rev) {
        int ldi, ldo, ldx;
        const float* in = rbuf(op.src, op.slot, ldi);
        float* const out = rbuf(op.dst, op.slot, ldo);
        float* const aux = rbuf(op.aux, op.slot, ldx);
        SsLayerCtx cx{in, ldi, wbuf, bbuf, ldw, K4, jn, nullptr, nullptr, out, lda, ldo,
                      racc, locs, iscs, row0, nrows, tx, ty, aux, ldx, save};
        if (jn <= 1) ss_layer<1, GRAD, TERMS>(args, op, cx);
        else if (jn == 2) ss_layer<2, GRAD, TERMS>(args, op, cx);
        else if (jn <= 4) ss_layer<4, GRAD, TERMS>(args, op, cx);
        else ss_layer<8, GRAD, TERMS>(args, op, cx);
      } else {
        const float* in;
        int ldi = lda;
        if (oi == 0) { in = xsel ? xb1 : xb0; ldi = args.ldxs; }
        else if (op.kind == SS_AFFINE || op.kind == SS_FINAL || op.first) in = actc;
        else { in = hp ? hid1 : hid0; ldi = ldh; }
        SsLayerCtx cx{in, ldi, wbuf, bbuf, ldw, K4, jn, actc, cur ? act0 : act1, (op.first || hp) ? hid0 : hid1, lda, ldh,
                      racc, locs, iscs, row0, nrows, tx, ty, cur ? act0 : act1, lda, save};   // (aux: dL/dz of the final op)
        if (jn <= 1) ss_layer<1, GRAD, TERMS>(args, op, cx);
        else if (jn == 2) ss_layer<2, GRAD, TERMS>(args, op, cx);
        else if (jn <= 4) ss_layer<4, GRAD, TERMS>(args, op, cx);
        else ss_layer<8, GRAD, TERMS>(args, op, cx);
        if (op.kind == SS_AFFINE) cur ^= 1;
        else if (op.kind == SS_HIDDEN) hp = (op.first || hp) ? 0 : 1;
        else if (op.kind == SS_COUPLING) hp = 0;
      }
      sbuf ^= 1;
    }
    xsel ^= 1;
    __syncthreads();
    if (tid < nrows) {
      if (args.out_lp != nullptr) args.out_lp[row0 + tid] = racc[tid];
      if (args.out_ladj != nullptr) args.out_ladj[row0 + tid] = racc[tid];
    }
  }
  cp_async_wait_all();
}

__global__ void __launch_bounds__(SS_THREADS, 2) usf_small_stack_kernel(const __grid_constant__ SsArgs args) {
  ss_body<false>(args);
}

// usf_small_stack_kernel that also stores the terms of log p (usf_stack_log_prob_terms)
__global__ void __launch_bounds__(SS_THREADS, 2) usf_small_stack_terms_kernel(const __grid_constant__ SsTermsArgs args) {
  ss_body<false, true>(args);
}

// log p and d log p / dx of a tile in one launch: the forward ops of usf_small_stack_kernel, then the reverse ops.
__global__ void __launch_bounds__(SS_THREADS, 2) usf_small_stack_grad_kernel(const __grid_constant__ SsGradArgs args) {
  ss_body<true>(args);
}

bool small_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("USF_SMALL_STACK"); on = (e != nullptr && e[0] == '0') ? 0 : 1; }
  return on == 1;
}

// Weight offsets of resident mode and the staging capacity: all layers resident when they fit in `budget` bytes beside
// the row buffers (then no weight travels per row tile), else one double-buffered layer at a time.
template <class A>
void layout_weights(A* a, size_t budget) {
  int total = 0, maxwb = 0;
  for (int i = 0; i < a->n_ops; ++i) {
    SsOp& o = a->ops[i];
    const int n16 = (o.N + 15) & ~15, w = n16 * (((o.K + 3) & ~3) + 4);
    if (w > maxwb) maxwb = w;
    if (!o.stage) continue;
    o.woff = total;
    o.boff = w;
    total += w + n16;
  }
  a->resident = (size_t)total * sizeof(float) <= budget ? 1 : 0;
  a->wbuf_floats = a->resident ? ((total + 3) & ~3) : ((maxwb + 3) & ~3);
}

// Fills `a` from the descriptor; false when the stack is not one this kernel runs.
template <class A>
bool build_args(const usf_stack_desc* st, A* a) {
  if (st == nullptr || st->D <= 0 || st->D + st->ctx_dim > 64 || st->n_blocks < 0) return false;
  int n = 0, maxa = 16, maxh = 16;
  auto aligned = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  // stored: 0 = the output stays in registers (coupling, final), 1 = activation buffer, 2 = hidden buffer;
  // in_hidden: the layer reads the hidden buffer
  auto push = [&](const usf_linear_desc& L, int N, int kind, int first, const usf_block_desc* blk, int stored, bool in_hidden) -> bool {
    if (n >= SS_MAX_OPS || L.W == nullptr || !aligned(L.W) || (L.ldw & 3) != 0 || N <= 0 || N > SS_MAXW || L.K <= 0 ||
        L.K > SS_MAXW || L.ldw < ((L.K + 3) & ~3))
      return false;
    SsOp& o = a->ops[n++];
    o = SsOp{};
    o.W = L.W; o.bias = L.bias; o.N = N; o.K = L.K; o.ldw = L.ldw; o.kind = kind; o.first = first;
    o.b_off = blk ? blk->b_off : 0; o.Db = blk ? blk->Db : 0; o.affine = blk ? blk->affine : 0; o.clamp = blk ? blk->clamp : 0.f;
    o.t_row = 64;
    o.slot = (int8_t)(blk ? blk - st->blocks : 0);
    o.stage = 1;
    o.src = o.dst = o.aux = SB_NONE;
    const int n16 = (N + 15) & ~15, k4 = (L.K + 3) & ~3;
    if (stored == 1 && n16 > maxa) maxa = n16;
    if (stored == 2 && n16 > maxh) maxh = n16;
    if (in_hidden) { if (k4 > maxh) maxh = k4; } else { if (k4 > maxa) maxa = k4; }
    return true;
  };
  for (int b = 0; b < st->n_blocks; ++b) {
    const usf_block_desc& blk = st->blocks[b];
    if (blk.n_mlp < 1 || blk.n_mlp > USF_MAX_MLP) return false;
    if (!push(blk.G, blk.G.N, SS_AFFINE, 0, &blk, 1, false)) return false;
    if (blk.b_off + blk.Db > blk.G.N || blk.Db <= 0 || blk.Db > 64 || blk.mlp[0].K > blk.b_off) return false;
    for (int l = 0; l < blk.n_mlp; ++l) {
      const bool last = l == blk.n_mlp - 1;
      if (!last) {
        if (!push(blk.mlp[l], blk.mlp[l].N, SS_HIDDEN, l == 0 ? 1 : 0, &blk, 2, l > 0)) return false;
        continue;
      }
      // the coupling tile must be the single [s(64) | t(64)] / [t(128)] tile of the fp32 packing; only the
      // round_up(Db, 16) columns of each parameter that carry coordinates are computed
      if (blk.mlp[l].N != 128 || blk.C != (blk.affine ? 64 : 128)) return false;
      const int db16 = (blk.Db + 15) & ~15;
      if (!push(blk.mlp[l], blk.affine ? 2 * db16 : db16, SS_COUPLING, l == 0 ? 1 : 0, &blk, 0, l > 0)) return false;
    }
  }
  if (st->G_final.N < st->D) return false;
  if (!push(st->G_final, st->D, SS_FINAL, 0, nullptr, 0, false)) return false;
  a->n_ops = n;
  a->lda = maxa + 4;
  a->ldh = maxh + 4;
  a->ldxs = ((st->D + st->ctx_dim + 3) & ~3) + 4;
  a->nhs = 2;
  a->save = nullptr;
  a->n_blocks = st->n_blocks;
  layout_weights(a, 96 * 1024);
  return true;
}

template <class A>
size_t smem_bytes(const A& a, bool saved_in_smem = false) {
  return sizeof(float) * ((size_t)2 * SS_ROWS * a.lda + (size_t)a.nhs * SS_ROWS * a.ldh + (size_t)2 * SS_ROWS * a.ldxs +
                          (size_t)(a.resident ? 1 : 2) * a.wbuf_floats + 2 * SS_MAXW + SS_ROWS + 128 +
                          (saved_in_smem ? (size_t)a.n_blocks * SS_ROWS * a.lda : 0));
}

// ---- the gradient kernel's arguments: the forward ops of build_args, then per block (last first) the reverse ops
//   hidden layers recomputed from the saved row into hidden slots 0 .. n_mlp - 2 (the forward ops themselves: the same
//   staged weights and code, so the ReLU gates and s are bitwise the forward pass's);
//   the coupling VJP (s columns only; additive: no product) writing [ds | dt] into the free activation row;
//   the conditioner dgrads with the transposed packs, each ReLU-gated by a hidden slot and written over it in place (a
//   thread reads its gate element, then stores the gradient there); the first layer's product is added to the
//   gradient row (pass-through residual on the conditioning columns);
//   the G^T product into the other activation row -- or, for block 0, the caller's out_grad.
// Before the blocks: G_final^T on dL/dz, which the final op leaves in the activation row it does not read.
// So the reverse pass needs no row buffers beyond the scoring kernel's, except hidden slots when n_mlp > 3.
constexpr size_t kGradResidentBytes = 96 * 1024;
constexpr int kGradSavedCtasPerSm = 2;   // CTAs per SM the workspace holds saved rows for (the launch is capped there)

struct GradLayout {
  bool saved_in_smem;
  size_t smem;
};

// `T` transposed from the forward `F` as usf_stack_grad_desc defines it; fills a reverse product op reading K columns.
bool push_transposed(SsGradArgs* a, int& n, const usf_linear_desc& T, const usf_linear_desc& F, int K) {
  if (n >= SS_MAX_GRAD_OPS || T.W == nullptr || T.N != ((F.K + 15) & ~15) || T.K != F.N || T.ldw != F.N || T.N > SS_MAXW ||
      K <= 0 || K > T.K)
    return false;
  SsOp& o = a->ops[n++];
  o = SsOp{};
  o.W = T.W; o.bias = nullptr; o.N = T.N; o.K = K; o.ldw = T.ldw; o.kind = SS_RPROD;
  o.rev = 1; o.stage = 1;
  o.src = o.dst = o.aux = SB_NONE;
  o.narrow = ((reinterpret_cast<uintptr_t>(T.W) & 15) != 0 || (T.ldw & 3) != 0 || (K & 3) != 0) ? 1 : 0;
  return true;
}

bool build_grad_args(const usf_stack_desc* st, const usf_stack_grad_desc* gd, SsGradArgs* a, GradLayout* L) {
  if (gd == nullptr || gd->n_blocks != st->n_blocks || (st->n_blocks > 0 && gd->blocks == nullptr) || !st->inverse ||
      st->base_kind < 0 || !build_args(st, a))
    return false;
  const int nb = st->n_blocks;
  int n = a->n_ops, ldg = std::max(a->lda - 4, (st->D + 15) & ~15), ldh = a->ldh - 4, nhs = 2;
  auto r16 = [](int v) { return (v + 15) & ~15; };
  auto r4 = [](int v) { return (v + 3) & ~3; };
  auto other = [](int id) { return id == SB_G0 ? SB_G1 : SB_G0; };
  // after the forward ops the final op's input is activation row nb % 2 (every affine op flips it), dL/dz the other
  int g = (nb & 1) ? SB_G1 : SB_G0;
  if (!push_transposed(a, n, gd->G_final, st->G_final, st->D)) return false;
  a->ops[n - 1].src = other(g);
  a->ops[n - 1].dst = nb == 0 ? SB_OUT : g;
  int written = r16(st->G_final.K);       // columns of the gradient row the last product wrote
  ldg = std::max(ldg, written);
  int f0 = a->n_ops - 1;                  // f0: first forward op of the block (walking back)
  for (int j = nb - 1; j >= 0; --j) {
    const usf_block_desc& blk = st->blocks[j];
    const usf_block_grad_desc& gb = gd->blocks[j];
    const int nm = blk.n_mlp, db16 = r16(blk.Db);
    f0 -= 1 + nm;
    if (r4(blk.G.N) > written) return false;   // the G^T product reads columns its producer did not write
    nhs = std::max(nhs, nm - 1);
    for (int l = 0; l + 1 < nm; ++l) {          // hidden layers, recomputed
      if (n >= SS_MAX_GRAD_OPS) return false;
      SsOp& o = a->ops[n++];
      o = a->ops[f0 + 1 + l];
      o.rev = 1; o.stage = 0;
      o.src = l == 0 ? SB_SAVE : SB_HID + l - 1;
      o.dst = SB_HID + l;
      o.aux = SB_NONE;
    }
    {                                           // coupling VJP
      if (n >= SS_MAX_GRAD_OPS) return false;
      SsOp& o = a->ops[n++];
      o = a->ops[f0 + nm];
      o.kind = SS_CVJP;
      o.rev = 1;
      o.N = db16;                               // s rows only (the first Db16 rows of the forward op's staged tile)
      o.stage = 0;
      if (!blk.affine) { o.K = 0; o.W = nullptr; o.bias = nullptr; o.woff = 0; o.boff = 0; }   // nothing to multiply
      o.src = nm >= 2 ? SB_HID + nm - 2 : SB_SAVE;
      o.dst = other(g);
      o.aux = g;
      ldg = std::max(ldg, blk.affine ? 2 * db16 : db16);
    }
    for (int l = nm - 1; l >= 0; --l) {         // conditioner dgrads
      const usf_linear_desc& F = blk.mlp[l];
      const int K = l == nm - 1 ? (blk.affine ? 2 * db16 : db16) : F.N;
      if (l < nm - 1 && r4(F.N) > r16(blk.mlp[l + 1].K)) return false;
      if (!push_transposed(a, n, gb.mlp[l], F, K)) return false;
      SsOp& o = a->ops[n - 1];
      if (l == nm - 1 && blk.affine) { o.ksplit = (int16_t)db16; o.kcol2 = (int16_t)blk.C; }
      if (l == nm - 1 && o.narrow) return false;   // (the coupling tile's pack is 128 wide: never narrow)
      o.src = l == nm - 1 ? other(g) : SB_HID + l;
      o.slot = (int8_t)j;
      if (l > 0) {
        o.dst = o.aux = SB_HID + l - 1;
        ldh = std::max(ldh, (int)o.N);
      } else {
        o.dst = g;
        o.resid = 1;
        o.ncols = (int16_t)F.K;
      }
    }
    // G_j^T: into the other gradient row, or the caller's out_grad
    if (!push_transposed(a, n, gb.G, blk.G, blk.G.N)) return false;
    SsOp& o = a->ops[n - 1];
    o.src = g;
    o.dst = j == 0 ? SB_OUT : other(g);
    o.slot = (int8_t)j;
    written = r16(blk.G.K);
    ldg = std::max(ldg, written);
    g = other(g);
  }
  // the adjustments below only change row strides and weight placement, never what a forward op computes
  a->n_ops = n;
  a->lda = ldg + 4;
  a->ldh = ldh + 4;
  a->nhs = nhs;
  a->n_blocks = nb;
  layout_weights(a, kGradResidentBytes);
  L->saved_in_smem = smem_bytes(*a, true) <= 227 * 1024;
  L->smem = smem_bytes(*a, L->saved_in_smem);
  return L->smem <= 227 * 1024;
}

size_t grad_saved_bytes(const SsGradArgs& a, const GradLayout& L) {
  return L.saved_in_smem ? 0
                         : (size_t)num_sms() * kGradSavedCtasPerSm * a.n_blocks * SS_ROWS * a.lda * sizeof(float);
}

}  // namespace

bool small_stack_supported(const usf_stack_desc* st, int precision) {
  if (precision != USF_PREC_FP32 || !small_enabled()) return false;
  static thread_local SsArgs probe;
  return build_args(st, &probe) && smem_bytes(probe) <= 227 * 1024;
}

bool small_grad_supported(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int precision) {
  if (!small_stack_supported(st, precision)) return false;
  static thread_local SsGradArgs probe;
  GradLayout L;
  return build_grad_args(st, gd, &probe, &L);
}

size_t small_grad_workspace_bytes(const usf_stack_desc* st, const usf_stack_grad_desc* gd) {
  static thread_local SsGradArgs a;
  GradLayout L;
  if (!build_grad_args(st, gd, &a, &L)) return 0;
  return 256 + grad_saved_bytes(a, L);
}

// The scoring launch of `kernel` (its own shared-memory attribute, set once per thread: one flag per instance of A).
template <class A>
int small_launch(void (*kernel)(A), const A& a, int64_t B, const char* name, cudaStream_t stream) {
  const size_t smem = smem_bytes(a);
  static thread_local bool attr_set = false;
  if (smem > 48 * 1024 && !attr_set) {
    USF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
    attr_set = true;
  }
  int per_sm = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, SS_THREADS, smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    per_sm = 1;
  }
  const int64_t tiles = ceil_div(B, SS_ROWS);
  int64_t grid = (int64_t)num_sms() * per_sm;
  if (grid > tiles) grid = tiles;
  kernel<<<(unsigned)grid, SS_THREADS, smem, stream>>>(a);
  const cudaError_t e = cudaGetLastError();
  return e != cudaSuccess ? cuda_fail(e, name) : USF_OK;
}

int small_stack_run(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob, float* out_y,
                    int64_t ldy, float* out_ladj, float* out_terms, int64_t ldt, cudaStream_t stream) {
  static thread_local SsTermsArgs a;
  USF_CHECK_ARG(build_args(st, &a), "small_stack_run: unsupported stack");
  const bool density = out_logprob != nullptr || out_terms != nullptr;
  a.d_in = st->D + st->ctx_dim;
  a.D = st->D;
  a.inverse = st->inverse;
  a.base_kind = density ? st->base_kind : -1;
  a.B = B;
  a.x = x;
  a.ldx = ldx;
  a.x_vec = ((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx & 3) == 0 && (a.d_in & 3) == 0) ? 1 : 0;
  a.out_lp = out_logprob;
  a.out_y = out_y;
  a.ldy = ldy;
  a.out_ladj = out_ladj;
  a.acc_init = density ? st->const_term : 0.f;
  a.loc = st->loc;
  a.inv_scale = st->inv_scale;
  a.out_terms = out_terms;
  a.ldt = ldt;
  if (out_terms != nullptr)
    return small_launch(usf_small_stack_terms_kernel, static_cast<const SsTermsArgs&>(a), B,
                        "launch of usf_small_stack_terms_kernel", stream);
  return small_launch(usf_small_stack_kernel, static_cast<const SsArgs&>(a), B, "launch of usf_small_stack_kernel", stream);
}

int small_grad_run(const usf_stack_desc* st, const usf_stack_grad_desc* gd, const float* x, int64_t ldx, int64_t B,
                   float* out_logprob, float* out_grad, int64_t ldg, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream) {
  static thread_local SsGradArgs a;
  GradLayout L;
  USF_CHECK_ARG(build_grad_args(st, gd, &a, &L), "small_grad_run: unsupported stack");
  const size_t need = 256 + grad_saved_bytes(a, L);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("usf_stack_log_prob_grad: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    return USF_E_WORKSPACE;
  }
  a.d_in = st->D + st->ctx_dim;
  a.D = st->D;
  a.inverse = 1;
  a.base_kind = st->base_kind;
  a.B = B;
  a.x = x;
  a.ldx = ldx;
  a.x_vec = ((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx & 3) == 0 && (a.d_in & 3) == 0) ? 1 : 0;
  a.out_lp = out_logprob;
  a.out_y = nullptr;
  a.ldy = 0;
  a.out_ladj = nullptr;
  a.acc_init = st->const_term;
  a.loc = st->loc;
  a.inv_scale = st->inv_scale;
  a.out_grad = out_grad;
  a.ldgo = ldg;
  a.save = L.saved_in_smem ? nullptr : static_cast<float*>(Arena(workspace).take(0));
  static thread_local bool attr_set = false;
  if (L.smem > 48 * 1024 && !attr_set) {
    USF_CUDA(cudaFuncSetAttribute(usf_small_stack_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(227 * 1024)));
    attr_set = true;
  }
  int per_sm = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, usf_small_stack_grad_kernel, SS_THREADS, L.smem) != cudaSuccess ||
      per_sm < 1) {
    cudaGetLastError();
    per_sm = 1;
  }
  if (!L.saved_in_smem && per_sm > kGradSavedCtasPerSm) per_sm = kGradSavedCtasPerSm;
  const int64_t tiles = ceil_div(B, SS_ROWS);
  int64_t grid = (int64_t)num_sms() * per_sm;
  if (grid > tiles) grid = tiles;
  usf_small_stack_grad_kernel<<<(unsigned)grid, SS_THREADS, L.smem, stream>>>(a);
  USF_LAUNCH_CHECK("usf_small_stack_grad_kernel");
  return USF_OK;
}

}  // namespace usf
