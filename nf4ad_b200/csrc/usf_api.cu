// Host side of the C ABI: error plumbing, device probe, and the fused-stack runner that turns a packed
// layer-descriptor array into one launch chain (Flow.log_prob / Flow.backward / Flow.forward).
#include <stdarg.h>
#include <stdlib.h>

#include <vector>

#include "usf_common.cuh"

namespace usf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return USF_E_CUDA;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

namespace {

// Measurement-only, thread-local: when enabled, usf_stack_run brackets every kernel it enqueues with
// CUDA events on the launching stream so bench.py can report the per-launch device time of each kernel.
struct Profile {
  bool on = false;
  int cap = 0;
  int n = 0;
  cudaEvent_t* ev = nullptr;  // 2 events per launch
  int* tag = nullptr;
};
thread_local Profile g_prof;

struct ProfScope {
  cudaStream_t s;
  int idx;
  ProfScope(cudaStream_t st, int tag) : s(st), idx(-1) {
    if (g_prof.on && g_prof.n < g_prof.cap) {
      idx = g_prof.n++;
      g_prof.tag[idx] = tag;
      cudaEventRecord(g_prof.ev[2 * idx], s);
    }
  }
  ~ProfScope() {
    if (idx >= 0) cudaEventRecord(g_prof.ev[2 * idx + 1], s);
  }
};

struct StackPlan {
  int64_t ld_act;     // activation leading dimension (elements)
  int64_t ld_hid;     // hidden leading dimension (elements)
  size_t act_bytes;   // one activation buffer for `rows` rows
  size_t hid_bytes;
  size_t acc_bytes;
  size_t small_bytes;  // fp32 path: split-K accumulator for small batches (rows <= kSmallRows)
  int det_slots;       // deterministic mode: partial-sum slots of one pass over the chain
  size_t det_bytes;
  size_t total;
};

// partial-sum slots one accumulating launch uses (the `sub` range of row_accumulate in its kernel)
inline int det_slots_of(int precision, int64_t N, int bn, bool fused) {
  if (fused) return 4;                                                       // MLP_EPI_PARTS warps per row
  if (precision == USF_PREC_FP32) return (int)ceil_div(N, 128);              // SIMT tile: 128 columns per blockIdx.y
  return 2 * (int)ceil_div(N, bn);                                           // tcgen05 kernels: 2 epilogue warps per N tile
}

// Deterministic mode (usf_set_deterministic, per thread): every per-row partial sum of the chain goes to its own slot of
// a scratch area and one last kernel adds the slots in order, instead of fp32 atomics whose order varies run to run.
thread_local int g_deterministic = 0;

}  // namespace

int deterministic_mode() { return g_deterministic; }

namespace {

constexpr int64_t kChunkRows = 131072;  // rows pushed through the stack per pass (bounds the workspace)
constexpr int64_t kSmallRows = 2048;    // fp32 path: batches up to this size may use the split-K + epilogue-kernel GEMM form

inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

int plan_stack(const usf_stack_desc* st, int64_t rows, int precision, StackPlan* p) {
  USF_CHECK_ARG(st != nullptr && st->D > 0 && st->n_blocks >= 0 && st->ctx_dim >= 0, "stack: bad descriptor");
  USF_CHECK_ARG(st->n_blocks == 0 || st->blocks != nullptr, "stack: blocks pointer is null");
  USF_CHECK_ARG(precision == USF_PREC_FP32 || precision == USF_PREC_BF16 || precision == USF_PREC_TF32X3 ||
                    precision == USF_PREC_BF16X2, "stack: unknown precision %d", precision);
  int64_t wmax = st->D + st->ctx_dim, hmax = 16, nmax = st->G_final.N;
  for (int b = 0; b < st->n_blocks; ++b) {
    const usf_block_desc& blk = st->blocks[b];
    USF_CHECK_ARG(blk.n_mlp >= 1 && blk.n_mlp <= USF_MAX_MLP, "stack: block %d has %d conditioner layers", b, blk.n_mlp);
    if (blk.G.N > wmax) wmax = blk.G.N;
    if (blk.G.K > wmax) wmax = blk.G.K;
    if (blk.G.N > nmax) nmax = blk.G.N;
    for (int l = 0; l < blk.n_mlp; ++l) {
      if (l + 1 < blk.n_mlp && blk.mlp[l].N > hmax) hmax = blk.mlp[l].N;
      if (blk.mlp[l].N > nmax) nmax = blk.mlp[l].N;
    }
  }
  if (st->G_final.K > wmax) wmax = st->G_final.K;
  const size_t esz = (precision == USF_PREC_BF16 || precision == USF_PREC_BF16X2) ? 2 : 4;
  p->ld_act = round_up(wmax, 16);
  p->ld_hid = round_up(hmax, 16);
  p->act_bytes = align256((size_t)rows * p->ld_act * esz);
  p->hid_bytes = align256((size_t)rows * p->ld_hid * esz);
  p->acc_bytes = align256((size_t)rows * sizeof(float));
  p->small_bytes = (precision == USF_PREC_FP32 && rows <= kSmallRows && !g_deterministic)
                       ? align256((size_t)rows * (size_t)nmax * sizeof(float)) : 0;   // (split-K sums atomically: not in deterministic mode)
  p->det_slots = 0;
  if (g_deterministic) {
    const bool tc = precision != USF_PREC_FP32;
    for (int b = 0; b < st->n_blocks; ++b) {
      const usf_block_desc& blk = st->blocks[b];
      if (!blk.affine) continue;                                  // additive couplings add nothing to the row sums
      const usf_linear_desc& L = blk.mlp[blk.n_mlp - 1];
      p->det_slots += tc ? (2 * (int)ceil_div(L.N, 2 * blk.C) > 4 ? 2 * (int)ceil_div(L.N, 2 * blk.C) : 4)
                         : det_slots_of(precision, L.N, 0, false);
    }
    p->det_slots += tc ? det_slots_of(precision, st->G_final.N, tc_pick_bn(st->G_final.N), false)
                       : det_slots_of(precision, st->D, 0, false);
  }
  p->det_bytes = align256((size_t)p->det_slots * (size_t)rows * sizeof(float));
  // 3xTF32 / bf16x2: every activation buffer has a low-part twin
  const size_t twins = (precision == USF_PREC_TF32X3 || precision == USF_PREC_BF16X2) ? 2 : 1;
  p->total = twins * (2 * p->act_bytes + 2 * p->hid_bytes) + p->acc_bytes + p->small_bytes + p->det_bytes + 256;
  return USF_OK;
}

}  // namespace
}  // namespace usf

using namespace usf;

extern "C" int usf_version(void) { return USF_VERSION; }

extern "C" int usf_stream_create(int priority, usf_stream_t* out) {
  USF_CHECK_ARG(out != nullptr, "usf_stream_create: null output");
  int least = 0, greatest = 0;          // numerically: greatest priority <= least priority
  USF_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
  if (priority < greatest) priority = greatest;
  if (priority > least) priority = least;
  cudaStream_t s = nullptr;
  USF_CUDA(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, priority));
  *out = reinterpret_cast<usf_stream_t>(s);
  return USF_OK;
}

extern "C" int usf_stream_destroy(usf_stream_t stream) {
  if (stream != nullptr) USF_CUDA(cudaStreamDestroy(reinterpret_cast<cudaStream_t>(stream)));
  return USF_OK;
}
extern "C" const char* usf_last_error(void) { return g_err; }

extern "C" int usf_device_ok(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return 0;
  }
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

extern "C" const char* usf_gemm_kernel_name(int precision) {
  return precision == USF_PREC_BF16 ? kTcGemmKernelName : kSimtGemmKernelName;
}

extern "C" int usf_debug_tc_timeout(int* flag, int reset) { return tc_timeout_flag(flag, reset); }

extern "C" int usf_debug_tc_trace(int on, unsigned long long* out, int max_records) {
  return tc_trace_ctl(on, out, max_records);
}

extern "C" int usf_linear_bf16(const uint16_t* x, int64_t ldx, const uint16_t* W, int64_t ldw, const float* bias,
                               int relu, void* y, int64_t ldy, int y_is_bf16, int64_t B, int64_t N, int64_t K,
                               usf_stream_t stream) {
  USF_CHECK_ARG(x && W && y, "usf_linear_bf16: null pointer");   // bias may be NULL (plain GEMM)
  EpiParams ep{};
  ep.mode = relu ? EPI_BIAS_RELU : EPI_BIAS;
  ep.bias = bias;
  ep.out = y;
  ep.ldo = ldy;
  ep.out_bf16 = y_is_bf16;
  return tc_gemm(x, ldx, W, ldw, B, N, K, tc_pick_bn(N), ep, as_stream(stream));
}

extern "C" int usf_split_lo(const float* x, int64_t ldx, float* lo, int64_t ldl, int64_t rows, int64_t cols,
                            usf_stream_t stream) {
  USF_CHECK_ARG(x && lo && ldx >= cols && ldl >= cols, "usf_split_lo: bad arguments");
  return launch_split_lo(x, ldx, nullptr, lo, ldl, rows, cols, as_stream(stream));
}

extern "C" int usf_linear_tf32x3(const float* x, const float* x_lo, int64_t ldx, const float* W, const float* W_lo,
                                 int64_t ldw, const float* bias, int relu, float* y, float* y_lo, int64_t ldy, int64_t B,
                                 int64_t N, int64_t K, usf_stream_t stream) {
  USF_CHECK_ARG(x && x_lo && W && W_lo && y, "usf_linear_tf32x3: null pointer");
  EpiParams ep{};
  ep.mode = relu ? EPI_BIAS_RELU : EPI_BIAS;
  ep.bias = bias;
  ep.out = y;
  ep.ldo = ldy;
  ep.out_bf16 = 0;
  return tc3_gemm(x, x_lo, ldx, W, W_lo, ldw, B, N, K, tc_pick_bn(N), ep, y_lo, nullptr, as_stream(stream));
}

extern "C" int usf_profile_begin(int max_launches) {
  USF_CHECK_ARG(max_launches > 0 && !g_prof.on, "usf_profile_begin: bad state");
  g_prof.ev = new cudaEvent_t[2 * (size_t)max_launches];
  g_prof.tag = new int[max_launches];
  for (int i = 0; i < 2 * max_launches; ++i) USF_CUDA(cudaEventCreate(&g_prof.ev[i]));
  g_prof.cap = max_launches;
  g_prof.n = 0;
  g_prof.on = true;
  return USF_OK;
}

extern "C" int usf_profile_end(float* ms, int* tags, int* n_out) {
  USF_CHECK_ARG(g_prof.on, "usf_profile_end: profiling is not active");
  g_prof.on = false;
  int rc = USF_OK;
  for (int i = 0; i < g_prof.n; ++i) {
    if (cudaEventSynchronize(g_prof.ev[2 * i + 1]) != cudaSuccess) rc = USF_E_CUDA;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]) != cudaSuccess) rc = USF_E_CUDA;
    if (ms) ms[i] = t;
    if (tags) tags[i] = g_prof.tag[i];
  }
  if (n_out) *n_out = g_prof.n;
  for (int i = 0; i < 2 * g_prof.cap; ++i) cudaEventDestroy(g_prof.ev[i]);
  delete[] g_prof.ev;
  delete[] g_prof.tag;
  g_prof = Profile();
  if (rc) set_error("usf_profile_end: event query failed");
  return rc;
}

extern "C" size_t usf_stack_workspace_bytes(const usf_stack_desc* st, int64_t B, int precision) {
  StackPlan p;
  const int64_t rows = B < kChunkRows ? (B > 0 ? B : 1) : kChunkRows;
  if (plan_stack(st, rows, precision, &p) != USF_OK) return 0;
  return p.total;
}

// x_bf16: x points to bf16 rows (ldx in bf16 elements) instead of fp32 ones -- usf_stack_run_bf16in
static int stack_run_eager(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob,
                           float* out_y, int64_t ldy, float* out_ladj, void* workspace, size_t workspace_bytes,
                           int precision, int* gpu_launches, usf_stream_t stream, int x_bf16) {
  USF_CHECK_ARG(st != nullptr && x != nullptr && B >= 0, "usf_stack_run: bad arguments");
  USF_CHECK_ARG(!x_bf16 || precision == USF_PREC_BF16, "usf_stack_run_bf16in: bf16 rows need the bf16 precision tier");
  USF_CHECK_ARG(!(out_logprob && (st->base_kind < 0 || !st->inverse)),
                "usf_stack_run: log_prob needs the inverse direction and a base distribution");
  USF_CHECK_ARG(!(out_logprob && out_ladj), "usf_stack_run: request log_prob or ladj, not both");
  const int64_t d_in = (int64_t)st->D + st->ctx_dim;   // input row = D coordinates + the context columns
  USF_CHECK_ARG(ldx >= d_in && (out_y == nullptr || ldy >= st->D), "usf_stack_run: leading dimension < D");
  if (gpu_launches) *gpu_launches = 0;
  if (B == 0) return USF_OK;
  // small event shapes (D + context <= 64, widths <= 128; fp32 weights): the whole stack in ONE kernel, rows resident
  // in shared memory across all layers (usf_small.cu) -- the chain below would be 8-40 launches of a few microseconds
  if (!x_bf16 && small_stack_supported(st, precision)) {
    USF_CHECK_ARG(out_logprob != nullptr || out_y != nullptr || out_ladj != nullptr, "usf_stack_run: nothing to compute (no output requested)");
    int rc1;
    {
      ProfScope ps(as_stream(stream), 6);
      rc1 = small_stack_run(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, as_stream(stream));
    }
    if (rc1 == USF_OK && gpu_launches) *gpu_launches = 1;
    return rc1;
  }
  const int64_t rows_max = B < kChunkRows ? B : kChunkRows;
  StackPlan p;
  int rc = plan_stack(st, rows_max, precision, &p);
  if (rc) return rc;
  if (workspace == nullptr || workspace_bytes < p.total) {
    set_error("usf_stack_run: workspace too small (%zu < %zu bytes)", workspace_bytes, p.total);
    return USF_E_WORKSPACE;
  }
  cudaStream_t s = as_stream(stream);
  const bool bf16 = precision == USF_PREC_BF16;
  const bool b2 = precision == USF_PREC_BF16X2;      // bf16 (hi, lo) operand pairs
  const size_t esz = (bf16 || b2) ? 2 : 4;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  uint8_t* act[2] = {base, base + p.act_bytes};
  uint8_t* hid[2] = {base + 2 * p.act_bytes, base + 2 * p.act_bytes + p.hid_bytes};
  float* small = p.small_bytes ? reinterpret_cast<float*>(base + 2 * p.act_bytes + 2 * p.hid_bytes + p.acc_bytes) : nullptr;
  const bool t3 = precision == USF_PREC_TF32X3;
  // low-part twins of the activation / hidden buffers (3xTF32 / bf16x2), placed after the accumulator region
  uint8_t* lo_base = base + 2 * p.act_bytes + 2 * p.hid_bytes + p.acc_bytes + p.small_bytes;
  uint8_t* act_lo[2] = {lo_base, lo_base + p.act_bytes};
  uint8_t* hid_lo[2] = {lo_base + 2 * p.act_bytes, lo_base + 2 * p.act_bytes + p.hid_bytes};
  auto lo_of = [&](const void* hi) -> float* {   // the twin of one of the four hi buffers (or of a pointer into it)
    if (!t3 && !b2) return nullptr;
    const uint8_t* h = reinterpret_cast<const uint8_t*>(hi);
    return reinterpret_cast<float*>(lo_base + (h - base));
  };
  (void)act_lo; (void)hid_lo;
  // deterministic mode: slot area for the per-row partial sums, after everything else
  const size_t twins_n = (t3 || b2) ? 2 : 1;
  float* det = p.det_slots > 0 ? reinterpret_cast<float*>(lo_base + (twins_n - 1) * (2 * p.act_bytes + 2 * p.hid_bytes)) : nullptr;
  int det_cursor = 0;
  // points an accumulating launch at its slots (n of them) instead of the atomics
  auto det_assign = [&](EpiParams& ep, int n, int64_t rows) {
    if (det == nullptr || ep.row_acc == nullptr) return;
    ep.row_part = det;
    ep.part_ld = rows;
    ep.part_slot = det_cursor;
    det_cursor += n;
  };

  int launches = 0;
  // Serpentine tile order (bf16 tier): every tensor-core kernel of the chain walks the row tiles in the opposite
  // direction of its predecessor, so that it starts on the rows that kernel wrote last and that are still in L2
  // (usf_tc.cu: tc_set_tile_order).  The input pack walks first -> last, so the first GEMM starts reversed.
  static const bool serpentine = []() { const char* e = getenv("USF_TC_SERPENTINE"); return !(e != nullptr && e[0] == '0'); }();
  int flip = 1;
  auto next_order = [&]() { tc_set_tile_order(serpentine ? flip : 0); flip ^= 1; };
  struct OrderReset { ~OrderReset() { tc_set_tile_order(0); } } order_reset;   // stand-alone GEMM calls stay first -> last

  // One GEMM of the chain at the chosen precision.
  auto gemm = [&](const void* A, int64_t lda, const usf_linear_desc& L, int bn, EpiParams& ep, int64_t rows) -> int {
    if (bf16) {
      USF_CHECK_ARG(L.Wb != nullptr, "usf_stack_run: bf16 weights missing in descriptor");
      next_order();
      return tc_gemm(reinterpret_cast<const uint16_t*>(A), lda, L.Wb, L.ldw, rows, L.N, L.K, bn, ep, s);
    }
    if (b2) {
      USF_CHECK_ARG(L.Wb != nullptr, "usf_stack_run: bf16 (hi, lo) weights missing in descriptor");
      const uint16_t* Ab = reinterpret_cast<const uint16_t*>(A);
      uint16_t* ub_lo = ep.ub != nullptr ? reinterpret_cast<uint16_t*>(lo_of(ep.ub)) : nullptr;
      uint16_t* out_lo = (ep.out != nullptr && (ep.mode == EPI_BIAS || ep.mode == EPI_BIAS_RELU) &&
                          reinterpret_cast<uint8_t*>(ep.out) >= base && reinterpret_cast<uint8_t*>(ep.out) < lo_base)
                             ? reinterpret_cast<uint16_t*>(lo_of(ep.out)) : nullptr;
      return tcb2_gemm(Ab, reinterpret_cast<const uint16_t*>(lo_of(Ab)), lda, L.Wb, L.Wb + (size_t)L.N * (size_t)L.ldw, L.ldw,
                       rows, L.N, L.K, bn, ep, out_lo, ub_lo, s);
    }
    USF_CHECK_ARG(L.W != nullptr, "usf_stack_run: fp32 weights missing in descriptor");
    if (t3) {
      const float* Af = reinterpret_cast<const float*>(A);
      float* ub_lo = ep.ub != nullptr ? lo_of(ep.ub) : nullptr;
      float* out_lo = (ep.out != nullptr && (ep.mode == EPI_BIAS || ep.mode == EPI_BIAS_RELU) &&
                       reinterpret_cast<uint8_t*>(ep.out) >= base && reinterpret_cast<uint8_t*>(ep.out) < lo_base)
                          ? lo_of(ep.out) : nullptr;
      return tc3_gemm(Af, lo_of(Af), lda, L.W, L.W + (size_t)L.N * (size_t)L.ldw, L.ldw, rows, L.N, L.K, bn, ep, out_lo,
                      ub_lo, s);
    }
    return simt_gemm(reinterpret_cast<const float*>(A), lda, 0, L.W, L.ldw, 0, rows, L.N, L.K, ep, s, small,
                     p.small_bytes / sizeof(float));
  };

  for (int64_t r0 = 0; r0 < B; r0 += kChunkRows) {
    const int64_t rows = (B - r0) < kChunkRows ? (B - r0) : kChunkRows;
    float* row_acc = out_logprob ? out_logprob + r0 : (out_ladj ? out_ladj + r0 : nullptr);
    const float acc_init = out_logprob ? st->const_term : 0.f;


    // stage 0: bring x into the activation layout (bf16, or padded fp32) and seed the per-row accumulator
    int cur = 0;
    flip = 1;
    det_cursor = 0;
    if (det != nullptr && row_acc != nullptr)
      USF_CUDA(cudaMemsetAsync(det, 0, (size_t)p.det_slots * (size_t)rows * sizeof(float), s));
    {
      ProfScope ps(s, 0);
      if (b2)
        rc = launch_split_rows_bf16x2(x + r0 * ldx, ldx, reinterpret_cast<uint16_t*>(act[0]),
                                      reinterpret_cast<uint16_t*>(lo_of(act[0])), p.ld_act, rows, d_in, row_acc, acc_init, s);
      else if (x_bf16)
        rc = launch_copy_rows_bf16(reinterpret_cast<const uint16_t*>(x) + r0 * ldx, ldx, reinterpret_cast<uint16_t*>(act[0]),
                                   p.ld_act, rows, d_in, row_acc, acc_init, s);
      else
        rc = launch_convert_rows(x + r0 * ldx, ldx, bf16 ? reinterpret_cast<uint16_t*>(act[0]) : nullptr,
                                 bf16 ? nullptr : reinterpret_cast<float*>(act[0]), p.ld_act, rows, d_in, row_acc,
                                 acc_init, s);
    }
    if (rc) return rc;
    ++launches;
    if (t3) {
      rc = launch_split_lo(reinterpret_cast<const float*>(act[0]), p.ld_act, reinterpret_cast<float*>(act[0]), lo_of(act[0]),
                           p.ld_act, rows, p.ld_act, s);
      if (rc) return rc;
      ++launches;
    }

    for (int b = 0; b < st->n_blocks; ++b) {
      const usf_block_desc& blk = st->blocks[b];
      // (1) dense affine map u = G x + g, written in [a | pad | b] column order
      {
        EpiParams ep{};
        ep.mode = EPI_BIAS;
        ep.bias = blk.G.bias;
        ep.out = act[cur ^ 1];
        ep.ldo = p.ld_act;
        ep.out_bf16 = bf16 || b2;
        {
          ProfScope ps(s, 1);
          rc = gemm(act[cur], p.ld_act, blk.G, (bf16 || t3 || b2) ? tc_pick_bn(blk.G.N) : 0, ep, rows);
        }
        if (rc) return rc;
        ++launches;
        cur ^= 1;
      }
      // (2) conditioner MLP on the a-part, last layer fused with the coupling update of the b-part
      bool fused = false;
      if (bf16 && blk.n_mlp >= 2) {
        int Ns[USF_MAX_MLP], Ks[USF_MAX_MLP], ldws[USF_MAX_MLP];
        const uint16_t* Wbs[USF_MAX_MLP];
        const float* biases[USF_MAX_MLP];
        bool have = true;
        for (int l = 0; l < blk.n_mlp; ++l) {
          Ns[l] = blk.mlp[l].N; Ks[l] = blk.mlp[l].K; ldws[l] = blk.mlp[l].ldw;
          Wbs[l] = blk.mlp[l].Wb; biases[l] = blk.mlp[l].bias;
          have = have && Wbs[l] != nullptr && biases[l] != nullptr;
        }
        if (have && blk.n_mlp <= 4 && tc_mlp_supported(blk.n_mlp, Ns, Ks, blk.Da)) {
          // ONE kernel: the whole conditioner chain with hidden activations resident in shared memory + coupling
          EpiParams ep{};
          if (blk.affine) ep.mode = st->inverse ? EPI_COUPLING_INV : EPI_COUPLING_FWD;
          else ep.mode = st->inverse ? EPI_ADD_INV : EPI_ADD_FWD;
          ep.ub = act[cur] + (size_t)blk.b_off * esz;
          ep.ldub = p.ld_act;
          ep.ub_bf16 = 1;
          ep.Db = blk.Db;
          ep.C = blk.C;
          ep.clamp = blk.clamp;
          ep.row_acc = row_acc;
          if (blk.affine) det_assign(ep, 2 * (int)ceil_div(blk.mlp[blk.n_mlp - 1].N, 2 * blk.C) > 4 ? 2 * (int)ceil_div(blk.mlp[blk.n_mlp - 1].N, 2 * blk.C) : 4, rows);
          next_order();
          {
            ProfScope ps(s, 5);
            rc = tc_mlp_coupling(reinterpret_cast<const uint16_t*>(act[cur]), p.ld_act, rows, blk.n_mlp, Wbs, ldws, biases,
                                 Ns, Ks, blk.affine ? 2 * blk.C : blk.C, ep, s);
          }
          if (rc) return rc;
          ++launches;
          fused = true;
        }
      }
      const void* in = act[cur];
      int64_t ld_in = p.ld_act;
      for (int l = 0; l < blk.n_mlp && !fused; ++l) {
        const usf_linear_desc& L = blk.mlp[l];
        EpiParams ep{};
        ep.bias = L.bias;
        int bn = 0;
        if (l + 1 < blk.n_mlp) {
          ep.mode = EPI_BIAS_RELU;
          ep.out = hid[l & 1];
          ep.ldo = p.ld_hid;
          ep.out_bf16 = bf16 || b2;
          if (bf16 || t3 || b2) bn = tc_pick_bn(L.N);
        } else {
          if (blk.affine) ep.mode = st->inverse ? EPI_COUPLING_INV : EPI_COUPLING_FWD;
          else ep.mode = st->inverse ? EPI_ADD_INV : EPI_ADD_FWD;
          ep.ub = act[cur] + (size_t)blk.b_off * esz;
          ep.ldub = p.ld_act;
          ep.ub_bf16 = bf16 || b2;
          ep.Db = blk.Db;
          ep.C = blk.C;
          ep.clamp = blk.clamp;
          ep.row_acc = row_acc;
          if (bf16 || t3 || b2) bn = blk.affine ? 2 * blk.C : blk.C;
          if (blk.affine)      // (the same slot count as the fused form of this block would take: see plan_stack)
            det_assign(ep, (bf16 || t3 || b2) ? (2 * (int)ceil_div(L.N, 2 * blk.C) > 4 ? 2 * (int)ceil_div(L.N, 2 * blk.C) : 4)
                                             : det_slots_of(precision, L.N, 0, false), rows);
        }
        {
          ProfScope ps(s, l + 1 < blk.n_mlp ? 2 : 3);
          rc = gemm(in, ld_in, L, bn, ep, rows);
        }
        if (rc) return rc;
        ++launches;
        in = hid[l & 1];
        ld_in = p.ld_hid;
      }
    }
    // (3) last affine map, fused with the base log-density when a density is requested
    {
      EpiParams ep{};
      ep.bias = st->G_final.bias;
      ep.n_valid = st->D;
      ep.out = out_y ? out_y + r0 * ldy : nullptr;
      ep.ldo = ldy;
      ep.out_bf16 = 0;
      if (out_logprob) {
        ep.mode = st->base_kind == 0 ? EPI_BASE_NORMAL : EPI_BASE_LAPLACE;
        ep.loc = st->loc;
        ep.inv_scale = st->inv_scale;
        ep.row_acc = row_acc;
        det_assign(ep, (bf16 || t3 || b2) ? det_slots_of(precision, st->G_final.N, tc_pick_bn(st->G_final.N), false)
                                          : det_slots_of(precision, st->D, 0, false), rows);
      } else {
        USF_CHECK_ARG(out_y != nullptr, "usf_stack_run: nothing to compute (no output requested)");
        ep.mode = EPI_BIAS;
      }
      // fp32 path: the SIMT kernel stores exactly N = D columns
      usf_linear_desc Lf = st->G_final;
      if (!bf16 && !t3 && !b2) Lf.N = st->D;
      {
        ProfScope ps(s, 4);
        rc = gemm(act[cur], p.ld_act, Lf, (bf16 || t3 || b2) ? tc_pick_bn(Lf.N) : 0, ep, rows);
      }
      if (rc) return rc;
      ++launches;
    }
    // deterministic mode: the slots, added in slot order, on top of the seeded accumulator
    if (det != nullptr && row_acc != nullptr && det_cursor > 0) {
      rc = launch_sum_row_parts(row_acc, det, rows, det_cursor, rows, s);
      if (rc) return rc;
      ++launches;
    }
  }
  if (gpu_launches) *gpu_launches = launches;
  return USF_OK;
}

// ------------------------------------------------------------------------------------------------------------
// CUDA-graph replay of the launch chain.  A scoring loop calls usf_stack_run with the SAME descriptors, buffers and
// row count step after step; the second identical call captures the chain (on a private capture stream) into a
// graph and later calls replay it with one cudaGraphLaunch, which takes the per-launch host cost (cluster launches
// with 227 KB of smem, tensor-map parameters) off the critical path.  The cache is per thread, bounded, keyed by a
// hash of every descriptor byte and pointer, and can be disabled with USF_GRAPHS=0.  A graph only bakes in
// addresses, shapes and scalars, never buffer contents, so re-using it after the weights were updated in place
// (same storage) is valid.
// ------------------------------------------------------------------------------------------------------------
namespace {

struct GraphEntry {
  uint64_t key = 0;                  // FNV hash of `bytes` (first-level filter only)
  std::vector<unsigned char> bytes;  // the full key material: a hit needs these to compare equal, not just the hash
  cudaGraphExec_t exec = nullptr;
  int launches = 0;
  int seen = 0;
  uint64_t stamp = 0;
};
constexpr int kGraphSlots = 16;
thread_local GraphEntry g_graphs[kGraphSlots];
thread_local cudaStream_t g_capture_stream = nullptr;
thread_local uint64_t g_graph_clock = 0;
// counters of this thread's usf_stack_run calls: {graph replays, successful captures, failed captures, eager runs}
thread_local long long g_graph_stats[4] = {0, 0, 0, 0};
thread_local char g_graph_fail[160] = "";

inline uint64_t fnv(uint64_t h, const void* data, size_t n) {
  const unsigned char* p = static_cast<const unsigned char*>(data);
  for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
  return h;
}

bool graphs_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("USF_GRAPHS"); on = (e != nullptr && e[0] == '0') ? 0 : 1; }
  return on == 1;
}

}  // namespace

extern "C" int usf_debug_graph_stats(long long* stats4, char* last_failure, int failure_bytes) {
  if (stats4 != nullptr)
    for (int i = 0; i < 4; ++i) stats4[i] = g_graph_stats[i];
  if (last_failure != nullptr && failure_bytes > 0) {
    strncpy(last_failure, g_graph_fail, (size_t)failure_bytes - 1);
    last_failure[failure_bytes - 1] = 0;
  }
  return USF_OK;
}

static int stack_run_cached(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob,
                            float* out_y, int64_t ldy, float* out_ladj, void* workspace, size_t workspace_bytes,
                            int precision, int* gpu_launches, usf_stream_t stream, int x_bf16) {
  if (st == nullptr || !graphs_enabled() || g_prof.on || B <= 0 || st->n_blocks < 0 ||
      (st->n_blocks > 0 && st->blocks == nullptr))
    return stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                           gpu_launches, stream, x_bf16);
  // key material = every descriptor byte and every call argument; the 64-bit hash only pre-filters, a hit compares
  // the bytes themselves (a hash collision must never replay another chain)
  const uint64_t extra[9] = {(uint64_t)(uintptr_t)x, (uint64_t)ldx, (uint64_t)B, (uint64_t)(uintptr_t)out_logprob,
                             (uint64_t)(uintptr_t)out_y, (uint64_t)ldy, (uint64_t)(uintptr_t)out_ladj,
                             (uint64_t)(uintptr_t)workspace,
                             (uint64_t)workspace_bytes * 16u + (uint64_t)precision + (x_bf16 ? 4u : 0u) + (g_deterministic ? 8u : 0u)};
  const size_t nb_bytes = st->n_blocks > 0 ? sizeof(usf_block_desc) * (size_t)st->n_blocks : 0;
  thread_local std::vector<unsigned char> kb;
  kb.resize(sizeof(*st) + nb_bytes + sizeof(extra));
  memcpy(kb.data(), st, sizeof(*st));
  if (nb_bytes) memcpy(kb.data() + sizeof(*st), st->blocks, nb_bytes);
  memcpy(kb.data() + sizeof(*st) + nb_bytes, extra, sizeof(extra));
  uint64_t key = fnv(1469598103934665603ull, kb.data(), kb.size());
  if (key == 0) key = 1;
  GraphEntry* slot = nullptr;
  GraphEntry* victim = &g_graphs[0];
  for (int i = 0; i < kGraphSlots; ++i) {
    if (g_graphs[i].key == key && g_graphs[i].bytes.size() == kb.size() &&
        memcmp(g_graphs[i].bytes.data(), kb.data(), kb.size()) == 0) { slot = &g_graphs[i]; break; }
    if (g_graphs[i].stamp < victim->stamp) victim = &g_graphs[i];
  }
  cudaStream_t s = as_stream(stream);
  if (slot != nullptr && slot->exec != nullptr) {
    slot->stamp = ++g_graph_clock;
    ++g_graph_stats[0];
    USF_CUDA(cudaGraphLaunch(slot->exec, s));
    if (gpu_launches) *gpu_launches = slot->launches;
    return USF_OK;
  }
  if (slot == nullptr) {   // first sighting: run eagerly and remember the key
    if (victim->exec != nullptr) cudaGraphExecDestroy(victim->exec);
    *victim = GraphEntry();
    victim->key = key;
    victim->bytes = kb;
    victim->seen = 1;
    victim->stamp = ++g_graph_clock;
    ++g_graph_stats[3];
    return stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                           gpu_launches, stream, x_bf16);
  }
  // second identical call: capture the chain, instantiate, replay
  slot->stamp = ++g_graph_clock;
  if (g_capture_stream == nullptr &&
      cudaStreamCreateWithFlags(&g_capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    return stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                           gpu_launches, stream, x_bf16);
  }
  int launches = 0;
  cudaGraph_t graph = nullptr;
  if (cudaStreamBeginCapture(g_capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    return stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                           gpu_launches, stream, x_bf16);
  }
  const int rc = stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                                 &launches, g_capture_stream, x_bf16);
  const cudaError_t ce = cudaStreamEndCapture(g_capture_stream, &graph);
  cudaGraphExec_t exec = nullptr;
  cudaError_t ie = cudaSuccess;
  if (rc != USF_OK || ce != cudaSuccess || graph == nullptr ||
      (ie = cudaGraphInstantiate(&exec, graph, 0)) != cudaSuccess) {
    ++g_graph_stats[2];
    snprintf(g_graph_fail, sizeof(g_graph_fail), "rc=%d endCapture=%s instantiate=%s", rc, cudaGetErrorName(ce),
             cudaGetErrorName(ie));
    cudaGetLastError();
    if (graph != nullptr) cudaGraphDestroy(graph);
    slot->key = 0;   // do not try again with this key
    return stack_run_eager(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                           gpu_launches, stream, x_bf16);
  }
  cudaGraphDestroy(graph);
  ++g_graph_stats[1];
  slot->exec = exec;
  slot->launches = launches;
  USF_CUDA(cudaGraphLaunch(exec, s));
  if (gpu_launches) *gpu_launches = launches;
  return USF_OK;
}

extern "C" int usf_set_deterministic(int on) {
  const int prev = g_deterministic;
  g_deterministic = on ? 1 : 0;
  return prev;
}

extern "C" int usf_stack_is_single_kernel(const usf_stack_desc* st, int precision) {
  return small_stack_supported(st, precision) ? 1 : 0;
}

extern "C" int usf_stack_run(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob,
                             float* out_y, int64_t ldy, float* out_ladj, void* workspace, size_t workspace_bytes,
                             int precision, int* gpu_launches, usf_stream_t stream) {
  return stack_run_cached(st, x, ldx, B, out_logprob, out_y, ldy, out_ladj, workspace, workspace_bytes, precision,
                          gpu_launches, stream, 0);
}

extern "C" int usf_stack_run_bf16in(const usf_stack_desc* st, const uint16_t* x_bf16, int64_t ldx, int64_t B,
                                    float* out_logprob, float* out_y, int64_t ldy, float* out_ladj, void* workspace,
                                    size_t workspace_bytes, int* gpu_launches, usf_stream_t stream) {
  return stack_run_cached(st, reinterpret_cast<const float*>(x_bf16), ldx, B, out_logprob, out_y, ldy, out_ladj, workspace,
                          workspace_bytes, USF_PREC_BF16, gpu_launches, stream, 1);
}
