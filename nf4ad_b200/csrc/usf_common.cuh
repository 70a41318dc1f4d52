// Shared declarations of the usflow_b200 library (internal; the public ABI is include/usflow_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/usflow_b200.h"

namespace usf {

// ---- thread-local error message -------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define USF_CHECK_ARG(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      ::usf::set_error(__VA_ARGS__);        \
      return USF_E_ARG;                     \
    }                                       \
  } while (0)

#define USF_CUDA(call)                                            \
  do {                                                            \
    cudaError_t _e = (call);                                      \
    if (_e != cudaSuccess) return ::usf::cuda_fail(_e, #call);    \
  } while (0)

#define USF_LAUNCH_CHECK(name)                                              \
  do {                                                                      \
    cudaError_t _e = cudaGetLastError();                                    \
    if (_e != cudaSuccess) return ::usf::cuda_fail(_e, "launch of " name);  \
  } while (0)

static inline cudaStream_t as_stream(usf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
__host__ __device__ static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ static inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }
inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

// Bump allocation from a caller's workspace: the start rounded up to 256 bytes, every buffer 256-byte aligned.
struct Arena {
  uint8_t* cur;
  explicit Arena(void* ws) : cur(reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255))) {}
  void* take(size_t bytes) {
    void* q = cur;
    cur += align256(bytes);
    return q;
  }
};

int num_sms();
int deterministic_mode();   // usf_set_deterministic of the calling thread

// ---- epilogue description shared by the SIMT and the tcgen05 GEMM kernels --------------------
// The GEMM computes acc[m, n] = sum_k A[m,k] * W[n,k]; the epilogue turns one accumulator tile into
// the layer's result without another pass over HBM.
enum EpiMode : int {
  EPI_BIAS = 0,          // out = acc + bias
  EPI_BIAS_RELU = 1,     // out = max(0, acc + bias)
  EPI_COUPLING_INV = 2,  // tile = [s(C) | t(C)]: xb = (ub - t) * exp(-clamp*tanh(s)); acc_row -= sum log_s
  EPI_COUPLING_FWD = 3,  // tile = [s(C) | t(C)]: yb = ub * exp(clamp*tanh(s)) + t;    acc_row += sum log_s
  EPI_ADD_INV = 4,       // tile = [t(C)]: xb = ub - t
  EPI_ADD_FWD = 5,       // tile = [t(C)]: yb = ub + t
  EPI_BASE_NORMAL = 6,   // z = acc + bias; acc_row += sum -0.5*((z-loc)*inv_scale)^2 ; optional z store
  EPI_BASE_LAPLACE = 7,  // z = acc + bias; acc_row += sum -|z-loc|*inv_scale       ; optional z store
};

struct EpiParams {
  int mode;
  const float* bias;     // indexed by packed output column n
  void* out;             // EPI_BIAS*/BASE: row-major output (fp32 or bf16), may be NULL for BASE
  int64_t ldo;
  int out_bf16;          // element type of `out`
  void* ub;              // coupling: pointer to the b-part (transformed coords) of the activation, in/out
  int64_t ldub;
  int ub_bf16;
  int Db;                // valid transformed coords
  int C;                 // coords per tile
  int n_valid;           // valid output columns (fp32 stores / base density); 0 = all N
  float clamp;
  float* row_acc;        // (M) per-row accumulator (log-det / log-density), atomically updated; may be NULL
  const float* loc;      // BASE: per output column
  const float* inv_scale;
  // deterministic mode (usf_set_deterministic): instead of an atomic add into row_acc -- whose order over the tiles /
  // warps that share a row is not fixed -- contributor `sub` of this launch stores its partial sum into its own slot
  // row_part[(part_slot + sub) * part_ld + row]; the chain ends with a kernel that adds the slots in slot order.
  float* row_part;
  int64_t part_ld;
  int part_slot;
};

#ifdef __CUDACC__
__device__ __forceinline__ void row_accumulate(const EpiParams& ep, int64_t row, int sub, float v) {
  if (ep.row_part != nullptr) ep.row_part[(int64_t)(ep.part_slot + sub) * ep.part_ld + row] = v;
  else atomicAdd(ep.row_acc + row, v);
}
#endif

// ---- SIMT fp32 GEMM (usf_simt.cu) -------------------------------------------------------------
// acc = A(MxK, lda) * W(NxK, ldw)^T with the epilogue above.  a_trans / w_trans select the
// storage order: a_trans=0: A[m*lda+k]; a_trans=1: A[k*lda+m]; w_trans=0: W[n*ldw+k]; 1: W[k*ldw+n].
// scratch (optional, scratch_floats >= M*N): enables the split-K + epilogue-kernel form for small batches.
int simt_gemm(const float* A, int64_t lda, int a_trans, const float* W, int64_t ldw, int w_trans,
              int64_t M, int64_t N, int64_t K, const EpiParams& ep, cudaStream_t stream, float* scratch = nullptr,
              size_t scratch_floats = 0);
// Plain C (+)= alpha * A*W^T style GEMM used by the backward pass (no bias), fp32 out with ldc.
int simt_gemm_plain(const float* A, int64_t lda, int a_trans, const float* W, int64_t ldw, int w_trans,
                    int64_t M, int64_t N, int64_t K, float* Cout, int64_t ldc, int accumulate,
                    cudaStream_t stream);

// ---- tcgen05 bf16 GEMM (usf_tc.cu) ------------------------------------------------------------
// A: (M, K) bf16 row-major with lda (multiple of 8); W: (N, K) bf16 row-major with ldw (multiple of 8).
// bn = N-tile width (multiple of 16, <= 256).
int tc_gemm(const uint16_t* A, int64_t lda, const uint16_t* W, int64_t ldw, int64_t M, int64_t N,
            int64_t K, int bn, const EpiParams& ep, cudaStream_t stream);
int tc_pick_bn(int64_t N);
void tc_set_tile_order(int reverse);   // tile walk of the next tcgen05 launches of this thread: 0 first -> last, 1 last -> first
// Split-operand GEMM (operands as hi + lo pairs: fp32-grade accuracy on the tensor cores).  T = float: 3xTF32
// (usf_tc3_gemm_kernel); T = uint16_t: bf16x2, bf16 pairs at a third of the bf16 rate (usf_tcb2_gemm_kernel).
template <class T>
int tc_split_gemm(const T* A, const T* Alo, int64_t lda, const T* W, const T* Wlo, int64_t ldw, int64_t M, int64_t N,
                  int64_t K, int bn, const EpiParams& ep, T* out_lo, T* ub_lo, cudaStream_t stream);
int launch_split_rows_bf16x2(const float* x, int64_t ldx, uint16_t* hi, uint16_t* lo, int64_t ldy, int64_t B, int64_t D,
                             float* row_init, float init_value, cudaStream_t stream);
// hi == NULL: lo against the truncated read of x; hi != NULL (may alias x): hi = x rounded to tf32, lo = x - hi
int launch_split_lo(const float* x, int64_t ldx, float* hi, float* lo, int64_t ldl, int64_t rows, int64_t cols, cudaStream_t stream);
bool tc_mlp_supported(int n_layers, const int* N, const int* K, int Da);
int tc_mlp_coupling(const uint16_t* A, int64_t lda, int64_t M, int n_layers, const uint16_t* const* Wb, const int* ldw,
                    const float* const* bias, const int* N, const int* K, int bn_last, const EpiParams& ep,
                    cudaStream_t stream);
extern const char* const kTcGemmKernelName;
extern const char* const kSimtGemmKernelName;
int64_t trsm_fast_scratch_floats(int64_t D);
bool trsm_fast_supported(int64_t D);
int trsm_rows_fast(const float* T, int64_t D, bool lower, bool unit, bool trans, const float* rhs, int64_t ldr,
                   const float* bias, float* X, int64_t ldx, int64_t B, float* scratch, cudaStream_t stream);
int64_t lu_inverse_scratch_floats(int64_t D);
int lu_inverse(const float* L_raw, const float* U_raw, int64_t D, float* A, float* scratch, cudaStream_t stream);
int tc_timeout_flag(int* out, int reset);
int trsm_rows(const float* T, int64_t D, bool lower, bool unit, bool trans, const float* rhs, int64_t ldr,
              const float* bias, float* X, int64_t ldx, int64_t B, cudaStream_t stream);

// ---- whole-stack kernel for small event shapes (usf_small.cu): one launch instead of the chain ------------------
bool small_stack_supported(const usf_stack_desc* st, int precision);
int small_stack_run(const usf_stack_desc* st, const float* x, int64_t ldx, int64_t B, float* out_logprob, float* out_y,
                    int64_t ldy, float* out_ladj, cudaStream_t stream);
// its gradient twin (usf_stack_log_prob_grad at fp32): log p and d log p / dx in one launch
bool small_grad_supported(const usf_stack_desc* st, const usf_stack_grad_desc* gd, int precision);
size_t small_grad_workspace_bytes(const usf_stack_desc* st, const usf_stack_grad_desc* gd);
int small_grad_run(const usf_stack_desc* st, const usf_stack_grad_desc* gd, const float* x, int64_t ldx, int64_t B,
                   float* out_logprob, float* out_grad, int64_t ldg, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream);

// ---- small helpers launched by the stack runner ---------------------------------------------
int launch_convert_rows(const float* x, int64_t ldx, uint16_t* y_bf16, float* y_f32, int64_t ldy,
                        int64_t B, int64_t D, float* row_init, float init_value, cudaStream_t stream);
int launch_copy_rows_bf16(const uint16_t* x, int64_t ldx, uint16_t* y, int64_t ldy, int64_t B, int64_t D, float* row_init,
                          float init_value, cudaStream_t stream);
// out[r] += sum over slots (in slot order) of part[s * ld + r]: the end of a deterministic launch chain
int launch_sum_row_parts(float* out, const float* part, int64_t ld, int slots, int64_t rows, cudaStream_t stream);
int launch_bf16_to_f32(const uint16_t* x, int64_t ldx, float* y, int64_t ldy, int64_t B, int64_t D,
                       cudaStream_t stream);

// ---- the forward launch chain of a packed stack (usf_api.cu): usf_stack_run and usf_stack_log_prob_grad ------------
// One row buffer of a chain: hi with leading dimension ld (elements), and lo its low-part twin when the operands travel
// as (hi, lo) pairs (3xTF32, bf16x2); lo is nullptr at fp32 / bf16 and for fp32 GEMM outputs.
struct Buf {
  void* hi;
  void* lo;
  int64_t ld;
};

// Deterministic mode: partial-sum slots (the `sub` range of row_accumulate) of the accumulating launch of block b's
// coupling (0 for an additive one), or of the final GEMM's base density at b == st->n_blocks.  Every chain sizes and
// assigns its slots with it, so that all of them add the same slots in the same order.
int det_slots(const usf_stack_desc* st, int b, int precision);

// One GEMM of a chain at `precision`: A (rows, L.K) times L^T, N output columns, N tile bn (0: tc_pick_bn(N); the SIMT
// kernel takes none), epilogue ep.  out_lo / ub_lo: the low-part twins of ep.out / ep.ub (3xTF32, bf16x2), or nullptr.
// scratch: the fp32 split-K accumulator of simt_gemm, or nullptr.
int chain_gemm(int precision, const Buf& A, const usf_linear_desc& L, int64_t rows, int64_t N, int bn,
               const EpiParams& ep, void* out_lo, void* ub_lo, float* scratch, size_t scratch_floats, cudaStream_t stream);

// Where one pass of run_chain puts its rows.
struct ChainIO {
  const Buf* act;            // act[0] receives the packed input, act[(j + 1) % n_act] block j's output row
  int n_act;
  const Buf* hid;            // the k-th hidden activation of the pass (counted over all blocks) goes to hid[k % n_hid]
  int n_hid;
  bool density;              // the final GEMM adds the base log-density to row_acc (else: the plain affine map into out)
  float* out;                // the final GEMM's rows (z or y, D columns), or nullptr
  int64_t ldo;
  float* row_acc;            // per-row log p / log-det, seeded with acc_init by the input pack; or nullptr
  float acc_init;
  float* det;                // deterministic mode: slot area of det_n slots of `rows` floats (nullptr: fp32 atomics)
  int det_n;
  float* scratch;            // fp32 split-K accumulator (chain_gemm), or nullptr
  size_t scratch_floats;
};

// The forward chain over `rows` rows of x (fp32 rows, or bf16 rows when x_bf16) at `precision`: input pack, per block
// the G GEMM, the conditioner GEMMs (or the fused bf16 conditioner kernel) ending in the coupling, the final GEMM, and
// in deterministic mode the slot sum.  Adds the launches it enqueues to *launches.
int run_chain(const usf_stack_desc* st, const void* x, int64_t ldx, bool x_bf16, int64_t rows, int precision,
              const ChainIO& io, int* launches, cudaStream_t stream);

}  // namespace usf
