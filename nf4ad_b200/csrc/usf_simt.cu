// fp32 SIMT kernels of the usflow_b200 library (sm_100a).
//
//  * simt_gemm: 128x128x16 register-tiled FFMA GEMM with the fused layer epilogues (EpiParams): the
//    fp32-accuracy path of every dense contraction (LU apply, conditioner MLP) and of the fused stack.
//  * trsm_rows: blocked triangular solve over batch rows (LUTransform.backward).
//  * row kernels (one warp per sample row): Householder, scale, coupling, base log-density and their
//    backward counterparts; small reductions.
//
// Roofline notes: the GEMM is FFMA-bound (fp32 pipe); all row kernels are HBM-bound (one read + one
// write of the (B,D) activation, coalesced, one warp per row, warp-shuffle reductions).
#include "usf_common.cuh"

namespace usf {

// ================================================================================================
// SIMT GEMM
// ================================================================================================
namespace {

constexpr int BM = 128, BN = 128, BK = 16, NTHREADS = 256, PAD = 4;

__device__ __forceinline__ float warp16_sum(float v) {
  // reduce over the 16 lanes that share ty (lanes differ in tx = lane & 15)
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float ld_act(const void* p, int64_t idx, int is_bf16) {
  if (is_bf16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[idx]);
  return reinterpret_cast<const float*>(p)[idx];
}
__device__ __forceinline__ void st_act(void* p, int64_t idx, int is_bf16, float v) {
  if (is_bf16) reinterpret_cast<__nv_bfloat16*>(p)[idx] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(p)[idx] = v;
}

// Loads an (ROWS=128) x (BK=16) operand tile into registers (8 floats / thread).
// trans == 0: element(r,k) = P[r*ld + k]  (k contiguous)  -> thread: r = tid/2, k = (tid%2)*8 + i
// trans == 1: element(r,k) = P[k*ld + r]  (r contiguous)  -> thread: k = tid/16, r = (tid%16)*8 + i
__device__ __forceinline__ void load_tile(const float* __restrict__ P, int64_t ld, int trans, int64_t r0,
                                          int64_t k0, int64_t R, int64_t K, int tid, float (&v)[8]) {
  if (!trans) {
    const int64_t r = r0 + (tid >> 1);
    const int64_t k = k0 + (tid & 1) * 8;
    const float* src = P + r * ld + k;
    if (r < R && k + 8 <= K && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
      const float4 a = *reinterpret_cast<const float4*>(src);
      const float4 b = *reinterpret_cast<const float4*>(src + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (r < R && k + i < K) ? src[i] : 0.f;
    }
  } else {
    const int64_t k = k0 + (tid >> 4);
    const int64_t r = r0 + (tid & 15) * 8;
    const float* src = P + k * ld + r;
    if (k < K && r + 8 <= R && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
      const float4 a = *reinterpret_cast<const float4*>(src);
      const float4 b = *reinterpret_cast<const float4*>(src + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (k < K && r + i < R) ? src[i] : 0.f;
    }
  }
}

__device__ __forceinline__ void store_tile(float (*S)[BM + PAD], int trans, int tid, const float (&v)[8]) {
  if (!trans) {
    const int r = tid >> 1, k = (tid & 1) * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) S[k + i][r] = v[i];
  } else {
    const int k = tid >> 4, r = (tid & 15) * 8;
    *reinterpret_cast<float4*>(&S[k][r]) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(&S[k][r + 4]) = make_float4(v[4], v[5], v[6], v[7]);
  }
}

struct PlainOut {
  float* C;
  int64_t ldc;
  int accumulate;  // 0: store, 1: += (non-atomic when split_k == 1, atomic otherwise)
  int split_k;
};

// One kernel body; FUSED selects the layer epilogues (EpiParams) vs the plain C output (backward).
template <bool FUSED>
__global__ void __launch_bounds__(NTHREADS)
usf_simt_gemm_kernel(const float* __restrict__ A, int64_t lda, int a_trans, const float* __restrict__ W,
                     int64_t ldw, int w_trans, int64_t M, int64_t N, int64_t K, EpiParams ep, PlainOut po) {
  __shared__ __align__(16) float As[2][BK][BM + PAD];
  __shared__ __align__(16) float Bs[2][BK][BN + PAD];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int64_t n0 = (int64_t)blockIdx.y * BN;

  // split-K range (plain variant only)
  int64_t kb = 0, ke = K;
  if (!FUSED && po.split_k > 1) {
    const int64_t chunk = round_up(ceil_div(K, po.split_k), BK);
    kb = (int64_t)blockIdx.z * chunk;
    ke = kb + chunk < K ? kb + chunk : K;
    if (kb >= ke) return;
  }

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float ra[8], rb[8];
  load_tile(A, lda, a_trans, m0, kb, M, ke, tid, ra);
  load_tile(W, ldw, w_trans, n0, kb, N, ke, tid, rb);
  store_tile(As[0], a_trans, tid, ra);
  store_tile(Bs[0], w_trans, tid, rb);
  __syncthreads();

  int buf = 0;
  for (int64_t k0 = kb; k0 < ke; k0 += BK) {
    const bool has_next = k0 + BK < ke;
    if (has_next) {
      load_tile(A, lda, a_trans, m0, k0 + BK, M, ke, tid, ra);
      load_tile(W, ldw, w_trans, n0, k0 + BK, N, ke, tid, rb);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (has_next) {
      store_tile(As[buf ^ 1], a_trans, tid, ra);
      store_tile(Bs[buf ^ 1], w_trans, tid, rb);
      __syncthreads();
      buf ^= 1;
    }
  }

  // ------------------------------------------------------------------ epilogue
  if (!FUSED) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      if (r >= M) continue;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int64_t c = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        if (c >= N) continue;
        float* dst = po.C + r * po.ldc + c;
        if (po.split_k > 1) atomicAdd(dst, acc[i][j]);
        else if (po.accumulate) *dst += acc[i][j];
        else *dst = acc[i][j];
      }
    }
    return;
  }

  const int mode = ep.mode;
  if (mode == EPI_BIAS || mode == EPI_BIAS_RELU) {
    float bj[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int64_t c = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      bj[j] = (ep.bias != nullptr && c < N) ? ep.bias[c] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      if (r >= M) continue;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int64_t c = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        if (c >= N) continue;
        float v = acc[i][j] + bj[j];
        if (mode == EPI_BIAS_RELU) v = fmaxf(v, 0.f);
        st_act(ep.out, r * ep.ldo + c, ep.out_bf16, v);
      }
    }
  } else if (mode == EPI_COUPLING_INV || mode == EPI_COUPLING_FWD) {
    // tile columns [0,64) = s of coords blockIdx.y*64 + [0,64); columns [64,128) = t of the same coords
    float bs[4], bt[4];
    int coord[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      coord[j] = (int)blockIdx.y * 64 + tx * 4 + j;
      bs[j] = ep.bias[n0 + tx * 4 + j];
      bt[j] = ep.bias[n0 + 64 + tx * 4 + j];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      float lsum = 0.f;
      if (r < M) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (coord[j] >= ep.Db) continue;
          const float s = acc[i][j] + bs[j];
          const float t = acc[i][4 + j] + bt[j];
          const float ls = ep.clamp * tanhf(s);
          const int64_t idx = r * ep.ldub + coord[j];
          const float u = ld_act(ep.ub, idx, ep.ub_bf16);
          const float y = (mode == EPI_COUPLING_INV) ? (u - t) * expf(-ls) : fmaf(u, expf(ls), t);
          st_act(ep.ub, idx, ep.ub_bf16, y);
          lsum += ls;
        }
      }
      lsum = warp16_sum(lsum);
      if (tx == 0 && r < M && ep.row_acc != nullptr)
        row_accumulate(ep, r, (int)blockIdx.y, mode == EPI_COUPLING_INV ? -lsum : lsum);
    }
  } else if (mode == EPI_ADD_INV || mode == EPI_ADD_FWD) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      if (r >= M) continue;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int64_t c = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        if (c >= ep.Db) continue;
        const float t = acc[i][j] + ep.bias[c];
        const int64_t idx = r * ep.ldub + c;
        const float u = ld_act(ep.ub, idx, ep.ub_bf16);
        st_act(ep.ub, idx, ep.ub_bf16, mode == EPI_ADD_INV ? u - t : u + t);
      }
    }
  } else {  // EPI_BASE_NORMAL / EPI_BASE_LAPLACE
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t r = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      float lsum = 0.f;
      if (r < M) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int64_t c = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
          if (c >= N) continue;
          const float z = acc[i][j] + ep.bias[c];
          if (ep.out != nullptr) st_act(ep.out, r * ep.ldo + c, ep.out_bf16, z);
          if (ep.loc != nullptr) {
            const float d = (z - ep.loc[c]) * ep.inv_scale[c];
            lsum += (mode == EPI_BASE_NORMAL) ? -0.5f * d * d : -fabsf(d);
          }
        }
      }
      lsum = warp16_sum(lsum);
      if (tx == 0 && r < M && ep.row_acc != nullptr && ep.loc != nullptr) row_accumulate(ep, r, (int)blockIdx.y, lsum);
    }
  }
}

}  // namespace

// Second phase of the small-batch form of the fused GEMM: the layer epilogue of usf_simt_gemm_kernel<true> applied to
// an accumulator that a split-K launch left in global memory (acc: M x N, leading dimension N).  One warp per row.
__global__ void usf_simt_epilogue_kernel(const float* __restrict__ acc, int64_t M, int64_t N, EpiParams ep) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= M) return;
  const float* a = acc + r * N;
  const int mode = ep.mode;
  if (mode == EPI_BIAS || mode == EPI_BIAS_RELU) {
    for (int64_t c = lane; c < N; c += 32) {
      float v = a[c] + (ep.bias != nullptr ? ep.bias[c] : 0.f);
      if (mode == EPI_BIAS_RELU) v = fmaxf(v, 0.f);
      st_act(ep.out, r * ep.ldo + c, ep.out_bf16, v);
    }
  } else if (mode == EPI_COUPLING_INV || mode == EPI_COUPLING_FWD) {
    float lsum = 0.f;
    for (int coord = lane; coord < ep.Db; coord += 32) {
      const int64_t cs = (int64_t)(coord >> 6) * 128 + (coord & 63);   // tile = [s(64) | t(64)]
      const float s = a[cs] + ep.bias[cs];
      const float t = a[cs + 64] + ep.bias[cs + 64];
      const float ls = ep.clamp * tanhf(s);
      const int64_t idx = r * ep.ldub + coord;
      const float u = ld_act(ep.ub, idx, ep.ub_bf16);
      st_act(ep.ub, idx, ep.ub_bf16, (mode == EPI_COUPLING_INV) ? (u - t) * expf(-ls) : fmaf(u, expf(ls), t));
      lsum += ls;
    }
    lsum = warp_sum(lsum);
    if (lane == 0 && ep.row_acc != nullptr) row_accumulate(ep, r, 0, mode == EPI_COUPLING_INV ? -lsum : lsum);
  } else if (mode == EPI_ADD_INV || mode == EPI_ADD_FWD) {
    for (int c = lane; c < ep.Db; c += 32) {
      const float t = a[c] + ep.bias[c];
      const int64_t idx = r * ep.ldub + c;
      const float u = ld_act(ep.ub, idx, ep.ub_bf16);
      st_act(ep.ub, idx, ep.ub_bf16, mode == EPI_ADD_INV ? u - t : u + t);
    }
  } else {  // EPI_BASE_NORMAL / EPI_BASE_LAPLACE
    float lsum = 0.f;
    for (int64_t c = lane; c < N; c += 32) {
      const float z = a[c] + ep.bias[c];
      if (ep.out != nullptr) st_act(ep.out, r * ep.ldo + c, ep.out_bf16, z);
      if (ep.loc != nullptr) {
        const float d = (z - ep.loc[c]) * ep.inv_scale[c];
        lsum += (mode == EPI_BASE_NORMAL) ? -0.5f * d * d : -fabsf(d);
      }
    }
    lsum = warp_sum(lsum);
    if (lane == 0 && ep.row_acc != nullptr && ep.loc != nullptr) row_accumulate(ep, r, 0, lsum);
  }
}

// out[r] += part[0][r] + part[1][r] + ... in slot order (deterministic mode: the end of the launch chain)
__global__ void usf_sum_row_parts_kernel(float* out, const float* __restrict__ part, int64_t ld, int slots, int64_t rows) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
    float v = out[r];
    for (int s = 0; s < slots; ++s) v += part[(int64_t)s * ld + r];
    out[r] = v;
  }
}

int launch_sum_row_parts(float* out, const float* part, int64_t ld, int slots, int64_t rows, cudaStream_t stream) {
  if (rows <= 0 || slots <= 0) return USF_OK;
  int64_t blocks = (rows + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  usf_sum_row_parts_kernel<<<(unsigned)blocks, 256, 0, stream>>>(out, part, ld, slots, rows);
  USF_LAUNCH_CHECK("usf_sum_row_parts_kernel");
  return USF_OK;
}

const char* const kSimtGemmKernelName = "usf_simt_gemm_kernel";

int simt_gemm(const float* A, int64_t lda, int a_trans, const float* W, int64_t ldw, int w_trans,
              int64_t M, int64_t N, int64_t K, const EpiParams& ep, cudaStream_t stream, float* scratch,
              size_t scratch_floats) {
  if (M <= 0 || N <= 0) return USF_OK;
  if ((ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD) && ep.C != 64) {
    set_error("simt_gemm: coupling epilogue needs C == 64 (got %d)", ep.C);
    return USF_E_ARG;
  }
  if (scratch != nullptr && (size_t)M * (size_t)N <= scratch_floats && K >= 64 &&
      ceil_div(M, BM) * ceil_div(N, BN) * 2 <= num_sms()) {
    // small batch: a handful of 128x128 tiles would walk K serially on a few SMs.  Split K across the SMs into the
    // caller's scratch accumulator, then apply the same epilogue from there (2 short launches instead of 1 long).
    int rc = simt_gemm_plain(A, lda, a_trans, W, ldw, w_trans, M, N, K, scratch, N, 0, stream);
    if (rc) return rc;
    const int warps = 8;
    usf_simt_epilogue_kernel<<<(unsigned)ceil_div(M, warps), warps * 32, 0, stream>>>(scratch, M, N, ep);
    USF_LAUNCH_CHECK("usf_simt_epilogue_kernel");
    return USF_OK;
  }
  dim3 grid((unsigned)ceil_div(M, BM), (unsigned)ceil_div(N, BN), 1);
  PlainOut po{nullptr, 0, 0, 1};
  usf_simt_gemm_kernel<true><<<grid, NTHREADS, 0, stream>>>(A, lda, a_trans, W, ldw, w_trans, M, N, K, ep, po);
  USF_LAUNCH_CHECK("usf_simt_gemm_kernel");
  return USF_OK;
}

int simt_gemm_plain(const float* A, int64_t lda, int a_trans, const float* W, int64_t ldw, int w_trans,
                    int64_t M, int64_t N, int64_t K, float* Cout, int64_t ldc, int accumulate,
                    cudaStream_t stream) {
  if (M <= 0 || N <= 0) return USF_OK;
  const int64_t tiles = ceil_div(M, BM) * ceil_div(N, BN);
  // Few output tiles (small batches, weight gradients of narrow layers): one 128x128 tile walks K serially at ~1 us
  // per 16-wide step with most SMs idle, so K is split over up to ~one CTA per SM (>= 32 columns each) and the
  // partial sums meet in atomics.
  int split = 1;
  if (K >= 64 && tiles * 2 <= num_sms()) {
    split = (int)(num_sms() / tiles);
    const int64_t max_split = ceil_div(K, 32);
    if (split > max_split) split = (int)max_split;
    if (split < 1) split = 1;
  }
  if (split > 1 && !accumulate) {
    // split-K accumulates atomically: clear the output first
    if (ldc == N) {
      USF_CUDA(cudaMemsetAsync(Cout, 0, sizeof(float) * (size_t)M * (size_t)N, stream));
    } else {
      USF_CUDA(cudaMemset2DAsync(Cout, sizeof(float) * ldc, 0, sizeof(float) * N, (size_t)M, stream));
    }
  }
  dim3 grid((unsigned)ceil_div(M, BM), (unsigned)ceil_div(N, BN), (unsigned)split);
  EpiParams ep{};
  PlainOut po{Cout, ldc, accumulate, split};
  usf_simt_gemm_kernel<false><<<grid, NTHREADS, 0, stream>>>(A, lda, a_trans, W, ldw, w_trans, M, N, K, ep, po);
  USF_LAUNCH_CHECK("usf_simt_gemm_kernel<plain>");
  return USF_OK;
}

// ================================================================================================
// Triangular solve over batch rows:  X E^T = R  (each row r: E x_r = rhs_r), E triangular D x D.
//   element E(i,j) = TRANS ? T[j*D+i] : T[i*D+j], used only inside the triangle; UNIT: implicit 1 diagonal.
// One CTA owns 64 batch rows and walks the 32-wide column blocks in dependency order, accumulating the
// already-solved part with an smem-tiled product and finishing each block by substitution.
// ================================================================================================
namespace {

constexpr int TR = 64, TB = 32;

template <bool LOWER, bool UNIT, bool TRANS>
__global__ void __launch_bounds__(256)
usf_trsm_rows_kernel(const float* __restrict__ T, int64_t D, const float* rhs, int64_t ldr,
                     const float* __restrict__ bias, float* X, int64_t ldx, int64_t B) {
  __shared__ float Xs[TR][TB + 1];
  __shared__ float Es[TB][TB + 1];
  __shared__ float Ts[TR][TB + 1];
  const int tid = threadIdx.x;
  const int c = tid & 31, rg = tid >> 5;  // accumulate mapping: column c, rows rg*8 + i
  const int64_t r0 = (int64_t)blockIdx.x * TR;
  const int nblk = (int)ceil_div(D, TB);

  for (int step = 0; step < nblk; ++step) {
    const int jb = LOWER ? step : nblk - 1 - step;
    const int64_t j0 = (int64_t)jb * TB;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    // already-solved column blocks: k-blocks before jb (LOWER) or after jb (UPPER)
    for (int s2 = 0; s2 < step; ++s2) {
      const int kbk = LOWER ? s2 : nblk - 1 - s2;
      const int64_t k0 = (int64_t)kbk * TB;
      // Xs[r][kk] = X[r0+r][k0+kk]
      for (int e = tid; e < TR * TB; e += 256) {
        const int r = e >> 5, kk = e & 31;
        const int64_t gr = r0 + r, gk = k0 + kk;
        Xs[r][kk] = (gr < B && gk < D) ? X[gr * ldx + gk] : 0.f;
      }
      // Es[cc][kk] = E(j0+cc, k0+kk)
      for (int e = tid; e < TB * TB; e += 256) {
        int cc, kk;
        if (TRANS) { kk = e >> 5; cc = e & 31; } else { cc = e >> 5; kk = e & 31; }
        const int64_t gi = j0 + cc, gk = k0 + kk;
        float v = 0.f;
        if (gi < D && gk < D) v = TRANS ? T[gk * D + gi] : T[gi * D + gk];
        Es[cc][kk] = v;
      }
      __syncthreads();
#pragma unroll 8
      for (int kk = 0; kk < TB; ++kk) {
        const float ev = Es[c][kk];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = fmaf(Xs[rg * 8 + i][kk], ev, acc[i]);
      }
      __syncthreads();
    }
    // Ts = rhs - bias - acc ; Es = diagonal block
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = rg * 8 + i;
      const int64_t gr = r0 + r, gc = j0 + c;
      float v = 0.f;
      if (gr < B && gc < D) {
        v = rhs[gr * ldr + gc] - acc[i];
        if (bias != nullptr) v -= bias[gc];
      }
      Ts[r][c] = v;
    }
    for (int e = tid; e < TB * TB; e += 256) {
      int cc, kk;
      if (TRANS) { kk = e >> 5; cc = e & 31; } else { cc = e >> 5; kk = e & 31; }
      const int64_t gi = j0 + cc, gk = j0 + kk;
      float v = (cc == kk) ? 1.f : 0.f;  // padding keeps the block non-singular
      if (gi < D && gk < D) {
        v = TRANS ? T[gk * D + gi] : T[gi * D + gk];
        if (UNIT && cc == kk) v = 1.f;
      }
      Es[cc][kk] = v;
    }
    __syncthreads();
    if (tid < TR) {
      const int r = tid;
      if (LOWER) {
        for (int cc = 0; cc < TB; ++cc) {
          float xv = Ts[r][cc];
          if (!UNIT) xv /= Es[cc][cc];
          Ts[r][cc] = xv;
          for (int c2 = cc + 1; c2 < TB; ++c2) Ts[r][c2] = fmaf(-xv, Es[c2][cc], Ts[r][c2]);
        }
      } else {
        for (int cc = TB - 1; cc >= 0; --cc) {
          float xv = Ts[r][cc];
          if (!UNIT) xv /= Es[cc][cc];
          Ts[r][cc] = xv;
          for (int c2 = 0; c2 < cc; ++c2) Ts[r][c2] = fmaf(-xv, Es[c2][cc], Ts[r][c2]);
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = rg * 8 + i;
      const int64_t gr = r0 + r, gc = j0 + c;
      if (gr < B && gc < D) X[gr * ldx + gc] = Ts[r][c];
    }
    __syncthreads();  // X writes visible to this CTA's next accumulation pass
  }
}

}  // namespace

int trsm_rows(const float* T, int64_t D, bool lower, bool unit, bool trans, const float* rhs, int64_t ldr,
              const float* bias, float* X, int64_t ldx, int64_t B, cudaStream_t stream) {
  if (B <= 0 || D <= 0) return USF_OK;
  dim3 grid((unsigned)ceil_div(B, TR));
#define USF_TRSM(L, U, TT) usf_trsm_rows_kernel<L, U, TT><<<grid, 256, 0, stream>>>(T, D, rhs, ldr, bias, X, ldx, B)
  if (lower) {
    if (unit) { if (trans) USF_TRSM(true, true, true); else USF_TRSM(true, true, false); }
    else      { if (trans) USF_TRSM(true, false, true); else USF_TRSM(true, false, false); }
  } else {
    if (unit) { if (trans) USF_TRSM(false, true, true); else USF_TRSM(false, true, false); }
    else      { if (trans) USF_TRSM(false, false, true); else USF_TRSM(false, false, false); }
  }
#undef USF_TRSM
  USF_LAUNCH_CHECK("usf_trsm_rows_kernel");
  return USF_OK;
}

// ================================================================================================
// Row kernels: one warp per sample row, 8 rows per CTA.
// ================================================================================================
namespace {

constexpr int ROWS_PER_CTA = 8;

__global__ void usf_householder_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ V,
                                       int nvs, int reverse, float* y, int64_t ldy, int64_t B, int64_t D) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * ROWS_PER_CTA + (threadIdx.x >> 5);
  if (r >= B) return;
  const float* src = x + r * ldx;
  float* dst = y + r * ldy;
  for (int it = 0; it < nvs; ++it) {
    const float* v = V + (int64_t)(reverse ? nvs - 1 - it : it) * D;
    float dot = 0.f, nrm = 0.f;
    for (int64_t d = lane; d < D; d += 32) {
      const float vv = v[d];
      dot = fmaf(src[d], vv, dot);
      nrm = fmaf(vv, vv, nrm);
    }
    dot = warp_sum(dot);
    nrm = warp_sum(nrm);
    const float coef = 2.f * dot / nrm;
    for (int64_t d = lane; d < D; d += 32) dst[d] = fmaf(-coef, v[d], src[d]);
    __syncwarp();
    src = dst;
  }
  if (nvs == 0 && src != dst)
    for (int64_t d = lane; d < D; d += 32) dst[d] = src[d];
}

__global__ void usf_scale_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ scale,
                                 int inverse, float* y, int64_t ldy, int64_t B, int64_t D) {
  // HBM-bound (4*D read + 4*D written per row): 16-byte accesses when the rows allow it, 4 columns per thread
  const bool vec = (D & 3) == 0 && (ldx & 3) == 0 && (ldy & 3) == 0 &&
                   ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(scale)) & 15) == 0;
  if (vec) {
    const int64_t D4 = D >> 2, total4 = B * D4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = i / D4, d4 = i - r * D4;
      const float4 v = *reinterpret_cast<const float4*>(x + r * ldx + 4 * d4);
      const float4 sc = *reinterpret_cast<const float4*>(scale + 4 * d4);
      float4 o;
      if (inverse) { o.x = v.x / sc.x; o.y = v.y / sc.y; o.z = v.z / sc.z; o.w = v.w / sc.w; }
      else { o.x = v.x * sc.x; o.y = v.y * sc.y; o.z = v.z * sc.z; o.w = v.w * sc.w; }
      *reinterpret_cast<float4*>(y + r * ldy + 4 * d4) = o;
    }
    return;
  }
  const int64_t total = B * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D, d = i - r * D;
    const float v = x[r * ldx + d];
    y[r * ldy + d] = inverse ? v / scale[d] : v * scale[d];
  }
}

__global__ void usf_sum_log_abs_kernel(const float* __restrict__ v, int64_t n, int64_t stride, float* out) {
  __shared__ float red[32];
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += logf(fabsf(v[i * stride]));
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    s = warp_sum(s);
    if (threadIdx.x == 0) out[0] = s;
  }
}

// y = m*x + (1-m)*(x*scale+t)  /  y = m*x + (1-m)*((x-t)/scale), ls = clamp*tanh(s)
//   act 0 ("exp", nf4ad/transforms.py:80-82,104-106,129-130):  scale = exp(ls), log-det term = ls
//   act 1 ("softplus", :83-85,107-108,131-132): scale = softplus(ls) + 1e-6, inverse divides by scale + 1e-12, and the
//          log-det term is log(softplus(ls) + 1e-12) -- WITHOUT the 1e-6 of the scale: the reference's own inconsistency,
//          kept so that results match it
__device__ __forceinline__ float softplus_f(float v) { return fmaxf(v, 0.f) + log1pf(expf(-fabsf(v))); }

__global__ void usf_coupling_kernel(const float* x, int64_t ldx, const float* __restrict__ s, int64_t lds,
                                    const float* __restrict__ t, int64_t ldt, const float* __restrict__ mask,
                                    float clamp, int inverse, int act, float* y, int64_t ldy, float* ladj, float ladj_coef,
                                    int64_t B, int64_t D) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * ROWS_PER_CTA + (threadIdx.x >> 5);
  if (r >= B) return;
  float lsum = 0.f;
  for (int64_t d = lane; d < D; d += 32) {
    const float m = mask[d];
    const float xv = x[r * ldx + d];
    const float tv = t[r * ldt + d];
    float ls = 0.f, inner;
    if (s != nullptr) ls = clamp * tanhf(s[r * lds + d]);
    if (act == 0 || s == nullptr) {
      inner = inverse ? (xv - tv) * expf(-ls) : fmaf(xv, expf(ls), tv);
    } else {
      const float sp = softplus_f(ls), sc = sp + 1e-6f;
      inner = inverse ? (xv - tv) / (sc + 1e-12f) : fmaf(xv, sc, tv);
      ls = logf(sp + 1e-12f);
    }
    y[r * ldy + d] = xv * m + (1.f - m) * inner;
    lsum = fmaf(1.f - m, ls, lsum);
  }
  if (ladj != nullptr) {
    lsum = warp_sum(lsum);
    if (lane == 0) ladj[r] += ladj_coef * lsum;
  }
}

__global__ void usf_coupling_bwd_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ dladj,
                                        float ladj_coef, const float* __restrict__ x, int64_t ldx,
                                        const float* __restrict__ s, int64_t lds, const float* __restrict__ t,
                                        int64_t ldt, const float* __restrict__ mask, float clamp, int inverse, int act,
                                        float* dx, int64_t lddx, float* ds, int64_t ldds, float* dt, int64_t lddt,
                                        int64_t B, int64_t D) {
  const int64_t total = B * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D, d = i - r * D;
    const float m = mask[d], om = 1.f - m;
    const float g = dy[r * lddy + d];
    const float xv = x[r * ldx + d];
    const float tv = t[r * ldt + d];
    float th = 0.f, ls = 0.f;
    if (s != nullptr) { th = tanhf(s[r * lds + d]); ls = clamp * th; }
    const float gl = dladj != nullptr ? dladj[r] * ladj_coef : 0.f;
    float gx, gt, gls;
    if (act == 0 || s == nullptr) {
      if (!inverse) {
        const float e = expf(ls);
        gx = g * (m + om * e);
        gt = g * om;
        gls = g * om * xv * e + gl * om;
      } else {
        const float e = expf(-ls);
        gx = g * (m + om * e);
        gt = -g * om * e;
        gls = -g * om * (xv - tv) * e + gl * om;
      }
    } else {
      // scale = softplus(ls) + 1e-6: d scale / d ls = sigmoid(ls); log-det term log(softplus(ls) + 1e-12)
      const float sp = softplus_f(ls), sg = 1.f / (1.f + expf(-ls));
      const float dl = sg / (sp + 1e-12f);
      if (!inverse) {
        const float sc = sp + 1e-6f;
        gx = g * (m + om * sc);
        gt = g * om;
        gls = g * om * xv * sg + gl * om * dl;
      } else {
        const float inv = 1.f / (sp + 1e-6f + 1e-12f);
        gx = g * (m + om * inv);
        gt = -g * om * inv;
        gls = -g * om * (xv - tv) * inv * inv * sg + gl * om * dl;
      }
    }
    dx[r * lddx + d] = gx;
    dt[r * lddt + d] = gt;
    if (ds != nullptr) ds[r * ldds + d] = gls * clamp * (1.f - th * th);
  }
}

__global__ void usf_base_logprob_kernel(int kind, const float* __restrict__ z, int64_t ldz,
                                        const float* __restrict__ loc, const float* __restrict__ scale,
                                        int64_t scale_numel, const float* __restrict__ add, float add_coef,
                                        float* out, int64_t B, int64_t D) {
  // HBM-bound (4*D read per row).  The normalisation sum_d (-log sc_d - const) is the same for every row: each CTA
  // computes it once (all 8 warps together) instead of one logf per element; the data term uses 16-byte loads.
  __shared__ float s_part[ROWS_PER_CTA];
  __shared__ float s_const;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  {
    float c = 0.f;
    for (int64_t d = threadIdx.x; d < D; d += ROWS_PER_CTA * 32) {
      const float sc = scale[scale_numel == 1 ? 0 : d];
      c += kind == 0 ? (-logf(sc) - 0.91893853320467274178f) : -logf(2.f * sc);
    }
    c = warp_sum(c);
    if (lane == 0) s_part[w] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < ROWS_PER_CTA; ++i) t += s_part[i];
      s_const = t;
    }
    __syncthreads();
  }
  // loc and 1/scale staged once per CTA (<= 2048 columns): the row loop is then one 16-byte load + 8 FMA-pipe ops per 4
  // columns, fully unrolled in groups so several loads are in flight per lane
  constexpr int SMAX = 2048;
  __shared__ __align__(16) float s_loc[SMAX];
  __shared__ __align__(16) float s_inv[SMAX];
  const bool staged = D <= SMAX;
  if (staged) {
    for (int64_t d = threadIdx.x; d < D; d += ROWS_PER_CTA * 32) {
      s_loc[d] = loc[d];
      s_inv[d] = 1.f / scale[scale_numel == 1 ? 0 : d];
    }
    __syncthreads();
  }
  const int64_t r = (int64_t)blockIdx.x * ROWS_PER_CTA + w;
  if (r >= B) return;
  const float* zr = z + r * ldz;
  float acc = 0.f;
  const bool vec = staged && (D & 3) == 0 && (ldz & 3) == 0 && (reinterpret_cast<uintptr_t>(z) & 15) == 0;
  if (vec) {
    const int n4 = (int)(D >> 2);
    for (int i0 = lane; i0 < n4; i0 += 128) {
      float4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = i0 + 32 * j;
        v[j] = i < n4 ? *reinterpret_cast<const float4*>(zr + 4 * i) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = i0 + 32 * j;
        if (i < n4) {
          const float4 l = *reinterpret_cast<const float4*>(s_loc + 4 * i);
          const float4 q = *reinterpret_cast<const float4*>(s_inv + 4 * i);
          const float u0 = (v[j].x - l.x) * q.x, u1 = (v[j].y - l.y) * q.y, u2 = (v[j].z - l.z) * q.z, u3 = (v[j].w - l.w) * q.w;
          if (kind == 0) acc += -0.5f * (u0 * u0 + u1 * u1 + u2 * u2 + u3 * u3);
          else acc += -(fabsf(u0) + fabsf(u1) + fabsf(u2) + fabsf(u3));
        }
      }
    }
  } else {
    for (int64_t d = lane; d < D; d += 32) {
      const float sc = scale[scale_numel == 1 ? 0 : d];
      const float u = (zr[d] - loc[d]) / sc;
      acc += kind == 0 ? -0.5f * u * u : -fabsf(u);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) out[r] = acc + s_const + (add != nullptr ? add_coef * add[r] : 0.f);
}

// dz = dout * dlogp/dz ; column sums for loc / scale grads via atomics (one partial per warp-row).
__global__ void usf_base_logprob_bwd_kernel(int kind, const float* __restrict__ dout, const float* __restrict__ z,
                                            int64_t ldz, const float* __restrict__ loc, const float* __restrict__ scale,
                                            int64_t scale_numel, float* dz, int64_t lddz, float* dloc, float* dscale,
                                            int64_t B, int64_t D) {
  // thread per column chunk: block handles 32 columns x all rows strided by gridDim.y
  const int64_t d = (int64_t)blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;  // 0..7
  float gl = 0.f, gs = 0.f;
  if (d < D) {
    const float sc = scale[scale_numel == 1 ? 0 : d];
    const float lc = loc[d];
    for (int64_t r = (int64_t)blockIdx.y * 8 + rl; r < B; r += (int64_t)gridDim.y * 8) {
      const float g = dout[r];
      const float u = (z[r * ldz + d] - lc) / sc;
      float dzv, dsc;
      if (kind == 0) { dzv = -u / sc; dsc = (u * u - 1.f) / sc; }
      else { const float sg = (u > 0.f) - (u < 0.f); dzv = -sg / sc; dsc = (fabsf(u) - 1.f) / sc; }
      if (dz != nullptr) dz[r * lddz + d] = g * dzv;
      gl += -g * dzv;
      gs += g * dsc;
    }
  }
  __shared__ float sl[8][33], ss[8][33];
  sl[rl][threadIdx.x & 31] = gl;
  ss[rl][threadIdx.x & 31] = gs;
  __syncthreads();
  if (rl == 0 && d < D) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < 8; ++i) { a += sl[i][threadIdx.x]; b += ss[i][threadIdx.x]; }
    if (dloc != nullptr) atomicAdd(dloc + d, a);
    if (dscale != nullptr) atomicAdd(dscale + (scale_numel == 1 ? 0 : d), b);
  }
}

// Householder backward for ONE reflection: given input x (before this reflection), dy -> dx, dv +=.
//   y = x - c v, c = 2 (x.v)/(v.v);  dx = dy - (2 (dy.v)/(v.v)) v
//   dv += -c dy - (2 (dy.v)/(v.v)) x + (4 (x.v)(dy.v)/(v.v)^2) v     (per row, reduced over rows)
__global__ void usf_householder_bwd_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ x,
                                           int64_t ldx, const float* __restrict__ v, float* dx, int64_t lddx,
                                           float* dv, int64_t B, int64_t D) {
  extern __shared__ float dv_s[];  // D floats, CTA-local accumulation of dv
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) dv_s[d] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int64_t r = (int64_t)blockIdx.x * nw + wid; r < B; r += (int64_t)gridDim.x * nw) {
    float xv = 0.f, gv = 0.f, vv = 0.f;
    for (int64_t d = lane; d < D; d += 32) {
      const float ve = v[d];
      xv = fmaf(x[r * ldx + d], ve, xv);
      gv = fmaf(dy[r * lddy + d], ve, gv);
      vv = fmaf(ve, ve, vv);
    }
    xv = warp_sum(xv); gv = warp_sum(gv); vv = warp_sum(vv);
    const float c = 2.f * xv / vv, e = 2.f * gv / vv, f = 4.f * xv * gv / (vv * vv);
    for (int64_t d = lane; d < D; d += 32) {
      const float g = dy[r * lddy + d], ve = v[d], xe = x[r * ldx + d];
      dx[r * lddx + d] = fmaf(-e, ve, g);
      atomicAdd(&dv_s[d], -c * g - e * xe + f * ve);
    }
  }
  __syncthreads();
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) atomicAdd(dv + d, dv_s[d]);
}

// Backward of y = x*scale (inverse: y = x/scale). `xy` is the layer input x (forward) or OUTPUT y (inverse).
//   forward: dx = dy*scale, dscale[d] += sum_b dy*x ;  inverse: dx = dy/scale, dscale[d] += -sum_b dy*y/scale
__global__ void usf_scale_bwd_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ xy,
                                     int64_t ldxy, const float* __restrict__ scale, int inverse, float* dx,
                                     int64_t lddx, float* dscale, int64_t B, int64_t D) {
  const int64_t d = (int64_t)blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;
  float gs = 0.f;
  if (d < D) {
    const float sc = scale[d];
    for (int64_t r = (int64_t)blockIdx.y * 8 + rl; r < B; r += (int64_t)gridDim.y * 8) {
      const float g = dy[r * lddy + d];
      const float v = xy[r * ldxy + d];
      if (!inverse) { dx[r * lddx + d] = g * sc; gs += g * v; }
      else { dx[r * lddx + d] = g / sc; gs -= g * v / sc; }
    }
  }
  __shared__ float sm[8][33];
  sm[rl][threadIdx.x & 31] = gs;
  __syncthreads();
  if (rl == 0 && d < D && dscale != nullptr) {
    float a = 0.f;
    for (int i = 0; i < 8; ++i) a += sm[i][threadIdx.x];
    atomicAdd(dscale + d, a);
  }
}

__global__ void usf_colsum_kernel(const float* __restrict__ a, int64_t lda, float* out, float coef, int64_t B,
                                  int64_t N) {
  // grid (N/32, row slices): each CTA reduces its row slice of 32 columns and adds ONE partial per column atomically
  const int64_t c = (int64_t)blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;
  float s = 0.f;
  if (c < N)
    for (int64_t r = (int64_t)blockIdx.y * 8 + rl; r < B; r += (int64_t)gridDim.y * 8) s += a[r * lda + c];
  __shared__ float sm[8][33];
  sm[rl][threadIdx.x & 31] = s;
  __syncthreads();
  if (rl == 0 && c < N) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sm[i][threadIdx.x];
    atomicAdd(out + c, coef * t);
  }
}

__global__ void usf_relu_mask_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ y,
                                     int64_t ldy, float* out, int64_t B, int64_t N) {
  const int64_t total = B * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / N, c = i - r * N;
    out[i] = y[r * ldy + c] > 0.f ? dy[r * lddy + c] : 0.f;
  }
}

// mode 0: out = tril(src,-1) + I ; mode 1: out = triu(src)
__global__ void usf_tri_copy_kernel(const float* __restrict__ src, float* out, int64_t D, int mode) {
  const int64_t total = D * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D, c = i - r * D;
    float v;
    if (mode == 0) v = c < r ? src[i] : (c == r ? 1.f : 0.f);
    else v = c >= r ? src[i] : 0.f;
    out[i] = v;
  }
}

// mode 0: dst += strict_lower(src) ; mode 1: dst += upper(src) (+ dlogdet / U_ii on the diagonal)
__global__ void usf_tri_add_kernel(const float* __restrict__ src, float* dst, int64_t D, int mode,
                                   const float* __restrict__ U_raw, float dlogdet) {
  const int64_t total = D * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D, c = i - r * D;
    if (mode == 0) { if (c < r) dst[i] += src[i]; }
    else {
      if (c >= r) dst[i] += src[i];
      if (c == r && dlogdet != 0.f) dst[i] += dlogdet / U_raw[i];
    }
  }
}

__global__ void usf_pack_matrix_kernel(const float* __restrict__ src, int64_t lds, const int32_t* __restrict__ row_idx,
                                       const int32_t* __restrict__ col_idx, int sub_row0, int transpose_src,
                                       int64_t n_rows, int64_t n_cols, float* out, __nv_bfloat16* out_bf16,
                                       int64_t ldo) {
  const int64_t total = n_rows * ldo;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ldo, c = i - r * ldo;
    float v = 0.f;
    if (c < n_cols) {
      const int64_t sr = row_idx ? row_idx[r] : r;
      const int64_t sc = col_idx ? col_idx[c] : c;
      if (sr >= 0 && sc >= 0) {
        if (!transpose_src) {
          v = src[sr * lds + sc];
          if (sub_row0) v -= src[sc];
        } else {  // out[r,c] = src[col_idx[c], row_idx[r]] - src[0, row_idx[r]]
          v = src[sc * lds + sr];
          if (sub_row0) v -= src[sr];
        }
      }
    }
    if (out) out[i] = v;
    if (out_bf16) out_bf16[i] = __float2bfloat16_rn(v);
  }
}

// fp32 (B,D) -> bf16 and/or fp32 copy with padded leading dimension (pad columns zeroed); optional row_init.
// Each thread converts 8 consecutive columns (ldy is a multiple of 8): two 16-byte loads when the source
// row is 16-byte aligned, one 16-byte bf16 store (or two fp32 stores).  HBM-bound: 4*D B read + 2*ldy B written.
__global__ void usf_convert_rows_kernel(const float* __restrict__ x, int64_t ldx, __nv_bfloat16* yb, float* yf,
                                        int64_t ldy, int64_t B, int64_t D, float* row_init, float init_value) {
  const int64_t groups = ldy >> 3;
  const int64_t total = B * groups;
  const bool vec_ok = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / groups, c = (i - r * groups) << 3;
    float v[8];
    const float* src = x + r * ldx + c;
    if (vec_ok && c + 8 <= D) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(src));
      const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 1);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = c + j < D ? src[j] : 0.f;
    }
    if (yb) {
      uint4 q;
      __nv_bfloat162 h;
      h = __floats2bfloat162_rn(v[0], v[1]); q.x = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(v[2], v[3]); q.y = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(v[4], v[5]); q.z = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(v[6], v[7]); q.w = *reinterpret_cast<uint32_t*>(&h);
      *reinterpret_cast<uint4*>(yb + r * ldy + c) = q;
    }
    if (yf) {
      float4* dst = reinterpret_cast<float4*>(yf + r * ldy + c);
      dst[0] = make_float4(v[0], v[1], v[2], v[3]);
      dst[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    if (c == 0 && row_init) row_init[r] = init_value;
  }
}

// The same stage for rows that arrive as bf16 already (usf_stack_run_bf16in: the host narrowed them before the
// PCIe copy): a padded copy, 8 columns per thread.
__global__ void usf_copy_rows_bf16_kernel(const uint16_t* __restrict__ x, int64_t ldx, uint16_t* y, int64_t ldy, int64_t B,
                                          int64_t D, float* row_init, float init_value) {
  const int64_t groups = ldy >> 3;
  const int64_t total = B * groups;
  const bool vec_ok = ((ldx & 7) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / groups, c = (i - r * groups) << 3;
    const uint16_t* src = x + r * ldx + c;
    uint4 q;
    if (vec_ok && c + 8 <= D) {
      q = __ldg(reinterpret_cast<const uint4*>(src));
    } else {
      uint16_t v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = c + j < D ? src[j] : (uint16_t)0;
      q.x = v[0] | ((uint32_t)v[1] << 16); q.y = v[2] | ((uint32_t)v[3] << 16);
      q.z = v[4] | ((uint32_t)v[5] << 16); q.w = v[6] | ((uint32_t)v[7] << 16);
    }
    *reinterpret_cast<uint4*>(y + r * ldy + c) = q;
    if (c == 0 && row_init) row_init[r] = init_value;
  }
}

__global__ void usf_bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, float* y, int64_t ldy,
                                       int64_t B, int64_t D) {
  const int64_t total = B * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D, c = i - r * D;
    y[r * ldy + c] = __bfloat162float(x[r * ldx + c]);
  }
}

inline unsigned ew_grid(int64_t total, int threads = 256) {
  int64_t g = ceil_div(total, threads);
  const int64_t cap = (int64_t)num_sms() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

}  // namespace

int launch_colsum(const float* a, int64_t lda, float* out, float coef, int accumulate, int64_t B, int64_t N,
                  cudaStream_t stream) {
  if (!accumulate) USF_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)N, stream));
  if (B <= 0) return USF_OK;
  int gy = (int)ceil_div(B, 8 * 32);
  if (gy < 1) gy = 1;
  if (gy > 64) gy = 64;
  dim3 grid((unsigned)ceil_div(N, 32), (unsigned)gy);
  usf_colsum_kernel<<<grid, 256, 0, stream>>>(a, lda, out, coef, B, N);
  USF_LAUNCH_CHECK("usf_colsum_kernel");
  return USF_OK;
}

int launch_convert_rows(const float* x, int64_t ldx, uint16_t* y_bf16, float* y_f32, int64_t ldy, int64_t B,
                        int64_t D, float* row_init, float init_value, cudaStream_t stream) {
  if (B <= 0) return USF_OK;
  if ((ldy & 7) != 0 || (reinterpret_cast<uintptr_t>(y_bf16) & 15) != 0 || (reinterpret_cast<uintptr_t>(y_f32) & 15) != 0) {
    set_error("convert_rows: destination must be 16-byte aligned with ld %% 8 == 0");
    return USF_E_ARG;
  }
  usf_convert_rows_kernel<<<ew_grid(B * (ldy >> 3)), 256, 0, stream>>>(
      x, ldx, reinterpret_cast<__nv_bfloat16*>(y_bf16), y_f32, ldy, B, D, row_init, init_value);
  USF_LAUNCH_CHECK("usf_convert_rows_kernel");
  return USF_OK;
}

int launch_copy_rows_bf16(const uint16_t* x, int64_t ldx, uint16_t* y, int64_t ldy, int64_t B, int64_t D, float* row_init,
                          float init_value, cudaStream_t stream) {
  if (B <= 0) return USF_OK;
  if ((ldy & 7) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0) {
    set_error("copy_rows_bf16: destination must be 16-byte aligned with ld %% 8 == 0");
    return USF_E_ARG;
  }
  usf_copy_rows_bf16_kernel<<<ew_grid(B * (ldy >> 3)), 256, 0, stream>>>(x, ldx, y, ldy, B, D, row_init, init_value);
  USF_LAUNCH_CHECK("usf_copy_rows_bf16_kernel");
  return USF_OK;
}

int launch_bf16_to_f32(const uint16_t* x, int64_t ldx, float* y, int64_t ldy, int64_t B, int64_t D,
                       cudaStream_t stream) {
  if (B <= 0) return USF_OK;
  usf_bf16_to_f32_kernel<<<ew_grid(B * D), 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), ldx, y, ldy, B, D);
  USF_LAUNCH_CHECK("usf_bf16_to_f32_kernel");
  return USF_OK;
}

}  // namespace usf

// ================================================================================================
// extern "C" layer entry points
// ================================================================================================
using namespace usf;

extern "C" int usf_lu_pack(const float* L_raw, const float* U_raw, int64_t D, float* W, float* logabsdet,
                           float* scratch, usf_stream_t stream) {
  USF_CHECK_ARG(L_raw && U_raw && W && scratch && D > 0, "usf_lu_pack: null pointer or D <= 0");
  cudaStream_t st = as_stream(stream);
  float* Lm = scratch;
  float* Um = scratch + D * D;
  usf_tri_copy_kernel<<<ew_grid(D * D), 256, 0, st>>>(L_raw, Lm, D, 0);
  usf_tri_copy_kernel<<<ew_grid(D * D), 256, 0, st>>>(U_raw, Um, D, 1);
  USF_LAUNCH_CHECK("usf_tri_copy_kernel");
  // W[i,j] = sum_k Lm[i,k] Um[k,j] : A = Lm (k contiguous), operand "W"(n=j,k) = Um[k*D+j] -> w_trans
  int rc = simt_gemm_plain(Lm, D, 0, Um, D, 1, D, D, D, W, D, 0, st);
  if (rc) return rc;
  if (logabsdet) {
    usf_sum_log_abs_kernel<<<1, 256, 0, st>>>(U_raw, D, D + 1, logabsdet);
    USF_LAUNCH_CHECK("usf_sum_log_abs_kernel");
  }
  return USF_OK;
}

namespace usf {
namespace {
// Operand preparation of the tensor-core training GEMMs.  One pass over an fp32 (B x N) matrix x (optionally gated by
// a ReLU output: v = mask[r,c] > 0 ? x[r,c] : 0) writes any of: a bf16 row-major copy (B x ldr, pad columns zero), a
// bf16 TRANSPOSED copy (N x ldt, pad columns zero: operand of the weight-gradient GEMM, which reduces over the
// batch), and the fp32 column sums (bias gradient; atomically accumulated, caller zeroes).  32x32 tiles through smem.
__global__ void usf_to_bf16_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mask, int64_t ldm,
                                   __nv_bfloat16* rows, int64_t ldr, __nv_bfloat16* tr, int64_t ldt, float* colsum,
                                   int64_t B, int64_t N, int64_t Bp, int64_t Np) {
  __shared__ float tile[32][33];
  // the tensor-core GEMM that consumes this pass is launched with programmatic stream serialization: let it run its
  // prologue (barrier init, TMEM allocation, tensor-map prefetch, cluster sync: 3-4 us) beside this kernel; it waits
  // (griddepcontrol.wait) for this grid to complete before it touches the operands
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  float cs = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = r0 + ty + 8 * i, c = c0 + tx;
    float v = 0.f;
    if (r < B && c < N) {
      v = x[r * ldx + c];
      if (mask != nullptr && !(mask[r * ldm + c] > 0.f)) v = 0.f;
    }
    tile[ty + 8 * i][tx] = v;
    cs += v;
    if (rows != nullptr && r < B && c < Np) rows[r * ldr + c] = __float2bfloat16_rn(v);
  }
  if (colsum != nullptr) {
    __shared__ float part[8][32];
    part[ty][tx] = cs;
    __syncthreads();
    if (ty == 0 && c0 + tx < N) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += part[i][tx];
      atomicAdd(colsum + c0 + tx, t);
    }
  }
  if (tr != nullptr) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t c = c0 + ty + 8 * i, r = r0 + tx;     // tr[c, r] = x[r, c]
      if (c < N && r < Bp) tr[c * ldt + r] = __float2bfloat16_rn(tile[tx][ty + 8 * i]);
    }
  }
}

// The same pass with 16-byte accesses: a 64 x 64 tile per CTA, float4 loads, bf16x4 stores in both orientations (the
// element-wise form above moves 2 bytes per thread and store: 2.3-2.9 TB/s on the 4096-row activations of the
// training step, where it is a quarter of the batch-sized chain).  Needs 16-byte aligned rows (x, mask) and 8-byte
// aligned output rows: usf_to_bf16 falls back otherwise.
__global__ void __launch_bounds__(256)
usf_to_bf16_v4_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mask, int64_t ldm,
                      __nv_bfloat16* rows, int64_t ldr, __nv_bfloat16* tr, int64_t ldt, float* colsum, int64_t B,
                      int64_t N, int64_t Bp, int64_t Np) {
  __shared__ float tile[64][65];
  __shared__ float part[16][64];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // (see usf_to_bf16_kernel)
  const int t = threadIdx.x;
  const int q = t & 15, g = t >> 4;                  // 16 threads x 4 columns across a row, 16 rows per pass
  const int64_t c0 = (int64_t)blockIdx.x * 64, r0 = (int64_t)blockIdx.y * 64;
  const int64_t c = c0 + 4 * q;
  float cs0 = 0.f, cs1 = 0.f, cs2 = 0.f, cs3 = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = g + 16 * i;
    const int64_t r = r0 + rl;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < B && c < N) {
      if (c + 4 <= N) {
        v = *reinterpret_cast<const float4*>(x + r * ldx + c);
        if (mask != nullptr) {
          const float4 m = *reinterpret_cast<const float4*>(mask + r * ldm + c);
          if (!(m.x > 0.f)) v.x = 0.f;
          if (!(m.y > 0.f)) v.y = 0.f;
          if (!(m.z > 0.f)) v.z = 0.f;
          if (!(m.w > 0.f)) v.w = 0.f;
        }
      } else {                                        // ragged last columns (N % 4 != 0)
        float e[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < 4 && c + j < N; ++j) {
          e[j] = x[r * ldx + c + j];
          if (mask != nullptr && !(mask[r * ldm + c + j] > 0.f)) e[j] = 0.f;
        }
        v = make_float4(e[0], e[1], e[2], e[3]);
      }
    }
    tile[rl][4 * q] = v.x; tile[rl][4 * q + 1] = v.y; tile[rl][4 * q + 2] = v.z; tile[rl][4 * q + 3] = v.w;
    cs0 += v.x; cs1 += v.y; cs2 += v.z; cs3 += v.w;
    if (rows != nullptr && r < B && c < Np) {         // (Np % 4 == 0: whole groups)
      const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
      uint2 o;
      o.x = *reinterpret_cast<const uint32_t*>(&lo);
      o.y = *reinterpret_cast<const uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(rows + r * ldr + c) = o;
    }
  }
  if (colsum != nullptr) {
    part[g][4 * q] = cs0; part[g][4 * q + 1] = cs1; part[g][4 * q + 2] = cs2; part[g][4 * q + 3] = cs3;
  }
  __syncthreads();
  if (colsum != nullptr && t < 64 && c0 + t < N) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) a += part[i][t];
    atomicAdd(colsum + c0 + t, a);
  }
  if (tr != nullptr) {
    // tr[cc, r0 + 4 q .. + 3] = x[r0 + 4 q .. + 3, cc]: 16 threads x 4 rows along one output row, 16 columns per pass
    const int64_t r = r0 + 4 * q;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int cl = g + 16 * i;
      const int64_t cc = c0 + cl;
      if (cc < N && r < Bp) {                         // (Bp % 4 == 0: whole groups; rows past B hold zeros)
        const __nv_bfloat162 lo = __floats2bfloat162_rn(tile[4 * q][cl], tile[4 * q + 1][cl]);
        const __nv_bfloat162 hi = __floats2bfloat162_rn(tile[4 * q + 2][cl], tile[4 * q + 3][cl]);
        uint2 o;
        o.x = *reinterpret_cast<const uint32_t*>(&lo);
        o.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(tr + cc * ldt + r) = o;
      }
    }
  }
}

// Same pass for the 3xTF32 training GEMMs: every output is an fp32 (hi, lo) pair, hi = value rounded to tf32,
// lo = value - hi (see usf_tc3_gemm_kernel).
__global__ void usf_to_tf32x3_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mask, int64_t ldm,
                                     float* rows_hi, float* rows_lo, int64_t ldr, float* tr_hi, float* tr_lo, int64_t ldt,
                                     float* colsum, int64_t B, int64_t N, int64_t Bp, int64_t Np) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  float cs = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = r0 + ty + 8 * i, c = c0 + tx;
    float v = 0.f;
    if (r < B && c < N) {
      v = x[r * ldx + c];
      if (mask != nullptr && !(mask[r * ldm + c] > 0.f)) v = 0.f;
    }
    tile[ty + 8 * i][tx] = v;
    cs += v;
    if (rows_hi != nullptr && r < B && c < Np) {
      const float h = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
      rows_hi[r * ldr + c] = h;
      rows_lo[r * ldr + c] = v - h;
    }
  }
  if (colsum != nullptr) {
    __shared__ float part[8][32];
    part[ty][tx] = cs;
    __syncthreads();
    if (ty == 0 && c0 + tx < N) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += part[i][tx];
      atomicAdd(colsum + c0 + tx, t);
    }
  }
  if (tr_hi != nullptr) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t c = c0 + ty + 8 * i, r = r0 + tx;     // tr[c, r] = x[r, c]
      if (c < N && r < Bp) {
        const float v = tile[tx][ty + 8 * i];
        const float h = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
        tr_hi[c * ldt + r] = h;
        tr_lo[c * ldt + r] = v - h;
      }
    }
  }
}

// y[r, c] = act(y[r, c] + bias[c]) in place: second phase of the split-K form of usf_linear
__global__ void usf_bias_act_kernel(float* y, int64_t ldy, const float* __restrict__ bias, int relu, int64_t B, int64_t N) {
  const int64_t total = B * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / N, c = i - r * N;
    float v = y[r * ldy + c] + (bias != nullptr ? bias[c] : 0.f);
    y[r * ldy + c] = relu ? fmaxf(v, 0.f) : v;
  }
}
}  // namespace
}  // namespace usf

extern "C" int usf_to_bf16(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, uint16_t* rows, int64_t ldr,
                           uint16_t* transposed, int64_t ldt, float* colsum, int64_t B, int64_t N, usf_stream_t stream) {
  USF_CHECK_ARG(x != nullptr && B >= 0 && N > 0 && ldx >= N, "usf_to_bf16: bad arguments");
  USF_CHECK_ARG(rows == nullptr || ldr >= N, "usf_to_bf16: ldr < N");
  USF_CHECK_ARG(transposed == nullptr || ldt >= B, "usf_to_bf16: ldt < B");
  if (B == 0) return USF_OK;
  // pad columns up to the leading dimension are written as zeros (B x ldr and N x ldt are fully defined)
  const int64_t Np = rows != nullptr ? ldr : N, Bp = transposed != nullptr ? ldt : B;
  const bool vec4 = (ldx % 4) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                    (relu_mask == nullptr || ((ldm % 4) == 0 && (reinterpret_cast<uintptr_t>(relu_mask) & 15) == 0)) &&
                    (rows == nullptr || ((ldr % 4) == 0 && (reinterpret_cast<uintptr_t>(rows) & 7) == 0)) &&
                    (transposed == nullptr || ((ldt % 4) == 0 && (reinterpret_cast<uintptr_t>(transposed) & 7) == 0));
  // (small matrices -- the D x D weight-space operands -- keep the 32 x 32 tiles: 64 x 64 would leave most SMs idle)
  if (vec4 && ceil_div(Np > N ? Np : N, 64) * ceil_div(Bp > B ? Bp : B, 64) >= 2 * 148) {
    dim3 grid4((unsigned)ceil_div(Np > N ? Np : N, 64), (unsigned)ceil_div(Bp > B ? Bp : B, 64));
    usf_to_bf16_v4_kernel<<<grid4, 256, 0, as_stream(stream)>>>(
        x, ldx, relu_mask, ldm, reinterpret_cast<__nv_bfloat16*>(rows), ldr, reinterpret_cast<__nv_bfloat16*>(transposed),
        ldt, colsum, B, N, Bp, Np);
    USF_LAUNCH_CHECK("usf_to_bf16_v4_kernel");
    return USF_OK;
  }
  dim3 grid((unsigned)ceil_div(Np > N ? Np : N, 32), (unsigned)ceil_div(Bp > B ? Bp : B, 32));
  usf_to_bf16_kernel<<<grid, dim3(32, 8), 0, as_stream(stream)>>>(
      x, ldx, relu_mask, ldm, reinterpret_cast<__nv_bfloat16*>(rows), ldr, reinterpret_cast<__nv_bfloat16*>(transposed), ldt,
      colsum, B, N, Bp, Np);
  USF_LAUNCH_CHECK("usf_to_bf16_kernel");
  return USF_OK;
}

extern "C" int usf_to_tf32x3(const float* x, int64_t ldx, const float* relu_mask, int64_t ldm, float* rows_hi,
                             float* rows_lo, int64_t ldr, float* t_hi, float* t_lo, int64_t ldt, float* colsum, int64_t B,
                             int64_t N, usf_stream_t stream) {
  USF_CHECK_ARG(x != nullptr && B >= 0 && N > 0 && ldx >= N, "usf_to_tf32x3: bad arguments");
  USF_CHECK_ARG((rows_hi == nullptr) == (rows_lo == nullptr) && (t_hi == nullptr) == (t_lo == nullptr),
                "usf_to_tf32x3: hi and lo outputs come in pairs");
  USF_CHECK_ARG(rows_hi == nullptr || ldr >= N, "usf_to_tf32x3: ldr < N");
  USF_CHECK_ARG(t_hi == nullptr || ldt >= B, "usf_to_tf32x3: ldt < B");
  if (B == 0) return USF_OK;
  const int64_t Np = rows_hi != nullptr ? ldr : N, Bp = t_hi != nullptr ? ldt : B;
  dim3 grid((unsigned)ceil_div(Np > N ? Np : N, 32), (unsigned)ceil_div(Bp > B ? Bp : B, 32));
  usf_to_tf32x3_kernel<<<grid, dim3(32, 8), 0, as_stream(stream)>>>(x, ldx, relu_mask, ldm, rows_hi, rows_lo, ldr, t_hi, t_lo,
                                                                   ldt, colsum, B, N, Bp, Np);
  USF_LAUNCH_CHECK("usf_to_tf32x3_kernel");
  return USF_OK;
}

extern "C" int usf_linear(const float* x, int64_t ldx, const float* W, int64_t ldw, const float* bias, int relu,
                          float* y, int64_t ldy, int64_t B, int64_t N, int64_t K, usf_stream_t stream) {
  USF_CHECK_ARG(W && ((x && y) || B == 0), "usf_linear: null pointer");   // (an empty batch may come with NULL rows)
  USF_CHECK_ARG(B >= 0 && N > 0 && K > 0 && ldx >= K && ldw >= K && ldy >= N, "usf_linear: bad sizes");
  if (B > 0 && K >= 64 && ceil_div(B, BM) * ceil_div(N, BN) * 2 <= num_sms()) {
    // small problem: split-K GEMM (atomic partial sums) + a bias/activation pass, instead of a few serial tiles
    int rc = simt_gemm_plain(x, ldx, 0, W, ldw, 0, B, N, K, y, ldy, 0, as_stream(stream));
    if (rc) return rc;
    usf_bias_act_kernel<<<ew_grid(B * N), 256, 0, as_stream(stream)>>>(y, ldy, bias, relu, B, N);
    USF_LAUNCH_CHECK("usf_bias_act_kernel");
    return USF_OK;
  }
  EpiParams ep{};
  ep.mode = relu ? EPI_BIAS_RELU : EPI_BIAS;
  ep.bias = bias;
  ep.out = y;
  ep.ldo = ldy;
  return simt_gemm(x, ldx, 0, W, ldw, 0, B, N, K, ep, as_stream(stream));
}

extern "C" int64_t usf_lu_solve_scratch_floats(int64_t D) { return D > 0 ? trsm_fast_scratch_floats(D) : 0; }

extern "C" int usf_lu_solve(const float* y, int64_t ldy, const float* L_raw, const float* U_raw, const float* bias,
                            int transpose, float* x, int64_t ldx, int64_t B, int64_t D, float* scratch,
                            usf_stream_t stream) {
  USF_CHECK_ARG(y && L_raw && U_raw && x && D > 0 && B >= 0, "usf_lu_solve: null pointer or bad size");
  cudaStream_t st = as_stream(stream);
  const bool fast = scratch != nullptr && trsm_fast_supported(D);
  auto solve = [&](const float* T, bool lower, bool unit, bool trans, const float* rhs, int64_t ldr, const float* b) {
    if (fast) return trsm_rows_fast(T, D, lower, unit, trans, rhs, ldr, b, x, ldx, B, scratch, st);
    return trsm_rows(T, D, lower, unit, trans, rhs, ldr, b, x, ldx, B, st);
  };
  int rc;
  if (!transpose) {
    // L z = y - b (unit lower), U x = z (upper)
    rc = solve(L_raw, true, true, false, y, ldy, bias);
    if (rc) return rc;
    return solve(U_raw, false, false, false, x, ldx, nullptr);
  }
  // (LU)^T x = y : U^T z = y (lower, non-unit), L^T x = z (upper, unit)
  rc = solve(U_raw, true, false, true, y, ldy, bias);
  if (rc) return rc;
  return solve(L_raw, false, true, true, x, ldx, nullptr);
}

extern "C" int64_t usf_lu_inverse_scratch_floats(int64_t D) {
  return D > 0 && trsm_fast_supported(D) ? lu_inverse_scratch_floats(D) : 0;
}

extern "C" int usf_lu_inverse(const float* L_raw, const float* U_raw, int64_t D, float* A, float* scratch,
                              usf_stream_t stream) {
  USF_CHECK_ARG(L_raw && U_raw && scratch && D > 0, "usf_lu_inverse: null pointer or bad size");
  USF_CHECK_ARG(trsm_fast_supported(D), "usf_lu_inverse: D too large for the resident solve (use usf_lu_solve)");
  return lu_inverse(L_raw, U_raw, D, A, scratch, as_stream(stream));
}

extern "C" int usf_householder(const float* x, int64_t ldx, const float* V, int64_t nvs, int reverse, float* y,
                               int64_t ldy, int64_t B, int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(x && y && (V || nvs == 0) && D > 0 && B >= 0 && nvs >= 0, "usf_householder: bad arguments");
  if (B == 0) return USF_OK;
  usf_householder_kernel<<<(unsigned)ceil_div(B, ROWS_PER_CTA), ROWS_PER_CTA * 32, 0, as_stream(stream)>>>(
      x, ldx, V, (int)nvs, reverse, y, ldy, B, D);
  USF_LAUNCH_CHECK("usf_householder_kernel");
  return USF_OK;
}

extern "C" int usf_scale(const float* x, int64_t ldx, const float* scale, int inverse, float* y, int64_t ldy,
                         int64_t B, int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(x && y && scale && D > 0 && B >= 0, "usf_scale: bad arguments");
  if (B == 0) return USF_OK;
  usf_scale_kernel<<<ew_grid(B * D), 256, 0, as_stream(stream)>>>(x, ldx, scale, inverse, y, ldy, B, D);
  USF_LAUNCH_CHECK("usf_scale_kernel");
  return USF_OK;
}

extern "C" int usf_sum_log_abs(const float* v, int64_t n, int64_t stride, float* out, usf_stream_t stream) {
  USF_CHECK_ARG(v && out && n >= 0 && stride > 0, "usf_sum_log_abs: bad arguments");
  usf_sum_log_abs_kernel<<<1, 256, 0, as_stream(stream)>>>(v, n, stride, out);
  USF_LAUNCH_CHECK("usf_sum_log_abs_kernel");
  return USF_OK;
}

extern "C" int usf_coupling(const float* x, int64_t ldx, const float* s, int64_t lds, const float* t, int64_t ldt,
                            const float* mask, float clamp, int inverse, int scale_activation, float* y, int64_t ldy,
                            float* ladj, float ladj_coef, int64_t B, int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(x && t && mask && y && D > 0 && B >= 0, "usf_coupling: bad arguments");
  USF_CHECK_ARG(scale_activation == 0 || scale_activation == 1, "usf_coupling: scale_activation must be 0 (exp) or 1 (softplus)");
  if (B == 0) return USF_OK;
  usf_coupling_kernel<<<(unsigned)ceil_div(B, ROWS_PER_CTA), ROWS_PER_CTA * 32, 0, as_stream(stream)>>>(
      x, ldx, s, lds, t, ldt, mask, clamp, inverse, scale_activation, y, ldy, ladj, ladj_coef, B, D);
  USF_LAUNCH_CHECK("usf_coupling_kernel");
  return USF_OK;
}

extern "C" int usf_base_logprob(int kind, const float* z, int64_t ldz, const float* loc, const float* scale,
                                int64_t scale_numel, const float* add, float add_coef, float* out, int64_t B,
                                int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(z && loc && scale && out && D > 0 && B >= 0, "usf_base_logprob: bad arguments");
  USF_CHECK_ARG(kind == 0 || kind == 1, "usf_base_logprob: kind must be 0 (Normal) or 1 (Laplace)");
  USF_CHECK_ARG(scale_numel == 1 || scale_numel == D, "usf_base_logprob: scale_numel must be 1 or D");
  if (B == 0) return USF_OK;
  usf_base_logprob_kernel<<<(unsigned)ceil_div(B, ROWS_PER_CTA), ROWS_PER_CTA * 32, 0, as_stream(stream)>>>(
      kind, z, ldz, loc, scale, scale_numel, add, add_coef, out, B, D);
  USF_LAUNCH_CHECK("usf_base_logprob_kernel");
  return USF_OK;
}

extern "C" size_t usf_linear_bwd_scratch_bytes(int64_t B, int64_t N) {
  return sizeof(float) * (size_t)(B > 0 ? B : 0) * (size_t)(N > 0 ? N : 0);
}

extern "C" int usf_linear_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* W,
                              int64_t ldw, const float* y_relu, int64_t ldyr, float* dx, int64_t lddx, float* dW,
                              int64_t lddw, float* db, int accumulate, float* scratch, int64_t B, int64_t N,
                              int64_t K, usf_stream_t stream) {
  // an empty batch may come with NULL rows (dy, x); it still defines dW = 0 and db = 0 when accumulate == 0, so it runs
  // through the same steps: the dgrad GEMM returns at M = 0, the wgrad GEMM stores (or adds) a K = 0 product, the
  // column sum clears its output before it looks at B
  USF_CHECK_ARG((dy || B == 0) && B >= 0 && N > 0 && K > 0, "usf_linear_bwd: bad arguments");
  USF_CHECK_ARG(!(dx && !W) && !(dW && !x && B > 0), "usf_linear_bwd: dx needs W, dW needs x");
  USF_CHECK_ARG(!(y_relu && !scratch), "usf_linear_bwd: relu backward needs scratch");
  cudaStream_t st = as_stream(stream);
  const float* g = dy;
  int64_t ldg = lddy;
  if (y_relu) {
    usf_relu_mask_kernel<<<ew_grid(B * N), 256, 0, st>>>(dy, lddy, y_relu, ldyr, scratch, B, N);
    USF_LAUNCH_CHECK("usf_relu_mask_kernel");
    g = scratch;
    ldg = N;
  }
  int rc;
  if (dx) {  // dx[b,k] = sum_n g[b,n] W[n,k]
    rc = simt_gemm_plain(g, ldg, 0, W, ldw, 1, B, K, N, dx, lddx, 0, st);
    if (rc) return rc;
  }
  if (dW) {  // dW[n,k] = sum_b g[b,n] x[b,k]
    rc = simt_gemm_plain(g, ldg, 1, x, ldx, 1, N, K, B, dW, lddw, accumulate, st);
    if (rc) return rc;
  }
  if (db) {
    rc = launch_colsum(g, ldg, db, 1.f, accumulate, B, N, st);
    if (rc) return rc;
  }
  return USF_OK;
}

extern "C" int usf_lu_pack_bwd(const float* dW, const float* L_raw, const float* U_raw, float dlogdet, int64_t D,
                               float* dL_raw, float* dU_raw, float* scratch, usf_stream_t stream) {
  USF_CHECK_ARG(L_raw && U_raw && dL_raw && dU_raw && scratch && D > 0, "usf_lu_pack_bwd: bad arguments");
  cudaStream_t st = as_stream(stream);
  float* Lm = scratch;
  float* Um = scratch + D * D;
  float* T1 = scratch + 2 * D * D;
  if (dW) {
    usf_tri_copy_kernel<<<ew_grid(D * D), 256, 0, st>>>(L_raw, Lm, D, 0);
    usf_tri_copy_kernel<<<ew_grid(D * D), 256, 0, st>>>(U_raw, Um, D, 1);
    USF_LAUNCH_CHECK("usf_tri_copy_kernel");
    // dL = strict_lower(dW U^T): [i,k] = sum_j dW[i,j] Um[k,j]
    int rc = simt_gemm_plain(dW, D, 0, Um, D, 0, D, D, D, T1, D, 0, st);
    if (rc) return rc;
    usf_tri_add_kernel<<<ew_grid(D * D), 256, 0, st>>>(T1, dL_raw, D, 0, nullptr, 0.f);
    USF_LAUNCH_CHECK("usf_tri_add_kernel");
    // dU = upper(L^T dW): [k,j] = sum_i Lm[i,k] dW[i,j]
    rc = simt_gemm_plain(Lm, D, 1, dW, D, 1, D, D, D, T1, D, 0, st);
    if (rc) return rc;
    usf_tri_add_kernel<<<ew_grid(D * D), 256, 0, st>>>(T1, dU_raw, D, 1, U_raw, dlogdet);
    USF_LAUNCH_CHECK("usf_tri_add_kernel");
  } else if (dlogdet != 0.f) {
    USF_CUDA(cudaMemsetAsync(T1, 0, sizeof(float) * D * D, st));
    usf_tri_add_kernel<<<ew_grid(D * D), 256, 0, st>>>(T1, dU_raw, D, 1, U_raw, dlogdet);
    USF_LAUNCH_CHECK("usf_tri_add_kernel");
  }
  return USF_OK;
}

extern "C" int usf_coupling_bwd(const float* dy, int64_t lddy, const float* dladj, float ladj_coef, const float* x,
                                int64_t ldx, const float* s, int64_t lds, const float* t, int64_t ldt,
                                const float* mask, float clamp, int inverse, int scale_activation, float* dx, int64_t lddx,
                                float* ds, int64_t ldds, float* dt, int64_t lddt, int64_t B, int64_t D,
                                usf_stream_t stream) {
  USF_CHECK_ARG(dy && x && t && mask && dx && dt && D > 0 && B >= 0, "usf_coupling_bwd: bad arguments");
  USF_CHECK_ARG(scale_activation == 0 || scale_activation == 1, "usf_coupling_bwd: scale_activation must be 0 or 1");
  USF_CHECK_ARG((s == nullptr) == (ds == nullptr), "usf_coupling_bwd: s and ds must both be given or both NULL");
  if (B == 0) return USF_OK;
  usf_coupling_bwd_kernel<<<ew_grid(B * D), 256, 0, as_stream(stream)>>>(
      dy, lddy, dladj, ladj_coef, x, ldx, s, lds, t, ldt, mask, clamp, inverse, scale_activation, dx, lddx, ds, ldds, dt, lddt,
      B, D);
  USF_LAUNCH_CHECK("usf_coupling_bwd_kernel");
  return USF_OK;
}

extern "C" int usf_householder_bwd(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* V,
                                   int64_t nvs, int reverse, float* dx, int64_t lddx, float* dV, float* scratch,
                                   int64_t B, int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(dy && x && dx && dV && (V || nvs == 0) && D > 0 && B >= 0, "usf_householder_bwd: bad arguments");
  USF_CHECK_ARG(nvs <= 1 || scratch, "usf_householder_bwd: scratch needed for nvs > 1");
  USF_CHECK_ARG(D * sizeof(float) <= 200 * 1024, "usf_householder_bwd: D too large");
  cudaStream_t st = as_stream(stream);
  if (B == 0) return USF_OK;
  if (nvs == 0) {
    USF_CUDA(cudaMemcpy2DAsync(dx, sizeof(float) * lddx, dy, sizeof(float) * lddy, sizeof(float) * D, B,
                               cudaMemcpyDeviceToDevice, st));
    return USF_OK;
  }
  // recompute the inputs of every reflection: xs[0] = x, xs[i+1] = reflect_i(xs[i]); scratch holds xs[1..nvs-1]
  // and one gradient ping buffer.
  const size_t smem = sizeof(float) * (size_t)D;
  if (smem > 48 * 1024)
    USF_CUDA(cudaFuncSetAttribute(usf_householder_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned rows_grid = (unsigned)ceil_div(B, ROWS_PER_CTA);
  for (int64_t i = 0; i + 1 < nvs; ++i) {
    const float* src = i == 0 ? x : scratch + (i - 1) * B * D;
    const int64_t lds_ = i == 0 ? ldx : D;
    const float* v = V + (reverse ? nvs - 1 - i : i) * D;
    usf_householder_kernel<<<rows_grid, ROWS_PER_CTA * 32, 0, st>>>(src, lds_, v, 1, 0, scratch + i * B * D, D, B, D);
    USF_LAUNCH_CHECK("usf_householder_kernel");
  }
  float* gbuf = scratch ? scratch + (nvs - 1) * B * D : nullptr;
  const float* g = dy;
  int64_t ldg = lddy;
  int nblocks = num_sms() * 2;
  if ((int64_t)nblocks * 8 > B) nblocks = (int)ceil_div(B, 8);
  for (int64_t i = nvs - 1; i >= 0; --i) {
    const float* xin = i == 0 ? x : scratch + (i - 1) * B * D;
    const int64_t ldxin = i == 0 ? ldx : D;
    const int64_t vi = reverse ? nvs - 1 - i : i;
    float* gout = (i == 0) ? dx : gbuf;
    const int64_t ldgout = (i == 0) ? lddx : D;
    // in-place on gbuf is safe: each element is read then written by the same thread
    usf_householder_bwd_kernel<<<nblocks, 256, smem, st>>>(g, ldg, xin, ldxin, V + vi * D, gout, ldgout,
                                                           dV + vi * D, B, D);
    USF_LAUNCH_CHECK("usf_householder_bwd_kernel");
    g = gout;
    ldg = ldgout;
  }
  return USF_OK;
}

extern "C" int usf_base_logprob_bwd(int kind, const float* dout, const float* z, int64_t ldz, const float* loc,
                                    const float* scale, int64_t scale_numel, float* dz, int64_t lddz, float* dloc,
                                    float* dscale, int64_t B, int64_t D, usf_stream_t stream) {
  USF_CHECK_ARG(dout && z && loc && scale && D > 0 && B >= 0, "usf_base_logprob_bwd: bad arguments");
  USF_CHECK_ARG(kind == 0 || kind == 1, "usf_base_logprob_bwd: kind must be 0 or 1");
  if (B == 0) return USF_OK;
  int gy = (int)ceil_div(B, 8 * 64);
  if (gy < 1) gy = 1;
  if (gy > 256) gy = 256;
  dim3 grid((unsigned)ceil_div(D, 32), (unsigned)gy);
  usf_base_logprob_bwd_kernel<<<grid, 256, 0, as_stream(stream)>>>(kind, dout, z, ldz, loc, scale, scale_numel, dz,
                                                                  lddz, dloc, dscale, B, D);
  USF_LAUNCH_CHECK("usf_base_logprob_bwd_kernel");
  return USF_OK;
}

extern "C" int usf_scale_bwd(const float* dy, int64_t lddy, const float* xy, int64_t ldxy, const float* scale,
                             int inverse, float* dx, int64_t lddx, float* dscale, int64_t B, int64_t D,
                             usf_stream_t stream) {
  USF_CHECK_ARG(dy && xy && scale && dx && D > 0 && B >= 0, "usf_scale_bwd: bad arguments");
  if (B == 0) return USF_OK;
  int gy = (int)ceil_div(B, 8 * 64);
  if (gy < 1) gy = 1;
  if (gy > 256) gy = 256;
  dim3 grid((unsigned)ceil_div(D, 32), (unsigned)gy);
  usf_scale_bwd_kernel<<<grid, 256, 0, as_stream(stream)>>>(dy, lddy, xy, ldxy, scale, inverse, dx, lddx, dscale, B, D);
  USF_LAUNCH_CHECK("usf_scale_bwd_kernel");
  return USF_OK;
}

extern "C" int usf_colsum(const float* a, int64_t lda, float coef, int accumulate, float* out, int64_t B, int64_t N,
                          usf_stream_t stream) {
  USF_CHECK_ARG(a && out && N > 0 && B >= 0, "usf_colsum: bad arguments");
  return launch_colsum(a, lda, out, coef, accumulate, B, N, as_stream(stream));
}

extern "C" int usf_gemm(const float* A, int64_t lda, int a_trans, const float* Bm, int64_t ldb, int b_trans,
                        float* C, int64_t ldc, int accumulate, int64_t M, int64_t N, int64_t K,
                        usf_stream_t stream) {
  USF_CHECK_ARG(A && Bm && C && M >= 0 && N >= 0 && K >= 0, "usf_gemm: bad arguments");
  return simt_gemm_plain(A, lda, a_trans, Bm, ldb, b_trans, M, N, K, C, ldc, accumulate, as_stream(stream));
}

extern "C" int usf_pack_matrix(const float* src, int64_t lds, const int32_t* row_idx, const int32_t* col_idx,
                               int sub_row0, int transpose_src, int64_t n_rows, int64_t n_cols, float* out,
                               uint16_t* out_bf16, int64_t ldo, usf_stream_t stream) {
  USF_CHECK_ARG(src && (out || out_bf16) && n_rows >= 0 && n_cols >= 0 && ldo >= n_cols, "usf_pack_matrix: bad arguments");
  if (n_rows == 0) return USF_OK;
  usf_pack_matrix_kernel<<<ew_grid(n_rows * ldo), 256, 0, as_stream(stream)>>>(
      src, lds, row_idx, col_idx, sub_row0, transpose_src, n_rows, n_cols, out, reinterpret_cast<__nv_bfloat16*>(out_bf16), ldo);
  USF_LAUNCH_CHECK("usf_pack_matrix_kernel");
  return USF_OK;
}

// ================================================================================================
// VAE-flow latent tail (nf4ad/vaeflow.py:176-179 reparameterize, :214-224 log q(z|x), :208-211 / :255-262 recon NLL):
// the element-wise steps either side of flow_prior.log_prob, one launch each, with the encoder-facing gradients.
// ================================================================================================
namespace usf {
namespace {

// one warp per row: z = mu + eps * exp(logvar / 2);  log_q[row] = sum_c (-eps^2 / 2 - logvar / 2) - L/2 log(2 pi)
// (the Normal(mu, std) log-density at z, where (z - mu) / std is eps itself)
__global__ void usf_vae_reparam_kernel(const float* __restrict__ mu, int64_t ldm, const float* __restrict__ lv, int64_t ldv,
                                       const float* __restrict__ eps, int64_t lde, float* z, int64_t ldz, float* log_q,
                                       int64_t B, int64_t L) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  for (int64_t c = lane; c < L; c += 32) {
    const float v = lv[row * ldv + c], e = eps[row * lde + c];
    z[row * ldz + c] = fmaf(e, expf(0.5f * v), mu[row * ldm + c]);
    acc += -0.5f * e * e - 0.5f * v;
  }
  acc = warp_sum(acc);
  if (lane == 0 && log_q != nullptr) log_q[row] = acc - 0.5f * (float)L * 1.8378770664093453f;
}

// dlogvar = dz * eps * exp(logvar / 2) / 2 - dlog_q[row] / 2   (dmu = dz: no kernel needed)
__global__ void usf_vae_reparam_bwd_kernel(const float* __restrict__ dz, int64_t lddz, const float* __restrict__ dlogq,
                                           const float* __restrict__ eps, int64_t lde, const float* __restrict__ lv,
                                           int64_t ldv, float* dlv, int64_t lddv, int64_t B, int64_t L) {
  const int64_t total = B * L;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / L, c = i - r * L;
    float g = 0.f;
    if (dz != nullptr) g = 0.5f * dz[r * lddz + c] * eps[r * lde + c] * expf(0.5f * lv[r * ldv + c]);
    if (dlogq != nullptr) g -= 0.5f * dlogq[r];
    dlv[r * lddv + c] = g;
  }
}

// one block per row: out[row] = sum (x - xr)^2 / (2 sigma2) + D/2 log(2 pi sigma2)
__global__ void usf_recon_nll_kernel(const float* __restrict__ x, const float* __restrict__ xr, int64_t D, float inv_2s2,
                                     float cst, float* out) {
  const int64_t row = blockIdx.x;
  const float* a = x + row * D;
  const float* b = xr + row * D;
  float acc = 0.f;
  for (int64_t c = threadIdx.x; c < D; c += blockDim.x) {
    const float d = a[c] - b[c];
    acc = fmaf(d, d, acc);
  }
  __shared__ float part[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) out[row] = fmaf(t, inv_2s2, cst);
  }
}

// dxr = -g[row] (x - xr) / sigma2 ; dx = -dxr (optional)
__global__ void usf_recon_nll_bwd_kernel(const float* __restrict__ x, const float* __restrict__ xr, const float* __restrict__ g,
                                         int64_t D, int64_t B, float inv_s2, float* dxr, float* dx) {
  const int64_t total = B * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = g[i / D] * (x[i] - xr[i]) * inv_s2;
    if (dxr != nullptr) dxr[i] = -v;
    if (dx != nullptr) dx[i] = v;
  }
}

}  // namespace
}  // namespace usf

extern "C" int usf_vae_reparam(const float* mu, int64_t ldm, const float* logvar, int64_t ldv, const float* eps, int64_t lde,
                               float* z, int64_t ldz, float* log_q, int64_t B, int64_t L, usf_stream_t stream) {
  USF_CHECK_ARG(mu && logvar && eps && z && B >= 0 && L > 0 && ldm >= L && ldv >= L && lde >= L && ldz >= L,
                "usf_vae_reparam: bad arguments");
  if (B == 0) return USF_OK;
  usf_vae_reparam_kernel<<<(unsigned)ceil_div(B, 8), 256, 0, as_stream(stream)>>>(mu, ldm, logvar, ldv, eps, lde, z, ldz, log_q,
                                                                                B, L);
  USF_LAUNCH_CHECK("usf_vae_reparam_kernel");
  return USF_OK;
}

extern "C" int usf_vae_reparam_bwd(const float* dz, int64_t lddz, const float* dlog_q, const float* eps, int64_t lde,
                                   const float* logvar, int64_t ldv, float* dlogvar, int64_t lddv, int64_t B, int64_t L,
                                   usf_stream_t stream) {
  USF_CHECK_ARG(eps && logvar && dlogvar && B >= 0 && L > 0 && lde >= L && ldv >= L && lddv >= L && (dz == nullptr || lddz >= L),
                "usf_vae_reparam_bwd: bad arguments");
  if (B == 0) return USF_OK;
  usf_vae_reparam_bwd_kernel<<<ew_grid(B * L), 256, 0, as_stream(stream)>>>(dz, lddz, dlog_q, eps, lde, logvar, ldv, dlogvar,
                                                                           lddv, B, L);
  USF_LAUNCH_CHECK("usf_vae_reparam_bwd_kernel");
  return USF_OK;
}

extern "C" int usf_recon_nll(const float* x, const float* x_recon, int64_t B, int64_t D, float sigma2, float* out,
                             usf_stream_t stream) {
  USF_CHECK_ARG(x && x_recon && out && B >= 0 && D > 0 && sigma2 > 0.f, "usf_recon_nll: bad arguments");
  if (B == 0) return USF_OK;
  const float cst = 0.5f * (float)D * logf(6.283185307179586f * sigma2);
  usf_recon_nll_kernel<<<(unsigned)B, 256, 0, as_stream(stream)>>>(x, x_recon, D, 0.5f / sigma2, cst, out);
  USF_LAUNCH_CHECK("usf_recon_nll_kernel");
  return USF_OK;
}

extern "C" int usf_recon_nll_bwd(const float* x, const float* x_recon, const float* dout, int64_t B, int64_t D, float sigma2,
                                 float* dx_recon, float* dx, usf_stream_t stream) {
  USF_CHECK_ARG(x && x_recon && dout && B >= 0 && D > 0 && sigma2 > 0.f, "usf_recon_nll_bwd: bad arguments");
  if (B == 0) return USF_OK;
  usf_recon_nll_bwd_kernel<<<ew_grid(B * D), 256, 0, as_stream(stream)>>>(x, x_recon, dout, D, B, 1.f / sigma2, dx_recon, dx);
  USF_LAUNCH_CHECK("usf_recon_nll_bwd_kernel");
  return USF_OK;
}

// ================================================================================================
// Adam step over many parameter tensors in one launch per 32 tensors (adbench_wrapper.py:369,391: torch.optim.Adam).
// Pointers travel as kernel parameters (baked into a captured graph node like every other launch of the step); the step
// count lives on the device so that the replayed graph advances it.
// ================================================================================================
namespace usf {
namespace {

constexpr int ADAM_MAX_TENSORS = 32;
constexpr int ADAM_CHUNK = 8192;      // elements per block

struct AdamBatch {
  float* p[ADAM_MAX_TENSORS];
  const float* g[ADAM_MAX_TENSORS];
  float* m[ADAM_MAX_TENSORS];
  float* v[ADAM_MAX_TENSORS];
  int64_t n[ADAM_MAX_TENSORS];
  int first_block[ADAM_MAX_TENSORS + 1];   // prefix sum of ceil(n / ADAM_CHUNK)
  int count;
};

__global__ void __launch_bounds__(256) usf_adam_kernel(const __grid_constant__ AdamBatch b, const float* __restrict__ step,
                                                       float lr, float beta1, float beta2, float eps, float wd, int decoupled,
                                                       const float* __restrict__ grad_scale) {
  int t = 0;
  while (t + 1 < b.count && (int)blockIdx.x >= b.first_block[t + 1]) ++t;
  const int64_t base = (int64_t)((int)blockIdx.x - b.first_block[t]) * ADAM_CHUNK;
  const int64_t n = b.n[t];
  const int64_t len = n - base < ADAM_CHUNK ? n - base : ADAM_CHUNK;
  float* __restrict__ p = b.p[t] + base;
  const float* __restrict__ g = b.g[t] + base;
  float* __restrict__ m = b.m[t] + base;
  float* __restrict__ v = b.v[t] + base;
  const float steps = *step;
  const float bc1 = 1.f - powf(beta1, steps), bc2 = 1.f - powf(beta2, steps);
  const float step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
  const float gs = grad_scale != nullptr ? *grad_scale : 1.f;
  auto upd = [&](float& pv, float gv, float& mv, float& vv) {
    gv *= gs;
    if (decoupled) pv *= 1.f - lr * wd; else gv = fmaf(wd, pv, gv);
    mv = fmaf(beta1, mv, (1.f - beta1) * gv);
    vv = fmaf(beta2, vv, (1.f - beta2) * gv * gv);
    pv -= step_size * mv / (sqrtf(vv) * inv_sqrt_bc2 + eps);
  };
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  if (vec) {
    const int64_t n4 = len >> 2;
    for (int64_t i = threadIdx.x; i < n4; i += blockDim.x) {
      float4 pv = reinterpret_cast<float4*>(p)[i], mv = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
      const float4 gv = __ldg(reinterpret_cast<const float4*>(g) + i);
      upd(pv.x, gv.x, mv.x, vv.x); upd(pv.y, gv.y, mv.y, vv.y); upd(pv.z, gv.z, mv.z, vv.z); upd(pv.w, gv.w, mv.w, vv.w);
      reinterpret_cast<float4*>(p)[i] = pv; reinterpret_cast<float4*>(m)[i] = mv; reinterpret_cast<float4*>(v)[i] = vv;
    }
    for (int64_t i = (n4 << 2) + threadIdx.x; i < len; i += blockDim.x) upd(p[i], g[i], m[i], v[i]);
  } else {
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) upd(p[i], g[i], m[i], v[i]);
  }
}

// SophiaG (Liu et al. 2023; `src.usflows.sophia.SophiaG`, experiments/gmm/gaussian_mixture_standart_base.yaml:45):
//   every `hess_every`-th step  h = b2 h + (1-b2) g^2      (diagonal Gauss-Newton-Bartlett estimate from the mini-batch gradient)
//   p *= 1 - lr wd;  m = b1 m + (1-b1) g;  p -= lr * sign(m) * min(|m| / (rho * bs * h + 1e-15), 1)
// same batching as the Adam kernel; `v` carries h.
__global__ void __launch_bounds__(256) usf_sophia_kernel(const __grid_constant__ AdamBatch b, const float* __restrict__ step,
                                                         float lr, float beta1, float beta2, float rho, float bs, float wd,
                                                         int hess_every, const float* __restrict__ grad_scale) {
  int t = 0;
  while (t + 1 < b.count && (int)blockIdx.x >= b.first_block[t + 1]) ++t;
  const int64_t base = (int64_t)((int)blockIdx.x - b.first_block[t]) * ADAM_CHUNK;
  const int64_t n = b.n[t];
  const int64_t len = n - base < ADAM_CHUNK ? n - base : ADAM_CHUNK;
  float* __restrict__ p = b.p[t] + base;
  const float* __restrict__ g = b.g[t] + base;
  float* __restrict__ m = b.m[t] + base;
  float* __restrict__ h = b.v[t] + base;
  const long long steps = (long long)(*step + 0.5f);                 // already incremented: 1, 2, ...
  const bool upd_h = hess_every <= 1 || ((steps - 1) % hess_every) == 0;
  const float gs = grad_scale != nullptr ? *grad_scale : 1.f;
  const float rb = rho * bs;
  for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
    const float gv = g[i] * gs;
    float hv = h[i];
    if (upd_h) { hv = fmaf(beta2, hv, (1.f - beta2) * gv * gv); h[i] = hv; }
    const float mv = fmaf(beta1, m[i], (1.f - beta1) * gv);
    m[i] = mv;
    const float ratio = fminf(fabsf(mv) / (rb * hv + 1e-15f), 1.f);
    p[i] = p[i] * (1.f - lr * wd) - lr * copysignf(ratio, mv) * (mv != 0.f ? 1.f : 0.f);
  }
}

}  // namespace
}  // namespace usf

extern "C" int usf_sophia_step(const usf_adam_tensor* tensors, int n_tensors, const float* step_dev, float lr, float beta1,
                               float beta2, float rho, float batch_size, float weight_decay, int hess_every,
                               const float* grad_scale_dev, usf_stream_t stream) {
  USF_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || tensors != nullptr) && step_dev != nullptr, "usf_sophia_step: bad arguments");
  int i = 0;
  while (i < n_tensors) {
    AdamBatch b;
    memset(&b, 0, sizeof(b));
    int blocks = 0;
    while (i < n_tensors && b.count < ADAM_MAX_TENSORS) {
      const usf_adam_tensor& t = tensors[i++];
      if (t.n <= 0) continue;
      USF_CHECK_ARG(t.p && t.g && t.m && t.v, "usf_sophia_step: null tensor pointer");
      b.p[b.count] = t.p; b.g[b.count] = t.g; b.m[b.count] = t.m; b.v[b.count] = t.v; b.n[b.count] = t.n;
      b.first_block[b.count] = blocks;
      blocks += (int)ceil_div(t.n, ADAM_CHUNK);
      ++b.count;
    }
    if (b.count == 0) continue;
    b.first_block[b.count] = blocks;
    usf_sophia_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(b, step_dev, lr, beta1, beta2, rho, batch_size,
                                                                      weight_decay, hess_every, grad_scale_dev);
    USF_LAUNCH_CHECK("usf_sophia_kernel");
  }
  return USF_OK;
}

extern "C" int usf_adam_step(const usf_adam_tensor* tensors, int n_tensors, const float* step_dev, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int decoupled, const float* grad_scale_dev,
                             usf_stream_t stream) {
  USF_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || tensors != nullptr) && step_dev != nullptr, "usf_adam_step: bad arguments");
  int i = 0;
  while (i < n_tensors) {
    AdamBatch b;
    memset(&b, 0, sizeof(b));
    int blocks = 0;
    while (i < n_tensors && b.count < ADAM_MAX_TENSORS) {
      const usf_adam_tensor& t = tensors[i++];
      if (t.n <= 0) continue;
      USF_CHECK_ARG(t.p && t.g && t.m && t.v, "usf_adam_step: null tensor pointer");
      b.p[b.count] = t.p; b.g[b.count] = t.g; b.m[b.count] = t.m; b.v[b.count] = t.v; b.n[b.count] = t.n;
      b.first_block[b.count] = blocks;
      blocks += (int)ceil_div(t.n, ADAM_CHUNK);
      ++b.count;
    }
    if (b.count == 0) continue;
    b.first_block[b.count] = blocks;
    usf_adam_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(b, step_dev, lr, beta1, beta2, eps, weight_decay, decoupled,
                                                                    grad_scale_dev);
    USF_LAUNCH_CHECK("usf_adam_kernel");
  }
  return USF_OK;
}
