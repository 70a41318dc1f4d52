// tcgen05 / TMEM / TMA bf16 GEMM with fused USFlow layer epilogues (sm_100a only).
//
//   acc[m, n] = sum_k A[m, k] * W[n, k]        A: activations (M x K, bf16), W: packed weights (N x K, bf16)
//
// Persistent, warp-specialised, 320 threads per CTA, one CTA per SM; two CTAs form a pair (cluster of 2, tcgen05
// cta_group::2) that owns a 256 x bn output tile:
//   warp 0   : TMA producer  -- cp.async.bulk.tensor (128B-swizzled boxes) into a 7-stage smem ring; each CTA of a
//                               pair stages its own 128 rows of A and HALF of the W tile; both count on the
//                               leader's mbarrier (one arrive.expect_tx for the pair's bytes)
//   warp 1   : MMA issuer    -- the leader CTA issues tcgen05.mma (M=256, N=bn<=256, K=16) into TMEM;
//                               tcgen05.commit (multicast to both CTAs) releases smem stages / publishes the accumulator
//   warps 2-9: epilogue      -- tcgen05.ld the fp32 accumulator (double-buffered in TMEM, 2 x 256 cols) and apply
//                               the layer epilogue (bias / ReLU / coupling / base density); column vectors resident
//                               in smem, coupling inputs prefetched a chunk ahead
// Warps 0 and 1 run their loops with all 32 lanes and issue from an elect.sync lane (a `lane == 0` branch makes the
// compiler wrap every UTMALDG / UTCHMMA / UTCBAR in an ELECT + R2UR.BROADCAST loop).  Programmatic dependent launch:
// griddepcontrol.launch_dependents at entry, griddepcontrol.wait after the prologue.
// Pipelines: smem full/empty mbarriers (TMA <-> MMA), TMEM full/empty mbarriers (MMA <-> epilogue).
// Every mbarrier wait is bounded (g_tc_timeout flag) so a protocol bug cannot hang the GPU.
// The same CTA-pair pipeline also runs the fused conditioner chain (usf_tc_mlp_coupling_kernel) and, with operands
// split into (hi, lo) pairs, the fp32-grade tiers (usf_tc3_gemm_kernel: 3xTF32, usf_tcb2_gemm_kernel: bf16x2).
//
// Measured bounds (profiles/r1b_*, DESIGN.md section 4): per SM the TMA unit delivers about one 128-byte box row per
// 3 cycles (232 rows per k-block here = ~700 cycles against 416 of MMA at N=208); the tensor pipe is 65-68 % active
// in the 65536 x 800 x 784 GEMM (1.23 PFLOP/s = 0.88 of the sustained cuBLAS figure measured on this pool).
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include <type_traits>

#include "usf_common.cuh"

namespace usf {

namespace {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;  // bf16 elements per k-block: 128 bytes = one swizzle row
constexpr int TC_UMMA_K = 16;
constexpr int TC_MAX_BN = 256;
constexpr int TC_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 2;      // 16 KB
constexpr uint32_t TC_BAR_BYTES = 256;
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_EPI_COLS = 1024;                    // per-column epilogue vectors resident in smem when N <= this
constexpr uint32_t TC_EPI_BYTES = 3 * TC_EPI_COLS * 4;  // bias / loc / inv_scale (N <= 1024: whole vectors, staged once;
                                                        // wider outputs: [2 stages][3][256] re-staged per tile)
// A CTA pair (cluster of 2) owns a 256 x bn tile, each CTA staging its own 128 rows of A and HALF of the W tile, which
// halves the L2->SMEM weight traffic per CTA (the measured bound of a single-CTA kernel) and the SMEM operand reads per MMA.
constexpr uint32_t TC_FIXED_BYTES = TC_BAR_BYTES + TC_EPI_BYTES + 1024;  // barriers + per-tile column vectors + alignment slack
constexpr uint32_t TC_SMEM_BYTES = 227 * 1024;                           // whole carve-out; the operand ring takes what is left
constexpr uint32_t TC_TMEM_COLS = 512;
constexpr long long TC_WAIT_LIMIT_CYCLES = 400000000LL;  // ~0.2 s

__device__ int g_tc_timeout = 0;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: returns false (and raises the global flag) if the barrier never completes.  The hot spin is
// try_wait only; the clock and the global abort flag (an L2 round trip) are looked at once per 1024 failed polls.
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return true;
  uint32_t spins = 0;
  long long t0 = 0;
  for (;;) {
    if (mbar_try_wait(bar, parity)) return true;
    if ((++spins & 1023u) == 0u) {
      if (*reinterpret_cast<volatile int*>(&g_tc_timeout) != 0) return false;
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > TC_WAIT_LIMIT_CYCLES) {
        atomicExch(&g_tc_timeout, 1);
        return false;
      }
    }
  }
}

// TMA load of a CTA pair: the load lands in this CTA's smem but signals the LEADER CTA's mbarrier (peer bit cleared).
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst_smem, const CUtensorMap* tmap, uint32_t bar, int c0, int c1) {
  uint32_t leader_bar;   // shared::cluster address of the same-offset barrier in CTA 0 of the pair
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(leader_bar) : "r"(bar), "r"(0));
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
// L2 prefetch of one box (no shared-memory destination, no barrier).
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* tmap, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the same-offset mbarrier of CTA `cta` of this cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 remote;\n\t"
      "mapa.shared::cluster.u32 remote, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remote];\n\t}"
      ::"r"(bar), "r"(cta)
      : "memory");
}

// One lane of a fully converged warp.  The producer / MMA warps run their loops with all 32 lanes (barrier waits are
// warp-wide) and issue the TMA / tcgen05 instructions from the elected lane: inside a `lane == 0` branch the compiler
// cannot prove the operands warp-uniform and wraps every UTMALDG / UTCHMMA / UTCBAR in an ELECT + R2UR.BROADCAST loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows at a 128-byte pitch, 8-row groups 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address
  d |= static_cast<uint64_t>(1) << 16;                      // leading byte offset (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // stride byte offset: 8 rows * 128 B
  d |= static_cast<uint64_t>(1) << 46;                      // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=m (128, or 256 for a CTA pair), N=n.
__device__ __forceinline__ uint32_t make_idesc(uint32_t n, uint32_t m) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit of a CTA-pair MMA: arrives on the same-offset mbarrier of BOTH CTAs
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void unpack_bf16x8(const uint4& q, float* f) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}

// 256-bit global accesses (sm_100: LDG.256 / STG.256): one LSU request per thread for a 32-byte row segment.  The
// epilogues are row-per-thread (TMEM lane = row), so every request hits a different row and the LSU request rate,
// not bytes, is their bound: halving the request count matters.  `p` must be 32-byte aligned.
__device__ __forceinline__ void ld_global_256(const void* p, uint4& lo, uint4& hi) {
  uint64_t a, b, c, d;
  asm volatile("ld.global.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
  lo = make_uint4((uint32_t)a, (uint32_t)(a >> 32), (uint32_t)b, (uint32_t)(b >> 32));
  hi = make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)d, (uint32_t)(d >> 32));
}
__device__ __forceinline__ void st_global_256(void* p, const uint4& lo, const uint4& hi) {
  const uint64_t a = (uint64_t)lo.x | ((uint64_t)lo.y << 32), b = (uint64_t)lo.z | ((uint64_t)lo.w << 32);
  const uint64_t c = (uint64_t)hi.x | ((uint64_t)hi.y << 32), d = (uint64_t)hi.z | ((uint64_t)hi.w << 32);
  asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// ---- coupling epilogue (row-per-thread: TMEM lane = row) ---------------------------------------------------------
// One 16-coordinate chunk of a masked coupling, affine or additive, either direction, in ONE branch-free form:
//   th = tanh(s + bs),  e = exp(+-clamp*th) = ex2(k1*th)   (additive: e = 1),   tt = t + bt
//   inverse (sgn = 1): y = (u - tt) * e          forward (sgn = 0): y = u * e + tt
//   both:              y = fma(u - sgn*tt, e, (1 - sgn)*tt)
// A single copy of this code serves every mode (the epilogue warps walk it in a rolled loop): with the 16-way
// unrolled per-mode variants the hot epilogue was ~32 KB of SASS and spent 40-50 % of its samples in instruction
// fetch (ncu stall_no_inst, profiles/r2).  tanh.approx / ex2.approx in fp32 (2 MUFU per coordinate; the MUFU pipe
// delivers 16 results/clk/SM).  Padded coordinates have zero weight rows and zero bias, so s = 0 and tanh(0) = 0
// adds nothing to the log-det.
// request the 16 transformed coordinates of one chunk (32 bytes, one LDG.256); partial / invalid chunks load nothing
__device__ __forceinline__ void cpl_load_u(const EpiParams& ep, int64_t row, bool rvalid, int coord0, uint4& q0, uint4& q1) {
  if (rvalid && coord0 + 16 <= ep.Db)
    ld_global_256(reinterpret_cast<const uint16_t*>(ep.ub) + row * ep.ldub + coord0, q0, q1);
}

// t_tile: TMEM address of the tile's first column for this warp's lanes; c: chunk offset inside the tile; ev: the tile's
// bias vector in smem ([bs(C) | bt(C)] or [bt(C)]).  Must be called by all 32 lanes (tcgen05.ld is warp-collective).
// Written stage by stage over all 16 coordinates (16-way ILP between the dependent FADD -> F2FP -> MUFU -> HMUL2 -> MUFU
// -> FFMA links); AFFINE / INV are compile-time so the executed path carries no selects (only one instantiation runs
// in any launch, so the instruction-cache footprint stays one chunk body).
template <bool AFFINE, bool INV>
__device__ __forceinline__ void cpl_chunk(uint32_t t_tile, int c, const float* ev, const EpiParams& ep, float k1,
                                          int64_t row, bool rvalid, int coord0, const uint4& q0, const uint4& q1, float& lsum) {
  const int C = ep.C;
  float sv[16], tv[16];
  if (AFFINE) {
    tmem_ld16(t_tile + c, sv);
    tmem_ld16(t_tile + C + c, tv);
  } else {
    tmem_ld16(t_tile + c, tv);
  }
  tmem_ld_wait();
  if (!rvalid || coord0 >= ep.Db) return;
  uint16_t* up = reinterpret_cast<uint16_t*>(ep.ub) + row * ep.ldub + coord0;
  const bool full = coord0 + 16 <= ep.Db;
  float u[16];
  if (full) {
    unpack_bf16x8(q0, u);
    unpack_bf16x8(q1, u + 8);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) u[j] = coord0 + j < ep.Db ? __uint_as_float((uint32_t)up[j] << 16) : 0.f;
  }
  const float4* bt4 = reinterpret_cast<const float4*>(AFFINE ? ev + C + c : ev + c);
#pragma unroll
  for (int j4 = 0; j4 < 4; ++j4) {
    const float4 b = bt4[j4];
    tv[4 * j4] += b.x; tv[4 * j4 + 1] += b.y; tv[4 * j4 + 2] += b.z; tv[4 * j4 + 3] += b.w;
  }
  if (AFFINE) {
    const float4* bs4 = reinterpret_cast<const float4*>(ev + c);
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
      const float4 b = bs4[j4];
      sv[4 * j4] += b.x; sv[4 * j4 + 1] += b.y; sv[4 * j4 + 2] += b.z; sv[4 * j4 + 3] += b.w;
    }
    // fp32 MUFU throughout: the packed f16x2 forms issue one MUFU.F16 per half (measured 16 results/clk/SM either
    // way, scripts/ubench/pipe_rates.cu), so they save nothing and cost 2x in log_prob error.
    float part = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) sv[j] = fast_tanh(sv[j]);
#pragma unroll
    for (int j = 0; j < 16; ++j) part += sv[j];
    lsum += part;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      float e;
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(k1 * sv[j]));
      u[j] = INV ? (u[j] - tv[j]) * e : fmaf(u[j], e, tv[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) u[j] = INV ? u[j] - tv[j] : u[j] + tv[j];
  }
  if (full) {
    uint4 o0, o1;
    o0.x = pack_bf16x2(u[0], u[1]);   o0.y = pack_bf16x2(u[2], u[3]);
    o0.z = pack_bf16x2(u[4], u[5]);   o0.w = pack_bf16x2(u[6], u[7]);
    o1.x = pack_bf16x2(u[8], u[9]);   o1.y = pack_bf16x2(u[10], u[11]);
    o1.z = pack_bf16x2(u[12], u[13]); o1.w = pack_bf16x2(u[14], u[15]);
    st_global_256(up, o0, o1);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (coord0 + j < ep.Db) up[j] = __bfloat16_as_ushort(__float2bfloat16_rn(u[j]));
  }
}

// runtime mode -> the one compile-time instantiation this launch executes
__device__ __forceinline__ void cpl_chunk_dispatch(int mode, uint32_t t_tile, int c, const float* ev, const EpiParams& ep,
                                                   float k1, int64_t row, bool rvalid, int coord0, const uint4& q0,
                                                   const uint4& q1, float& lsum) {
  if (mode == EPI_COUPLING_INV) cpl_chunk<true, true>(t_tile, c, ev, ep, k1, row, rvalid, coord0, q0, q1, lsum);
  else if (mode == EPI_COUPLING_FWD) cpl_chunk<true, false>(t_tile, c, ev, ep, k1, row, rvalid, coord0, q0, q1, lsum);
  else if (mode == EPI_ADD_INV) cpl_chunk<false, true>(t_tile, c, ev, ep, k1, row, rvalid, coord0, q0, q1, lsum);
  else cpl_chunk<false, false>(t_tile, c, ev, ep, k1, row, rvalid, coord0, q0, q1, lsum);
}

struct TcArgs {
  int64_t M, N, K;
  int bn;        // N-tile width (multiple of 16, <= 256)
  int n_tiles;   // ceil(N / bn)
  int m_tiles;   // ceil(M / 256)
  int n_valid;   // valid output columns for fp32 stores / base density (<= N)
  int reverse;                // walk the tiles from the last row tile to the first (see tc_set_tile_order)
  int stages;                 // smem ring depth (<= TC_MAX_STAGES)
  uint32_t stage_bytes;       // bytes per stage (A tile + this CTA's W rows), multiple of 1024
  EpiParams ep;
};

__global__ void __launch_bounds__(TC_THREADS, 1)
usf_tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, TcArgs args) {
  // runtime ring geometry: a stage holds 128 rows of A and bn/2 rows of W (1 KB granularity), as many stages as fit
  const int TC_STAGES = args.stages;
  const uint32_t TC_STAGE_BYTES = args.stage_bytes;
  extern __shared__ uint8_t smem_raw[];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next kernel of the chain may start its prologue
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + TC_STAGES * TC_STAGE_BYTES;
  const uint32_t cta_rank = cluster_ctarank();   // 0 = leader of the pair (issues the MMAs)
  const int unit = (int)(blockIdx.x >> 1), num_units = (int)(gridDim.x >> 1);   // persistent work unit: a CTA pair
  // barrier layout (8 bytes each): full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2]; then tmem ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (TC_STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * TC_STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * TC_STAGES + 2 + a); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * TC_STAGES + 4);
  const uint32_t epi_base = bar_base + TC_BAR_BYTES;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(full_bar(s), 1);        // the leader's arrive.expect_tx; the peer's loads only add transaction bytes
      mbar_init(empty_bar(s), 1);       // one tcgen05.commit (multicast to both CTAs of the pair)
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 16);     // 8 epilogue warps per CTA, all arriving on the leader's barrier
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();   // the peer's barriers must be initialised before any remote arrive / TMA signal
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_addr) : "memory");
  // Programmatic dependent launch: this grid may have been started while the previous kernel of the chain was still
  // draining (its CTAs that ran out of tiles free their SMs early); everything above -- barrier init, TMEM
  // allocation, tensor-map prefetch, cluster sync -- touched no data of that kernel.  From here on we read and write
  // the activation buffers, so wait for it to complete (a no-op when the launch carried no such dependency).
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const int total_tiles = args.m_tiles * args.n_tiles;
  const int num_kb = (int)((args.K + TC_BK - 1) / TC_BK);
  // bytes landing per stage on the leader's full barrier: each CTA of the pair loads 128 rows of A and bn/2 rows of W
  const uint32_t stage_tx = 2u * (TC_A_BYTES + (uint32_t)(args.bn / 2) * TC_BK * 2);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (whole warp, one elected lane issues)
    {
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int t = unit; t < total_tiles && ok; t += num_units) {
        const int tt = args.reverse ? total_tiles - 1 - t : t;
        const int mt = tt / args.n_tiles, nt = tt - mt * args.n_tiles;
        int width = (int)(args.N - (int64_t)nt * args.bn);
        if (width > args.bn) width = args.bn;
        // the pair splits the tile's N columns evenly: CTA r stages W rows [n0 + r*width/2, +width/2)
        const int w_row = nt * args.bn + (int)cta_rank * (width >> 1);
        const int a_row = (mt * 2 + (int)cta_rank) * TC_BM;
        for (int kb = 0; kb < num_kb; ++kb) {
          ok = mbar_wait(empty_bar(s), ph ^ 1u);
          if (!ok) break;
          const uint32_t a_dst = smem_base + s * TC_STAGE_BYTES;
          if (elect_one()) {
            // The peer's bytes can only land in the leader's CURRENT phase: its empty barrier for this slot was
            // released by the commit that followed the MMAs which consumed the slot's previous contents.
            if (cta_rank == 0) mbar_expect_tx(full_bar(s), stage_tx);
            tma_load_2d_2sm(a_dst, &tmA, full_bar(s), kb * TC_BK, a_row);
            tma_load_2d_2sm(a_dst + TC_A_BYTES, &tmW, full_bar(s), kb * TC_BK, w_row);
          }
          if (++s == TC_STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA; whole warp, one elected lane issues)
    if (cta_rank == 0) {
      int s = 0, a = 0;
      uint32_t ph = 0, aph = 0;
      bool ok = true;
      // K=16 steps of the last k-block (earlier k-blocks always run all four)
      const int tail_steps = ((int)args.K - (num_kb - 1) * TC_BK + TC_UMMA_K - 1) / TC_UMMA_K;
      // operand descriptors: only the 14-bit start-address field changes from stage to stage
      const uint64_t desc_hi = make_smem_desc(0);
      const uint32_t desc_lo0 = (smem_base & 0x3FFFFu) >> 4, desc_stage = TC_STAGE_BYTES >> 4;
      for (int t = unit; t < total_tiles && ok; t += num_units) {
        const int nt = (args.reverse ? total_tiles - 1 - t : t) % args.n_tiles;
        int width = (int)(args.N - (int64_t)nt * args.bn);
        if (width > args.bn) width = args.bn;
        const uint32_t idesc = make_idesc((uint32_t)width, 2 * TC_BM);
        ok = mbar_wait(tempty_bar(a), aph ^ 1u);
        if (!ok) break;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)a * TC_MAX_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          // TMA (async proxy) -> mbarrier -> tcgen05.mma needs no further fence
          ok = mbar_wait(full_bar(s), ph);
          if (!ok) break;
          if (elect_one()) {
            // descriptors advance by 32 bytes (2 x 16-byte units) per K=16 step inside the 128-byte swizzle row
            const uint64_t ad0 = desc_hi | (uint64_t)(desc_lo0 + (uint32_t)s * desc_stage);
            const uint64_t bd0 = ad0 + (TC_A_BYTES >> 4);
            if (kb + 1 < num_kb) {
#pragma unroll
              for (int k = 0; k < TC_BK / TC_UMMA_K; ++k)
                umma_bf16_2sm(d_tmem, ad0 + 2u * k, bd0 + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            } else {
              for (int k = 0; k < tail_steps; ++k)
                umma_bf16_2sm(d_tmem, ad0 + 2u * k, bd0 + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_2sm(empty_bar(s));   // smem stage reusable in both CTAs once these MMAs retire
          }
          if (++s == TC_STAGES) { s = 0; ph ^= 1u; }
        }
        if (!ok) break;
        // accumulator ready for the epilogue (each CTA of the pair holds its own 128 rows in its TMEM)
        if (elect_one()) umma_commit_2sm(tfull_bar(a));
        a ^= 1;
        if (a == 0) aph ^= 1u;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (2..9)
    // Two warps per TMEM lane group (32 rows): `half` 0/1 takes the even/odd 16-column chunks.
    const int lane_grp = warp & 3;  // TMEM lanes [32*lane_grp, +32) are accessible to this warp
    const int half = (warp - 2) >> 2;
    const int et = (int)threadIdx.x - 64;  // 0..255 within the epilogue group
    const EpiParams& ep = args.ep;
    float* epi = reinterpret_cast<float*>(smem_raw + (epi_base - smem_u32(smem_raw)));  // [2][3][256]
    const bool is_cpl = ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD;
    const bool is_add = ep.mode == EPI_ADD_INV || ep.mode == EPI_ADD_FWD;
    const bool is_base = ep.mode == EPI_BASE_NORMAL || ep.mode == EPI_BASE_LAPLACE;
    const float k1 = (ep.mode == EPI_COUPLING_INV ? -ep.clamp : ep.clamp) * 1.4426950408889634f;   // +-clamp * log2(e)
    // per-column vectors: staged once for the whole kernel when they fit, else re-staged per tile
    const bool resident = args.N <= TC_EPI_COLS;
    if (resident) {
      for (int i = et; i < (int)args.N; i += 256) {
        epi[i] = ep.bias != nullptr ? ep.bias[i] : 0.f;
        if (is_base) {
          const bool v2 = i < args.n_valid && ep.loc != nullptr;
          epi[TC_EPI_COLS + i] = v2 ? ep.loc[i] : 0.f;
          epi[2 * TC_EPI_COLS + i] = v2 ? ep.inv_scale[i] : 0.f;
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    int a = 0;
    uint32_t aph = 0;
    for (int t = unit; t < total_tiles; t += num_units) {
      const int tt = args.reverse ? total_tiles - 1 - t : t;
      const int mt = tt / args.n_tiles, nt = tt - mt * args.n_tiles;
      const int64_t row = (int64_t)(mt * 2 + (int)cta_rank) * TC_BM + lane_grp * 32 + lane;
      const bool rvalid = row < args.M;
      const int64_t n0 = (int64_t)nt * args.bn;
      int width = (int)(args.N - n0);
      if (width > args.bn) width = args.bn;
      // bias / loc / inv_scale of this tile's columns
      float* ev = resident ? epi + n0 : epi + a * 768;
      const float* ev_loc = resident ? ev + TC_EPI_COLS : ev + 256;
      const float* ev_isc = resident ? ev + 2 * TC_EPI_COLS : ev + 512;

      // (1) not resident: stage the per-column vectors of this tile in shared memory (one element per epilogue thread)
      if (!resident) {
        const int64_t col = n0 + et;
        const bool cv = et < width;
        ev[et] = (cv && ep.bias != nullptr) ? ep.bias[col] : 0.f;
        if (is_base) {
          const bool v2 = cv && col < args.n_valid && ep.loc != nullptr;
          ev[256 + et] = v2 ? ep.loc[col] : 0.f;
          ev[512 + et] = v2 ? ep.inv_scale[col] : 0.f;
        }
      }
      // (2) coupling: request the first chunk of transformed coordinates of this thread's row (independent of the MMA)
      uint4 cq0 = make_uint4(0, 0, 0, 0), cq1 = cq0;
      if (is_cpl || is_add) cpl_load_u(ep, row, rvalid, nt * ep.C + half * 16, cq0, cq1);
      if (!resident) asm volatile("bar.sync 1, 256;" ::: "memory");

      if (mbar_wait(tfull_bar(a), aph)) {
        tc_fence_after();
        const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)a * TC_MAX_BN;

        if ((ep.mode == EPI_BIAS || ep.mode == EPI_BIAS_RELU) && ep.out_bf16) {
          for (int c = half * 16; c < width; c += 32) {
            float v[16];
            tmem_ld16(t_base + c, v);
            tmem_ld_wait();
            if (rvalid) {
              const float4* bv = reinterpret_cast<const float4*>(ev + c);
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b4 = bv[j4];
                v[4 * j4] += b4.x; v[4 * j4 + 1] += b4.y; v[4 * j4 + 2] += b4.z; v[4 * j4 + 3] += b4.w;
              }
              if (ep.mode == EPI_BIAS_RELU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
              }
              uint4 q0, q1;
              q0.x = pack_bf16x2(v[0], v[1]);   q0.y = pack_bf16x2(v[2], v[3]);
              q0.z = pack_bf16x2(v[4], v[5]);   q0.w = pack_bf16x2(v[6], v[7]);
              q1.x = pack_bf16x2(v[8], v[9]);   q1.y = pack_bf16x2(v[10], v[11]);
              q1.z = pack_bf16x2(v[12], v[13]); q1.w = pack_bf16x2(v[14], v[15]);
              st_global_256(reinterpret_cast<uint16_t*>(ep.out) + row * ep.ldo + n0 + c, q0, q1);
            }
          }
        } else if (ep.mode == EPI_BIAS || ep.mode == EPI_BIAS_RELU) {   // fp32 output
          for (int c = half * 16; c < width; c += 32) {
            float v[16];
            tmem_ld16(t_base + c, v);
            tmem_ld_wait();
            if (rvalid) {
              const float4* bv = reinterpret_cast<const float4*>(ev + c);
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b4 = bv[j4];
                v[4 * j4] += b4.x; v[4 * j4 + 1] += b4.y; v[4 * j4 + 2] += b4.z; v[4 * j4 + 3] += b4.w;
              }
              if (ep.mode == EPI_BIAS_RELU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
              }
              float* dst = reinterpret_cast<float*>(ep.out) + row * ep.ldo + n0 + c;
              if (n0 + c + 16 <= args.n_valid && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                // full, 16-byte aligned chunk (the training GEMMs: fp32 gradients / activations): 4 x 128-bit stores
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4)
                  reinterpret_cast<float4*>(dst)[j4] = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (n0 + c + j < args.n_valid) dst[j] = v[j];
              }
            }
          }
        } else if (is_cpl || is_add) {
          // rolled chunk loop (one copy of the chunk code); the next chunk's coordinates are requested before the
          // current chunk is processed
          float lsum = 0.f;
          for (int c = half * 16; c < ep.C; c += 32) {
            uint4 nq0 = make_uint4(0, 0, 0, 0), nq1 = nq0;
            if (c + 32 < ep.C) cpl_load_u(ep, row, rvalid, nt * ep.C + c + 32, nq0, nq1);
            cpl_chunk_dispatch(ep.mode, t_base, c, ev, ep, k1, row, rvalid, nt * ep.C + c, cq0, cq1, lsum);
            cq0 = nq0;
            cq1 = nq1;
          }
          if (is_cpl && rvalid && ep.row_acc != nullptr)
            row_accumulate(ep, row, nt * 2 + half, (ep.mode == EPI_COUPLING_INV ? -ep.clamp : ep.clamp) * lsum);
        } else {  // EPI_BASE_NORMAL / EPI_BASE_LAPLACE  (padded columns have inv_scale = 0 -> contribute 0)
          float lsum = 0.f;
          for (int c = half * 16; c < width; c += 32) {
            float v[16];
            tmem_ld16(t_base + c, v);
            tmem_ld_wait();
            if (rvalid) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float z = v[j] + ev[c + j];
                if (ep.out != nullptr && n0 + c + j < args.n_valid)
                  reinterpret_cast<float*>(ep.out)[row * ep.ldo + n0 + c + j] = z;
                const float d = (z - ev_loc[c + j]) * ev_isc[c + j];
                lsum += (ep.mode == EPI_BASE_NORMAL) ? -0.5f * d * d : -fabsf(d);
              }
            }
          }
          if (rvalid && ep.row_acc != nullptr && ep.loc != nullptr) row_accumulate(ep, row, nt * 2 + half, lsum);
        }

        // accumulator drained: hand the TMEM buffer back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (cta_rank == 0) mbar_arrive(tempty_bar(a));
          else mbar_arrive_cluster(tempty_bar(a), 0);
        }
      }
      a ^= 1;
      if (a == 0) aph ^= 1u;
    }
  }

  tc_fence_before();
  cluster_sync_all();   // the peer may still be reading this CTA's smem / arriving on its barriers
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

// ================================================================================================
// Fused conditioner chain + coupling (CTA pairs, cta_group::2):   per 256-row tile, ONE kernel runs
//   h_1 = relu(u_a W_1^T + b_1), ..., h_{L-1} = relu(h_{L-2} W_{L-1}^T + b_{L-1}),  (s|t) = h_{L-1} W_L^T + b_L,
// followed by the coupling update of the transformed columns and the per-row log-det.  Hidden activations never
// leave the SM: each hidden epilogue writes its bf16 tile straight into shared memory in the K-major / 128B-swizzled
// layout the next layer's tcgen05.mma reads as operand A (in place: layer l+1's output overwrites layer l's, which is
// safe because its epilogue only starts after every MMA that read the old contents has completed).  Weights stream
// from L2 through the same TMA ring as the plain GEMM (each CTA stages half of every W tile); only layer 1 also
// streams A (the conditioning columns of the activation).  Replaces L launches + 2(L-1) HBM round trips of h.
// ================================================================================================
constexpr int MLP_MAX_LAYERS = 4;
// Epilogue warps of the fused kernel: 16 (four per scheduler).  Its epilogues alternate between TMEM reads
// (~75 B/clk/SM measured), MUFU-heavy and FMA-heavy stretches; with two warps per scheduler those phases barely
// overlapped (issue slots 29 % busy, ncu profiles/r2).  Warp w owns TMEM lanes 32*(w%4)..+32 and every
// MLP_EPI_PARTS-th 16-column chunk.
constexpr int MLP_EPI_WARPS = 16;
constexpr int MLP_EPI_PARTS = MLP_EPI_WARPS / 4;
constexpr int MLP_EPI_THREADS = MLP_EPI_WARPS * 32;
constexpr int MLP_THREADS = 64 + MLP_EPI_THREADS;   // warp 0 TMA, warp 1 MMA, warps 2.. epilogue
// Operand ring: 9 slots of 16 KB, ONE TMA box per slot (128 activation rows, or this CTA's <= 128 weight rows, of one
// 64-wide k-block).  Layers >= 2 stream only weights, so with [A|W] stage pairs half of the ring sat empty and only 4
// k-blocks were in flight -- at the measured 2-3.5k-cycle loaded TMA latency that, not the MMA rate, set the pace of
// the second and third layer (profiles/r2).  Layer 1 takes two slots per k-block, the others one.
constexpr int MLP_SLOTS = 9;
constexpr uint32_t MLP_SLOT_BYTES = TC_A_BYTES;
constexpr int MLP_H_KB = 4;                                   // k-blocks of the hidden tile
constexpr uint32_t MLP_H_BYTES = MLP_H_KB * TC_A_BYTES;       // 128 rows x 256 cols bf16 = 4 k-blocks of 16 KB
constexpr uint32_t MLP_SMEM_BYTES = MLP_SLOTS * MLP_SLOT_BYTES + MLP_H_BYTES + TC_BAR_BYTES + TC_EPI_BYTES + 1024;

struct MlpMaps {
  CUtensorMap w[MLP_MAX_LAYERS];
};

struct MlpArgs {
  int64_t M;
  int m_tiles;                   // 256-row pair tiles
  int L;                         // layers: L-1 hidden + the coupling layer
  int K[MLP_MAX_LAYERS];         // valid K of layer l
  int N[MLP_MAX_LAYERS];         // packed N of layer l (multiple of 16)
  int bn[MLP_MAX_LAYERS];        // N-tile width of layer l (hidden: = N <= 256)
  int ntile[MLP_MAX_LAYERS];
  int boff[MLP_MAX_LAYERS];      // offset of layer l's bias vector in the resident smem copy (prefix sums of N)
  const float* bias[MLP_MAX_LAYERS];
  EpiParams ep;                  // coupling epilogue of the last layer
  int reverse;                   // walk the row tiles from the last to the first (see tc_set_tile_order)
};

__global__ void __launch_bounds__(MLP_THREADS, 1)
usf_tc_mlp_coupling_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ MlpMaps maps, MlpArgs args) {
  extern __shared__ uint8_t smem_raw[];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next kernel of the chain may start its prologue
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t h_base = smem_base + MLP_SLOTS * MLP_SLOT_BYTES;   // hidden activation tile (operand A of layers >= 2)
  const uint32_t bar_base = h_base + MLP_H_BYTES;
  const uint32_t cta_rank = cluster_ctarank();
  const int unit = (int)(blockIdx.x >> 1), num_units = (int)(gridDim.x >> 1);
  // barriers (8 bytes each): full[SLOTS], empty[SLOTS], tmem_full[2], tmem_empty[2], hready[H_KB]; then the tmem pointer
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MLP_SLOTS + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * MLP_SLOTS + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * MLP_SLOTS + 2 + a); };
  auto hready_bar = [&](int kb) { return bar_base + 8u * (2 * MLP_SLOTS + 4 + kb); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * MLP_SLOTS + 4 + MLP_H_KB);
  const uint32_t epi_base = bar_base + TC_BAR_BYTES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < MLP_SLOTS; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * MLP_EPI_WARPS);
    }
    // one per 64-column k-block of the hidden tile: the next layer's MMAs over k-block i start as soon as every
    // epilogue warp of both CTAs has written its columns of that k-block
    for (int kb = 0; kb < MLP_H_KB; ++kb) mbar_init(hready_bar(kb), 2 * MLP_EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    for (int l = 0; l < args.L; ++l)
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&maps.w[l])) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_addr) : "memory");
  // Programmatic dependent launch: this grid may have been started while the previous kernel of the chain was still
  // draining (its CTAs that ran out of tiles free their SMs early); everything above -- barrier init, TMEM
  // allocation, tensor-map prefetch, cluster sync -- touched no data of that kernel.  From here on we read and write
  // the activation buffers, so wait for it to complete (a no-op when the launch carried no such dependency).
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int L = args.L;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs; whole warp, elected lane issues)
    {
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      // one box into the next free slot; the pair's bytes are accounted on the leader's barrier
      auto load = [&](const CUtensorMap* tm, uint32_t bytes_per_cta, int c0, int c1) {
        ok = mbar_wait(empty_bar(s), ph ^ 1u);
        if (!ok) return;
        if (elect_one()) {
          if (cta_rank == 0) mbar_expect_tx(full_bar(s), 2u * bytes_per_cta);
          tma_load_2d_2sm(smem_base + s * MLP_SLOT_BYTES, tm, full_bar(s), c0, c1);
        }
        if (++s == MLP_SLOTS) { s = 0; ph ^= 1u; }
      };
      const int nkb0 = (args.K[0] + TC_BK - 1) / TC_BK;
      for (int t = unit; t < args.m_tiles && ok; t += num_units) {
        const int rt = args.reverse ? args.m_tiles - 1 - t : t;       // row tile
        const int a_row = (rt * 2 + (int)cta_rank) * TC_BM;
        // All CTAs run their first layer at about the same time, and its activation rows come from HBM: that phase
        // was HBM-bound (~5.4 TB/s) while HBM idled through the rest of the row tile.  The NEXT row tile's rows are
        // therefore requested into L2 while this tile's last layer streams its (L2-resident) weights.
        int pf_kb = 0;
        const int pf_row = t + num_units < args.m_tiles
                               ? ((args.reverse ? args.m_tiles - 1 - (t + num_units) : t + num_units) * 2 + (int)cta_rank) * TC_BM
                               : -1;
        for (int l = 0; l < L && ok; ++l) {
          const int nkb = (args.K[l] + TC_BK - 1) / TC_BK;
          const uint32_t w_bytes = (uint32_t)(args.bn[l] >> 1) * TC_BK * 2;
          for (int nt = 0; nt < args.ntile[l] && ok; ++nt) {
            int width = args.N[l] - nt * args.bn[l];
            if (width > args.bn[l]) width = args.bn[l];
            const int w_row = nt * args.bn[l] + (int)cta_rank * (width >> 1);
            for (int kb = 0; kb < nkb && ok; ++kb) {
              if (l == 0) load(&tmA, TC_A_BYTES, kb * TC_BK, a_row);
              if (ok) load(&maps.w[l], w_bytes, kb * TC_BK, w_row);
              if (l == L - 1 && pf_row >= 0 && pf_kb < nkb0) {
                if (elect_one()) tma_prefetch_2d(&tmA, pf_kb * TC_BK, pf_row);
                ++pf_kb;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only; whole warp, elected lane issues)
    if (cta_rank == 0) {
      int s = 0, a = 0;
      uint32_t ph = 0, aph = 0, hph = 0;
      bool ok = true;
      const uint64_t desc_hi = make_smem_desc(0);
      const uint32_t slot_lo0 = (smem_base & 0x3FFFFu) >> 4, h_lo0 = (h_base & 0x3FFFFu) >> 4;
      for (int t = unit; t < args.m_tiles && ok; t += num_units) {
        for (int l = 0; l < L && ok; ++l) {
          const int nkb = (args.K[l] + TC_BK - 1) / TC_BK;
          for (int nt = 0; nt < args.ntile[l] && ok; ++nt) {
            int width = args.N[l] - nt * args.bn[l];
            if (width > args.bn[l]) width = args.bn[l];
            const uint32_t idesc = make_idesc((uint32_t)width, TC_BM * 2);
            ok = mbar_wait(tempty_bar(a), aph ^ 1u);
            if (!ok) break;
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)a * TC_MAX_BN;
            for (int kb = 0; kb < nkb; ++kb) {
              uint32_t a_lo;
              int sa = -1;
              if (l == 0) {                 // operand A streams through the ring (its own slot)
                ok = mbar_wait(full_bar(s), ph);
                if (!ok) break;
                sa = s;
                a_lo = slot_lo0 + (uint32_t)s * (MLP_SLOT_BYTES >> 4);
                if (++s == MLP_SLOTS) { s = 0; ph ^= 1u; }
              } else {                      // operand A = k-block kb of the hidden tile (written by the previous epilogue)
                if (nt == 0) {
                  ok = mbar_wait(hready_bar(kb), hph);
                  if (!ok) break;
                  tc_fence_after();
                }
                a_lo = h_lo0 + (uint32_t)kb * (TC_A_BYTES >> 4);
              }
              ok = mbar_wait(full_bar(s), ph);
              if (!ok) break;
              int krem = args.K[l] - kb * TC_BK;
              if (krem > TC_BK) krem = TC_BK;
              const int ksteps = (krem + TC_UMMA_K - 1) / TC_UMMA_K;
              if (elect_one()) {
                const uint64_t ad0 = desc_hi | (uint64_t)a_lo;
                const uint64_t bd0 = desc_hi | (uint64_t)(slot_lo0 + (uint32_t)s * (MLP_SLOT_BYTES >> 4));
                if (ksteps == TC_BK / TC_UMMA_K) {
#pragma unroll
                  for (int k = 0; k < TC_BK / TC_UMMA_K; ++k)
                    umma_bf16_2sm(d_tmem, ad0 + 2u * k, bd0 + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
                } else {
                  for (int k = 0; k < ksteps; ++k)
                    umma_bf16_2sm(d_tmem, ad0 + 2u * k, bd0 + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
                }
                if (sa >= 0) umma_commit_2sm(empty_bar(sa));
                umma_commit_2sm(empty_bar(s));
              }
              if (++s == MLP_SLOTS) { s = 0; ph ^= 1u; }
            }
            if (!ok) break;
            if (elect_one()) umma_commit_2sm(tfull_bar(a));
            a ^= 1;
            if (a == 0) aph ^= 1u;
          }
          if (l > 0) hph ^= 1u;   // every hready barrier completed exactly once for this layer
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (2..), both CTAs
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;   // which of the MLP_EPI_PARTS column interleaves this warp takes
    const int et = (int)threadIdx.x - 64;
    const EpiParams& ep = args.ep;
    float* epi = reinterpret_cast<float*>(smem_raw + (epi_base - smem_u32(smem_raw)));
    uint4* hp = reinterpret_cast<uint4*>(smem_raw + (h_base - smem_u32(smem_raw)));   // H as uint4[kb][128 rows][8 pieces]
    const bool is_cpl = ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD;   // else: additive
    const int rloc = lane_grp * 32 + lane;           // row within this CTA's 128-row tile
    const float k1 = (ep.mode == EPI_COUPLING_INV ? -ep.clamp : ep.clamp) * 1.4426950408889634f;   // +-clamp * log2(e)
    // every layer's bias vector stays in shared memory for the whole kernel (sum of N <= 3 * TC_EPI_COLS, host-checked)
    for (int l = 0; l < L; ++l)
      for (int i = et; i < args.N[l]; i += MLP_EPI_THREADS) epi[args.boff[l] + i] = args.bias[l][i];
    asm volatile("bar.sync 1, %0;" ::"n"(MLP_EPI_THREADS) : "memory");
    int a = 0;
    uint32_t aph = 0;
    const int ntl = args.ntile[L - 1];
    for (int t = unit; t < args.m_tiles; t += num_units) {
      const int64_t row = (int64_t)((args.reverse ? args.m_tiles - 1 - t : t) * 2 + (int)cta_rank) * TC_BM + rloc;
      const bool rvalid = row < args.M;
      // accumulator hand-over: wait until the MMAs of the next GEMM of the chain are complete / give the buffer back
      auto acquire = [&]() -> bool {
        const bool ok = mbar_wait(tfull_bar(a), aph);
        if (ok) tc_fence_after();
        return ok;
      };
      auto release = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (cta_rank == 0) mbar_arrive(tempty_bar(a));
          else mbar_arrive_cluster(tempty_bar(a), 0);
        }
      };
      auto advance = [&]() {
        a ^= 1;
        if (a == 0) aph ^= 1u;
      };
      // the first coupling chunk's coordinates travel while the hidden layers run
      uint4 cq0 = make_uint4(0, 0, 0, 0), cq1 = cq0;
      cpl_load_u(ep, row, rvalid, half * 16, cq0, cq1);

      // ---- hidden layers: bias + ReLU -> bf16 -> operand-A layout of the next layer (in place in shared memory)
      for (int l = 0; l + 1 < L; ++l) {
        const int width = args.N[l];
        const float* ev = epi + args.boff[l];
        if (acquire()) {
          const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)a * TC_MAX_BN;
          // chunk i of this warp = columns [16*part + 64*i, +16): one 16-byte-pair piece of k-block i of the next
          // layer's operand A.  After each chunk the warp publishes its part of that k-block (hready[i]), so the MMA
          // warp can start the next layer on k-block 0 while the later k-blocks are still being converted.
          const int nkb_h = (width + TC_BK - 1) / TC_BK;
          for (int i = 0; i < nkb_h; ++i) {
            const int c = half * 16 + i * TC_BK;
            if (c < width) {   // warp-uniform
              float v[16];
              tmem_ld16(t_base + c, v);
              tmem_ld_wait();
              const float4* bv = reinterpret_cast<const float4*>(ev + c);
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b4 = bv[j4];
                v[4 * j4] = fmaxf(v[4 * j4] + b4.x, 0.f);
                v[4 * j4 + 1] = fmaxf(v[4 * j4 + 1] + b4.y, 0.f);
                v[4 * j4 + 2] = fmaxf(v[4 * j4 + 2] + b4.z, 0.f);
                v[4 * j4 + 3] = fmaxf(v[4 * j4 + 3] + b4.w, 0.f);
              }
              uint4 q0, q1;
              q0.x = pack_bf16x2(v[0], v[1]);   q0.y = pack_bf16x2(v[2], v[3]);
              q0.z = pack_bf16x2(v[4], v[5]);   q0.w = pack_bf16x2(v[6], v[7]);
              q1.x = pack_bf16x2(v[8], v[9]);   q1.y = pack_bf16x2(v[10], v[11]);
              q1.z = pack_bf16x2(v[12], v[13]); q1.w = pack_bf16x2(v[14], v[15]);
              const int p = (c & 63) >> 3;    // 16-byte piece within the 128-byte row of k-block i
              uint4* rowp = hp + (size_t)i * (TC_A_BYTES / 16) + rloc * 8;
              rowp[p ^ (rloc & 7)] = q0;
              rowp[(p + 1) ^ (rloc & 7)] = q1;
              asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to tcgen05.mma
            }
            __syncwarp();
            if (lane == 0) {
              if (cta_rank == 0) mbar_arrive(hready_bar(i));
              else mbar_arrive_cluster(hready_bar(i), 0);
            }
          }
          // k-blocks this layer does not have complete too (their phase must flip once per layer)
          if (lane == 0) {
            for (int i = nkb_h; i < MLP_H_KB; ++i) {
              if (cta_rank == 0) mbar_arrive(hready_bar(i));
              else mbar_arrive_cluster(hready_bar(i), 0);
            }
          }
          release();
        }
        advance();
      }

      // ---- last layer: coupling update of the transformed columns.  This warp walks its chunks of every [s|t] (or
      //      [t]) tile in ONE rolled loop; the coordinates of the next chunk (possibly of the next tile) are requested
      //      before the current chunk is processed, so their latency hides behind ~one chunk of work.
      const float* evl = epi + args.boff[L - 1];
      const int C = ep.C, bnl = args.bn[L - 1];
      float lsum = 0.f;
      if (half * 16 >= C) {
        // no chunk of any tile belongs to this warp (narrow tiles): only hand the accumulators back
        for (int nt = 0; nt < ntl; ++nt) {
          if (acquire()) release();
          advance();
        }
      } else {
        int nt = 0, c = half * 16;
        bool ok = true;
        uint32_t t_tile = 0;
        while (nt < ntl) {
          int nc = c + 16 * MLP_EPI_PARTS, nnt = nt;
          if (nc >= C) { nc = half * 16; nnt = nt + 1; }
          uint4 nq0 = make_uint4(0, 0, 0, 0), nq1 = nq0;
          if (nnt < ntl) cpl_load_u(ep, row, rvalid, nnt * C + nc, nq0, nq1);
          if (c == half * 16) {   // first chunk of the tile
            ok = acquire();
            t_tile = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)a * TC_MAX_BN;
          }
          if (ok) cpl_chunk_dispatch(ep.mode, t_tile, c, evl + nt * bnl, ep, k1, row, rvalid, nt * C + c, cq0, cq1, lsum);
          if (nnt != nt) {        // last chunk of the tile
            if (ok) release();
            advance();
          }
          cq0 = nq0;
          cq1 = nq1;
          c = nc;
          nt = nnt;
        }
      }
      if (is_cpl && rvalid && ep.row_acc != nullptr)     // `half` = this warp's part (0 .. MLP_EPI_PARTS - 1)
        row_accumulate(ep, row, half, (ep.mode == EPI_COUPLING_INV ? -ep.clamp : ep.clamp) * lsum);
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}


// ================================================================================================
// Split-operand GEMMs: fp32-grade accuracy on the tensor cores.  Every operand is a pair hi + lo and each MMA step
// issues three MMAs into the same fp32 TMEM accumulator:
//     a w ~= a_hi w_hi + a_hi w_lo + a_lo w_hi
// Same CTA-pair pipeline as usf_tc_gemm_kernel; a stage holds [A_hi | A_lo | W_hi | W_lo] of one k-block (128-byte
// rows).  Epilogues write their results as (hi, lo) pairs again, the next GEMM's operands.  Two operand formats:
//   3xTF32 (usf_tc3_gemm_kernel, the <= 1e-4 tier without the FFMA pipe): fp32 hi = the value the tensor core sees
//     when it reads fp32 as tf32 (it drops the low 13 mantissa bits), lo = a - hi (exact in fp32, precomputed by the
//     producing kernel / at weight-pack time).  k-blocks of 32 columns, kind::tf32 MMAs of K=8; the dropped
//     a_lo w_lo term is ~2^-21 relative.
//   bf16x2 (usf_tcb2_gemm_kernel: the bf16 rate / 3, twice the 3xTF32 rate at half its operand bytes): hi = bf16(v),
//     lo = bf16(v - hi), 16 mantissa bits together.  k-blocks of 64 columns, kind::f16 MMAs of K=16; the dropped term
//     is ~2^-16 relative.
// ================================================================================================
template <class T>
struct SplitArgs {
  int64_t M, N, K;
  int bn, n_tiles, m_tiles, n_valid, stages;
  uint32_t stage_bytes, w_bytes;   // w_bytes: this CTA's W rows of one k-block, rounded up to 1 KB
  EpiParams ep;
  T* out_lo;    // EPI_BIAS*: low part of the output (same leading dimension as ep.out); NULL: plain fp32 output
  T* ub_lo;     // coupling modes: low part of the transformed columns (same leading dimension as ep.ub)
};

__device__ __forceinline__ void umma_tf32_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::tf32 instruction descriptor: D=f32, A=B=tf32 (format 2), both K-major
__device__ __forceinline__ uint32_t make_idesc_tf32(uint32_t n, uint32_t m) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// hi = v rounded to nearest tf32 (low 13 mantissa bits zero, so the tensor core's truncating read is exact);
// lo = v - hi is exact in fp32 and at most 2^-12 |v|
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u); }

// tanh / exp for the fp32-grade tiers from two MUFU ops each instead of the ~25-instruction libm paths:
//   tanh(x) = 1 - 2 / (exp(2x) + 1)   (ex2.approx: 2^-22 relative; absolute error of the result ~1e-7, which is what
//   the log-det sum sees; saturates correctly for |x| large: ex2 -> inf or 0)
__device__ __forceinline__ float ex2_fast(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}
__device__ __forceinline__ float tanh_mufu(float x) { return 1.f - __fdividef(2.f, ex2_fast(x * 2.8853900817779268f) + 1.f); }

__device__ __forceinline__ void st16_f32(float* dst, const float (&v)[16]) {
#pragma unroll
  for (int j4 = 0; j4 < 4; ++j4)
    reinterpret_cast<float4*>(dst)[j4] = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
}

// (a, b) -> packed bf16x2 of the high parts and of the low parts
__device__ __forceinline__ void split_bf16x2_pair(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ha = __float2bfloat16_rn(a), hb = __float2bfloat16_rn(b);
  hi = (uint32_t)__bfloat16_as_ushort(ha) | ((uint32_t)__bfloat16_as_ushort(hb) << 16);
  lo = pack_bf16x2(a - __bfloat162float(ha), b - __bfloat162float(hb));
}

// Operand formats of split_gemm.  Each gives the element type T, the k-block and MMA-step widths, the three MMAs of one
// step, and the epilogue's 16-value row accesses: load16 reads hi + lo, store16 splits v into (hi, lo) and writes both.
// Both take `full` (one vector access per array) or else touch only the first n values; out_full / ub_full are the
// format's conditions for a full chunk of the bias output and of the coupling's transformed columns.
struct Tf32x3 {
  using T = float;
  static constexpr int BK = 32, UMMA_K = 8;
  __device__ static uint32_t idesc(uint32_t n) { return make_idesc_tf32(n, 2 * TC_BM); }
  __device__ static void mma3(uint32_t d, uint64_t ah, uint64_t al, uint64_t wh, uint64_t wl, uint32_t idesc, uint32_t acc) {
    umma_tf32_2sm(d, ah, wh, idesc, acc);
    umma_tf32_2sm(d, ah, wl, idesc, 1u);
    umma_tf32_2sm(d, al, wh, idesc, 1u);
  }
  __device__ static bool out_full(const float* hi, int n) { return n >= 16 && (reinterpret_cast<uintptr_t>(hi) & 15) == 0; }
  // 64 contiguous bytes of the row per array: two 256-bit loads each, which need 32-byte alignment
  __device__ static bool ub_full(const float* hi, int n) { return n >= 16 && (reinterpret_cast<uintptr_t>(hi) & 31) == 0; }
  __device__ static void load16(const float* hi, const float* lo, bool full, int n, float (&u)[16]) {
    if (full) {
      uint4 q[4], ql[4];
      ld_global_256(hi, q[0], q[1]);
      ld_global_256(hi + 8, q[2], q[3]);
      ld_global_256(lo, ql[0], ql[1]);
      ld_global_256(lo + 8, ql[2], ql[3]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        u[4 * i] = __uint_as_float(q[i].x) + __uint_as_float(ql[i].x);
        u[4 * i + 1] = __uint_as_float(q[i].y) + __uint_as_float(ql[i].y);
        u[4 * i + 2] = __uint_as_float(q[i].z) + __uint_as_float(ql[i].z);
        u[4 * i + 3] = __uint_as_float(q[i].w) + __uint_as_float(ql[i].w);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) u[j] = j < n ? hi[j] + lo[j] : 0.f;
    }
  }
  __device__ static void store16(float* hi, float* lo, bool full, int n, float (&v)[16]) {
    float l[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float h = tf32_hi(v[j]);
      l[j] = v[j] - h;
      v[j] = h;
    }
    if (full) {
      st16_f32(hi, v);
      st16_f32(lo, l);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j < n) {
          hi[j] = v[j];
          lo[j] = l[j];
        }
    }
  }
};

struct Bf16x2 {
  using T = uint16_t;
  static constexpr int BK = TC_BK, UMMA_K = TC_UMMA_K;
  __device__ static uint32_t idesc(uint32_t n) { return make_idesc(n, 2 * TC_BM); }
  __device__ static void mma3(uint32_t d, uint64_t ah, uint64_t al, uint64_t wh, uint64_t wl, uint32_t idesc, uint32_t acc) {
    umma_bf16_2sm(d, ah, wh, idesc, acc);
    umma_bf16_2sm(d, ah, wl, idesc, 1u);
    umma_bf16_2sm(d, al, wh, idesc, 1u);
  }
  // the (hi, lo) outputs are activation rows padded to the N tile: every chunk is stored whole
  __device__ static bool out_full(const uint16_t*, int) { return true; }
  // 16 coordinates = 32 bytes of the row per array: one 256-bit load each
  __device__ static bool ub_full(const uint16_t*, int n) { return n >= 16; }
  __device__ static void load16(const uint16_t* hi, const uint16_t* lo, bool full, int n, float (&u)[16]) {
    if (full) {
      uint4 q0, q1, l0, l1;
      float uh[16], ul[16];
      ld_global_256(hi, q0, q1);
      ld_global_256(lo, l0, l1);
      unpack_bf16x8(q0, uh);
      unpack_bf16x8(q1, uh + 8);
      unpack_bf16x8(l0, ul);
      unpack_bf16x8(l1, ul + 8);
#pragma unroll
      for (int j = 0; j < 16; ++j) u[j] = uh[j] + ul[j];
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        u[j] = j < n ? __uint_as_float((uint32_t)hi[j] << 16) + __uint_as_float((uint32_t)lo[j] << 16) : 0.f;
    }
  }
  __device__ static void store16(uint16_t* hi, uint16_t* lo, bool full, int n, float (&v)[16]) {
    if (full) {
      uint32_t ph[8], pl[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) split_bf16x2_pair(v[2 * j], v[2 * j + 1], ph[j], pl[j]);
      st_global_256(hi, make_uint4(ph[0], ph[1], ph[2], ph[3]), make_uint4(ph[4], ph[5], ph[6], ph[7]));
      st_global_256(lo, make_uint4(pl[0], pl[1], pl[2], pl[3]), make_uint4(pl[4], pl[5], pl[6], pl[7]));
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j < n) {
          const __nv_bfloat16 h = __float2bfloat16_rn(v[j]);
          hi[j] = __bfloat16_as_ushort(h);
          lo[j] = __bfloat16_as_ushort(__float2bfloat16_rn(v[j] - __bfloat162float(h)));
        }
    }
  }
};

template <class F>
__device__ __forceinline__ void split_gemm(const CUtensorMap& tmA, const CUtensorMap& tmAlo, const CUtensorMap& tmW,
                                           const CUtensorMap& tmWlo, const SplitArgs<typename F::T>& args) {
  using T = typename F::T;
  const int STAGES = args.stages;
  const uint32_t STAGE_BYTES = args.stage_bytes;
  extern __shared__ uint8_t smem_raw[];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  const uint32_t cta_rank = cluster_ctarank();
  const int unit = (int)(blockIdx.x >> 1), num_units = (int)(gridDim.x >> 1);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * STAGES + 4);
  const uint32_t epi_base = bar_base + TC_BAR_BYTES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 16);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_addr) : "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const int total_tiles = args.m_tiles * args.n_tiles;
  const int num_kb = (int)((args.K + F::BK - 1) / F::BK);
  const uint32_t w_rows_bytes = (uint32_t)(args.bn >> 1) * 128u;
  const uint32_t stage_tx = 2u * (2u * TC_A_BYTES + 2u * w_rows_bytes);
  const uint32_t off_alo = TC_A_BYTES, off_w = 2u * TC_A_BYTES, off_wlo = 2u * TC_A_BYTES + args.w_bytes;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    bool ok = true;
    for (int t = unit; t < total_tiles && ok; t += num_units) {
      const int mt = t / args.n_tiles, nt = t - mt * args.n_tiles;
      int width = (int)(args.N - (int64_t)nt * args.bn);
      if (width > args.bn) width = args.bn;
      const int w_row = nt * args.bn + (int)cta_rank * (width >> 1);
      const int a_row = (mt * 2 + (int)cta_rank) * TC_BM;
      for (int kb = 0; kb < num_kb; ++kb) {
        ok = mbar_wait(empty_bar(s), ph ^ 1u);
        if (!ok) break;
        const uint32_t dst = smem_base + s * STAGE_BYTES;
        if (elect_one()) {
          if (cta_rank == 0) mbar_expect_tx(full_bar(s), stage_tx);
          tma_load_2d_2sm(dst, &tmA, full_bar(s), kb * F::BK, a_row);
          tma_load_2d_2sm(dst + off_alo, &tmAlo, full_bar(s), kb * F::BK, a_row);
          tma_load_2d_2sm(dst + off_w, &tmW, full_bar(s), kb * F::BK, w_row);
          tma_load_2d_2sm(dst + off_wlo, &tmWlo, full_bar(s), kb * F::BK, w_row);
        }
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (cta_rank == 0) {
      int s = 0, a = 0;
      uint32_t ph = 0, aph = 0;
      bool ok = true;
      const int tail_steps = ((int)args.K - (num_kb - 1) * F::BK + F::UMMA_K - 1) / F::UMMA_K;
      const uint64_t desc_hi = make_smem_desc(0);
      const uint32_t lo0 = (smem_base & 0x3FFFFu) >> 4, stage16 = STAGE_BYTES >> 4;
      for (int t = unit; t < total_tiles && ok; t += num_units) {
        const int nt = t % args.n_tiles;
        int width = (int)(args.N - (int64_t)nt * args.bn);
        if (width > args.bn) width = args.bn;
        const uint32_t idesc = F::idesc((uint32_t)width);
        ok = mbar_wait(tempty_bar(a), aph ^ 1u);
        if (!ok) break;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)a * TC_MAX_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          ok = mbar_wait(full_bar(s), ph);
          if (!ok) break;
          if (elect_one()) {
            // one MMA step is 32 bytes of the 128-byte swizzle row: the descriptors advance by 2 x 16-byte units
            const uint64_t ah = desc_hi | (uint64_t)(lo0 + (uint32_t)s * stage16);
            const uint64_t al = ah + (off_alo >> 4), wh = ah + (off_w >> 4), wl = ah + (off_wlo >> 4);
            const int ksteps = kb + 1 < num_kb ? F::BK / F::UMMA_K : tail_steps;
            for (int k = 0; k < ksteps; ++k)
              F::mma3(d_tmem, ah + 2u * k, al + 2u * k, wh + 2u * k, wl + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2sm(empty_bar(s));
          }
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        if (!ok) break;
        if (elect_one()) umma_commit_2sm(tfull_bar(a));
        a ^= 1;
        if (a == 0) aph ^= 1u;
      }
    }
  } else {
    const int lane_grp = warp & 3;
    const int half = (warp - 2) >> 2;
    const int et = (int)threadIdx.x - 64;
    const EpiParams& ep = args.ep;
    float* epi = reinterpret_cast<float*>(smem_raw + (epi_base - smem_u32(smem_raw)));
    const int mode = ep.mode;
    const bool is_cpl = mode == EPI_COUPLING_INV || mode == EPI_COUPLING_FWD;
    const bool is_add = mode == EPI_ADD_INV || mode == EPI_ADD_FWD;
    const bool is_base = mode == EPI_BASE_NORMAL || mode == EPI_BASE_LAPLACE;
    // column vectors resident for the whole kernel (host guarantees N <= TC_EPI_COLS)
    for (int i = et; i < (int)args.N; i += 256) {
      epi[i] = ep.bias != nullptr ? ep.bias[i] : 0.f;
      if (is_base) {
        const bool v2 = i < args.n_valid && ep.loc != nullptr;
        epi[TC_EPI_COLS + i] = v2 ? ep.loc[i] : 0.f;
        epi[2 * TC_EPI_COLS + i] = v2 ? ep.inv_scale[i] : 0.f;
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    int a = 0;
    uint32_t aph = 0;
    for (int t = unit; t < total_tiles; t += num_units) {
      const int mt = t / args.n_tiles, nt = t - mt * args.n_tiles;
      const int64_t row = (int64_t)(mt * 2 + (int)cta_rank) * TC_BM + lane_grp * 32 + lane;
      const bool rvalid = row < args.M;
      const int64_t n0 = (int64_t)nt * args.bn;
      int width = (int)(args.N - n0);
      if (width > args.bn) width = args.bn;
      const float* ev = epi + n0;
      const bool ok = mbar_wait(tfull_bar(a), aph);
      if (ok) {
        tc_fence_after();
        const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)a * TC_MAX_BN;
        if (mode == EPI_BIAS || mode == EPI_BIAS_RELU) {
          for (int c = half * 16; c < width; c += 32) {
            float v[16];
            tmem_ld16(t_base + c, v);
            tmem_ld_wait();
            if (rvalid) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                v[j] += ev[c + j];
                if (mode == EPI_BIAS_RELU) v[j] = fmaxf(v[j], 0.f);
              }
              const int64_t off = row * ep.ldo + n0 + c;
              const int n = args.n_valid - (int)(n0 + c);   // valid columns of this chunk
              if (args.out_lo != nullptr) {
                // the output travels as (hi, lo), hi + lo = v: the next GEMM's A
                T* dh = reinterpret_cast<T*>(ep.out) + off;
                F::store16(dh, args.out_lo + off, F::out_full(dh, n), n, v);
              } else {
                float* dst = reinterpret_cast<float*>(ep.out) + off;
                if (n >= 16 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                  st16_f32(dst, v);
                } else {
#pragma unroll
                  for (int j = 0; j < 16; ++j)
                    if (j < n) dst[j] = v[j];
                }
              }
            }
          }
        } else if (is_cpl || is_add) {
          const int C = ep.C;
          float lsum = 0.f;
          for (int c = half * 16; c < C; c += 32) {
            float sv[16], tv[16];
            if (is_cpl) {
              tmem_ld16(t_base + c, sv);
              tmem_ld16(t_base + C + c, tv);
            } else {
              tmem_ld16(t_base + c, tv);
            }
            tmem_ld_wait();
            const int coord0 = nt * C + c;
            if (rvalid && coord0 < ep.Db) {
              T* up = reinterpret_cast<T*>(ep.ub) + row * ep.ldub + coord0;
              T* ulo = args.ub_lo + row * ep.ldub + coord0;
              const float* bt = is_cpl ? ev + C + c : ev + c;
              const int n = ep.Db - coord0;   // valid coordinates of this chunk
              const bool full = F::ub_full(up, n);
              float u[16];
              F::load16(up, ulo, full, n, u);
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float tt = tv[j] + bt[j];
                if (is_cpl) {
                  const float ls = ep.clamp * tanh_mufu(sv[j] + ev[c + j]);   // padded coordinates: s = 0 -> ls = 0
                  const float e = ex2_fast((mode == EPI_COUPLING_INV ? -ls : ls) * 1.4426950408889634f);
                  u[j] = mode == EPI_COUPLING_INV ? (u[j] - tt) * e : fmaf(u[j], e, tt);
                  lsum += ls;
                } else {
                  u[j] = mode == EPI_ADD_INV ? u[j] - tt : u[j] + tt;
                }
              }
              F::store16(up, ulo, full, n, u);
            }
          }
          if (is_cpl && rvalid && ep.row_acc != nullptr)
            row_accumulate(ep, row, nt * 2 + half, mode == EPI_COUPLING_INV ? -lsum : lsum);
        } else {   // base density
          float lsum = 0.f;
          const float* ev_loc = ev + TC_EPI_COLS;
          const float* ev_isc = ev + 2 * TC_EPI_COLS;
          for (int c = half * 16; c < width; c += 32) {
            float v[16];
            tmem_ld16(t_base + c, v);
            tmem_ld_wait();
            if (rvalid) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float z = v[j] + ev[c + j];
                if (ep.out != nullptr && n0 + c + j < args.n_valid)
                  reinterpret_cast<float*>(ep.out)[row * ep.ldo + n0 + c + j] = z;
                const float d = (z - ev_loc[c + j]) * ev_isc[c + j];
                lsum += (mode == EPI_BASE_NORMAL) ? -0.5f * d * d : -fabsf(d);
              }
            }
          }
          if (rvalid && ep.row_acc != nullptr && ep.loc != nullptr) row_accumulate(ep, row, nt * 2 + half, lsum);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (cta_rank == 0) mbar_arrive(tempty_bar(a));
          else mbar_arrive_cluster(tempty_bar(a), 0);
        }
      }
      a ^= 1;
      if (a == 0) aph ^= 1u;
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

__global__ void __launch_bounds__(TC_THREADS, 1)
usf_tc3_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAlo,
                    const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmWlo, SplitArgs<float> args) {
  split_gemm<Tf32x3>(tmA, tmAlo, tmW, tmWlo, args);
}

__global__ void __launch_bounds__(TC_THREADS, 1)
usf_tcb2_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAlo,
                     const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmWlo, SplitArgs<uint16_t> args) {
  split_gemm<Bf16x2>(tmA, tmAlo, tmW, tmWlo, args);
}

// (hi, lo) split of a (rows x cols) fp32 matrix: hi = x rounded to tf32 (written to `hi`, which may alias x, or skipped
// when NULL -- then lo is taken against the truncated value the tensor core would read from x itself), lo = x - hi
__global__ void usf_split_lo_kernel(const float* x, int64_t ldx, float* hi, float* lo, int64_t ldl, int64_t rows, int64_t cols) {
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols, c = i - r * cols;
    const float v = x[r * ldx + c];
    const float h = hi != nullptr ? tf32_hi(v) : __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    lo[r * ldl + c] = v - h;
    if (hi != nullptr) hi[r * ldx + c] = h;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 row-major tensor (rows x cols, leading dimension ld elements), box = box_rows x 64 cols, 128B swizzle.
// Encoding costs a driver call (~several us); a launch chain re-uses the same few (pointer, shape) combinations every
// step (packed weights, workspace slices), so encoded maps are memoised per thread.
struct TmapKey {
  const void* base;
  int64_t rows, cols, ld;
  int box_rows, elem_bytes;
  bool operator==(const TmapKey& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows &&
           elem_bytes == o.elem_bytes;
  }
};
struct TmapSlot {
  TmapKey key;
  CUtensorMap map;
  bool used;
};
constexpr int TMAP_CACHE_SLOTS = 256;

// elem_bytes = 2 (bf16, box of 64 columns) or 4 (fp32 read as tf32, box of 32 columns): one box row is always 128 bytes.
int make_tmap(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, int elem_bytes = 2) {
  static thread_local TmapSlot cache[TMAP_CACHE_SLOTS];
  const TmapKey key{base, rows, cols, ld, box_rows, elem_bytes};
  const uint64_t h = (reinterpret_cast<uintptr_t>(base) >> 4) * 0x9E3779B97F4A7C15ull ^ (uint64_t)rows * 0xC2B2AE3D27D4EB4Full ^
                     (uint64_t)cols * 0x165667B19E3779F9ull ^ (uint64_t)ld * 31 ^ (uint64_t)box_rows ^ ((uint64_t)elem_bytes << 40);
  TmapSlot& slot = cache[(h >> 20) % TMAP_CACHE_SLOTS];
  if (slot.used && slot.key == key) {
    *tm = slot.map;
    return USF_OK;
  }
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return USF_E_CUDA;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * (cuuint64_t)elem_bytes};
  const cuuint32_t box[2] = {(cuuint32_t)(128 / elem_bytes), (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(tm, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): base=%p rows=%lld cols=%lld ld=%lld box_rows=%d", (int)r,
              (const void*)base, (long long)rows, (long long)cols, (long long)ld, box_rows);
    return USF_E_CUDA;
  }
  slot.key = key;
  slot.map = *tm;
  slot.used = true;
  return USF_OK;
}

}  // namespace

const char* const kTcGemmKernelName = "usf_tc_gemm_kernel";

// USF_PDL=0 disables programmatic dependent launch of the tensor-core kernels.
static bool tc_pdl() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("USF_PDL"); v = (e != nullptr && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// Launch of a persistent CTA-pair kernel: one cluster of 2 CTAs per two SMs (at most one per work unit), with
// programmatic dependent launch unless USF_PDL=0.
template <class... Params, class... Args>
static int launch_pairs(void (*kernel)(Params...), int64_t units, int threads, uint32_t smem_bytes, cudaStream_t stream,
                        const Args&... args) {
  int64_t pairs = num_sms() / 2;
  if (pairs > units) pairs = units;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * pairs));
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = tc_pdl() ? 2 : 1;
  USF_CUDA(cudaLaunchKernelEx(&cfg, kernel, args...));
  return USF_OK;
}

// Tile order of the next tensor-core launches on this thread.  A launch chain alternates it kernel by kernel
// ("serpentine"): a kernel walks its row tiles first -> last and leaves the rows it wrote LAST in L2 (126 MB; the two
// ping-pong activation buffers of a 65536-row chunk are 2 x 105 MB), so the next kernel walks last -> first and reads
// what is still resident instead of streaming the whole buffer through an LRU cache in exactly the order that evicts
// every line just before it is needed (ncu, round 1: the GEMM read its whole 106 MB operand from DRAM).
// Measured on one box, alternating (profiles/r2/ab_matrix.txt): affine GEMM 69.6 -> 67.8 us, fused conditioner kernel
// 85.5 -> 82.9 us per launch.  (Tried with it and dropped: L2 eviction-priority hints on the TMA loads -- evict_first
// for the dead activation operand, evict_last for the weights -- cost 1 us per launch.)
static thread_local int g_tile_reverse = 0;
void tc_set_tile_order(int reverse) { g_tile_reverse = reverse ? 1 : 0; }

int tc_pick_bn(int64_t N) {
  // balanced N tiles: as few tiles as possible, equal width, multiple of 16, <= 256
  const int64_t nt = ceil_div(N, TC_MAX_BN);
  return (int)round_up(ceil_div(N, nt), 16);
}

int tc_gemm(const uint16_t* A, int64_t lda, const uint16_t* W, int64_t ldw, int64_t M, int64_t N, int64_t K, int bn,
            const EpiParams& ep, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return USF_OK;
  USF_CHECK_ARG(A && W, "tc_gemm: null operand");
  USF_CHECK_ARG((lda % 8) == 0 && (ldw % 8) == 0, "tc_gemm: leading dimensions must be multiples of 8 (got %lld, %lld)",
                (long long)lda, (long long)ldw);
  USF_CHECK_ARG((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
                "tc_gemm: operands must be 16-byte aligned");
  USF_CHECK_ARG(bn >= 16 && bn <= TC_MAX_BN && (bn % 16) == 0 && (N % 16) == 0 && K > 0,
                "tc_gemm: bad tile/shape (bn=%d N=%lld K=%lld)", bn, (long long)N, (long long)K);
  if (ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD)
    USF_CHECK_ARG(bn == 2 * ep.C && (ep.C % 16) == 0 && (N % bn) == 0 && (reinterpret_cast<uintptr_t>(ep.ub) & 31) == 0 &&
                      (ep.ldub % 16) == 0,
                  "tc_gemm: coupling tile must be [s(C)|t(C)] and the b-part 32-byte aligned");
  if ((ep.mode == EPI_BIAS || ep.mode == EPI_BIAS_RELU) && ep.out_bf16)
    USF_CHECK_ARG((reinterpret_cast<uintptr_t>(ep.out) & 31) == 0 && (ep.ldo % 16) == 0, "tc_gemm: bf16 output must be 32-byte aligned");
  if (ep.mode == EPI_ADD_INV || ep.mode == EPI_ADD_FWD)
    USF_CHECK_ARG(bn == ep.C && ep.C <= 128 && (N % bn) == 0 && (reinterpret_cast<uintptr_t>(ep.ub) & 31) == 0 &&
                      (ep.ldub % 16) == 0,
                  "tc_gemm: additive tile must be [t(C <= 128)] and the b-part 32-byte aligned");

  static bool attr_set = false;
  if (!attr_set) {
    USF_CUDA(cudaFuncSetAttribute(usf_tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
    attr_set = true;
  }
  CUtensorMap tmA, tmW;
  int rc = make_tmap(&tmA, A, M, K, lda, TC_BM);
  if (rc) return rc;
  rc = make_tmap(&tmW, W, N, K, ldw, bn / 2);
  if (rc) return rc;

  TcArgs args;
  args.M = M;
  args.N = N;
  args.K = K;
  args.bn = bn;
  args.n_tiles = (int)ceil_div(N, bn);
  args.m_tiles = (int)ceil_div(M, 2 * TC_BM);
  args.n_valid = ep.n_valid > 0 ? ep.n_valid : (int)N;
  args.ep = ep;
  args.reverse = g_tile_reverse;
  args.stage_bytes = TC_A_BYTES + (uint32_t)round_up((int64_t)(bn / 2) * TC_BK * 2, 1024);
  args.stages = (int)((TC_SMEM_BYTES - TC_FIXED_BYTES) / args.stage_bytes);
  if (args.stages > TC_MAX_STAGES) args.stages = TC_MAX_STAGES;
  if (args.stages < 2) { set_error("tc_gemm: tile does not fit in shared memory"); return USF_E_ARG; }
  return launch_pairs(usf_tc_gemm_kernel, (int64_t)args.m_tiles * args.n_tiles, TC_THREADS, TC_SMEM_BYTES, stream, tmA, tmW,
                      args);
}

// Split-operand GEMM launcher (see split_gemm): T = float runs 3xTF32 (usf_tc3_gemm_kernel), T = uint16_t bf16x2
// (usf_tcb2_gemm_kernel).  A, Alo: (M, lda); W, Wlo: (N, ldw); leading dimensions of 16-byte pitches, N multiple of 16
// and <= TC_EPI_COLS.
template <class T>
int tc_split_gemm(const T* A, const T* Alo, int64_t lda, const T* W, const T* Wlo, int64_t ldw, int64_t M, int64_t N,
                  int64_t K, int bn, const EpiParams& ep, T* out_lo, T* ub_lo, cudaStream_t stream) {
  constexpr bool t3 = std::is_same<T, float>::value;
  void (*kernel)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, SplitArgs<T>);
  if constexpr (t3) kernel = usf_tc3_gemm_kernel;
  else kernel = usf_tcb2_gemm_kernel;
  if (M <= 0 || N <= 0) return USF_OK;
  USF_CHECK_ARG(A && Alo && W && Wlo, "tc_split_gemm: null operand");
  USF_CHECK_ARG((lda * sizeof(T)) % 16 == 0 && (ldw * sizeof(T)) % 16 == 0,
                "tc_split_gemm: leading dimensions must be multiples of 16 bytes");
  USF_CHECK_ARG(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Alo) | reinterpret_cast<uintptr_t>(W) |
                  reinterpret_cast<uintptr_t>(Wlo)) & 15) == 0, "tc_split_gemm: operands must be 16-byte aligned");
  USF_CHECK_ARG(bn >= 16 && bn <= TC_MAX_BN && (bn % 16) == 0 && (N % 16) == 0 && K > 0 && N <= TC_EPI_COLS,
                "tc_split_gemm: bad tile/shape (bn=%d N=%lld K=%lld)", bn, (long long)N, (long long)K);
  const bool cpl = ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD;
  const bool add = ep.mode == EPI_ADD_INV || ep.mode == EPI_ADD_FWD;
  if (cpl) USF_CHECK_ARG(bn == 2 * ep.C && (N % bn) == 0 && ub_lo != nullptr && !ep.ub_bf16 == t3, "tc_split_gemm: bad coupling tile");
  if (add) USF_CHECK_ARG(bn == ep.C && (N % bn) == 0 && ub_lo != nullptr && !ep.ub_bf16 == t3, "tc_split_gemm: bad additive tile");
  static bool attr_set = false;
  if (!attr_set) {
    USF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
    attr_set = true;
  }
  CUtensorMap tmA, tmAlo, tmW, tmWlo;
  int rc = make_tmap(&tmA, A, M, K, lda, TC_BM, sizeof(T));
  if (!rc) rc = make_tmap(&tmAlo, Alo, M, K, lda, TC_BM, sizeof(T));
  if (!rc) rc = make_tmap(&tmW, W, N, K, ldw, bn / 2, sizeof(T));
  if (!rc) rc = make_tmap(&tmWlo, Wlo, N, K, ldw, bn / 2, sizeof(T));
  if (rc) return rc;
  SplitArgs<T> args;
  memset(&args, 0, sizeof(args));
  args.M = M; args.N = N; args.K = K; args.bn = bn;
  args.n_tiles = (int)ceil_div(N, bn);
  args.m_tiles = (int)ceil_div(M, 2 * TC_BM);
  args.n_valid = ep.n_valid > 0 ? ep.n_valid : (int)N;
  args.ep = ep;
  args.out_lo = out_lo;
  args.ub_lo = ub_lo;
  args.w_bytes = (uint32_t)round_up((int64_t)(bn / 2) * 128, 1024);
  args.stage_bytes = 2u * TC_A_BYTES + 2u * args.w_bytes;
  args.stages = (int)((TC_SMEM_BYTES - TC_FIXED_BYTES) / args.stage_bytes);
  if (args.stages > TC_MAX_STAGES) args.stages = TC_MAX_STAGES;
  if (args.stages < 2) { set_error("tc_split_gemm: tile does not fit in shared memory"); return USF_E_ARG; }
  return launch_pairs(kernel, (int64_t)args.m_tiles * args.n_tiles, TC_THREADS, TC_SMEM_BYTES, stream, tmA, tmAlo, tmW,
                      tmWlo, args);
}
template int tc_split_gemm<float>(const float*, const float*, int64_t, const float*, const float*, int64_t, int64_t,
                                  int64_t, int64_t, int, const EpiParams&, float*, float*, cudaStream_t);
template int tc_split_gemm<uint16_t>(const uint16_t*, const uint16_t*, int64_t, const uint16_t*, const uint16_t*, int64_t,
                                     int64_t, int64_t, int64_t, int, const EpiParams&, uint16_t*, uint16_t*, cudaStream_t);

// fp32 rows -> (hi, lo) bf16 pairs in the activation layout (pad columns zero), optional per-row accumulator seed.
// HBM-bound (4 D bytes read, 4 ldy written per row): 8 columns per thread, 16-byte loads when the source row allows,
// one 16-byte store per output array.
__global__ void usf_split_rows_bf16x2_kernel(const float* __restrict__ x, int64_t ldx, uint16_t* hi, uint16_t* lo,
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
    uint32_t ph[4], pl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_bf16x2_pair(v[2 * j], v[2 * j + 1], ph[j], pl[j]);
    *reinterpret_cast<uint4*>(hi + r * ldy + c) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    *reinterpret_cast<uint4*>(lo + r * ldy + c) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
    if (c == 0 && row_init != nullptr) row_init[r] = init_value;
  }
}

int launch_split_rows_bf16x2(const float* x, int64_t ldx, uint16_t* hi, uint16_t* lo, int64_t ldy, int64_t B, int64_t D,
                             float* row_init, float init_value, cudaStream_t stream) {
  if (B <= 0) return USF_OK;
  const int64_t total = B * (ldy >> 3);          // ldy is a multiple of 16
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  usf_split_rows_bf16x2_kernel<<<(unsigned)blocks, 256, 0, stream>>>(x, ldx, hi, lo, ldy, B, D, row_init, init_value);
  USF_LAUNCH_CHECK("usf_split_rows_bf16x2_kernel");
  return USF_OK;
}

int launch_split_lo(const float* x, int64_t ldx, float* hi, float* lo, int64_t ldl, int64_t rows, int64_t cols, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return USF_OK;
  const int64_t total = rows * cols;
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  usf_split_lo_kernel<<<(unsigned)blocks, 256, 0, stream>>>(x, ldx, hi, lo, ldl, rows, cols);
  USF_LAUNCH_CHECK("usf_split_lo_kernel");
  return USF_OK;
}

// Fused conditioner chain + coupling (see usf_tc_mlp_coupling_kernel).  Returns USF_E_UNSUPPORTED when the shapes do
// not fit the fused kernel (the caller then runs the layer-by-layer chain).
bool tc_mlp_supported(int n_layers, const int* N, const int* K, int Da) {
  if (n_layers < 2 || n_layers > MLP_MAX_LAYERS) return false;
  if (K[0] != Da || Da <= 0) return false;
  int total_n = 0;
  for (int l = 0; l < n_layers; ++l) total_n += N[l];
  if (total_n > 3 * TC_EPI_COLS) return false;   // all bias vectors stay resident in shared memory
  for (int l = 0; l + 1 < n_layers; ++l)
    if (N[l] > 256 || (N[l] % 16) != 0 || K[l + 1] > N[l]) return false;
  static int off = -1;
  if (off < 0) { const char* e = getenv("USF_TC_FUSED_MLP"); off = (e != nullptr && e[0] == '0') ? 1 : 0; }
  return off == 0;
}

int tc_mlp_coupling(const uint16_t* A, int64_t lda, int64_t M, int n_layers, const uint16_t* const* Wb, const int* ldw,
                    const float* const* bias, const int* N, const int* K, int bn_last, const EpiParams& ep,
                    cudaStream_t stream) {
  if (M <= 0) return USF_OK;
  USF_CHECK_ARG(tc_mlp_supported(n_layers, N, K, K[0]), "tc_mlp_coupling: unsupported shape");
  USF_CHECK_ARG((lda % 8) == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0, "tc_mlp_coupling: bad activation layout");
  static bool attr_set = false;
  if (!attr_set) {
    USF_CUDA(cudaFuncSetAttribute(usf_tc_mlp_coupling_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MLP_SMEM_BYTES));
    attr_set = true;
  }
  MlpArgs args;
  memset(&args, 0, sizeof(args));
  MlpMaps maps;
  memset(&maps, 0, sizeof(maps));
  CUtensorMap tmA;
  int rc = make_tmap(&tmA, A, M, K[0], lda, TC_BM);
  if (rc) return rc;
  args.M = M;
  args.m_tiles = (int)ceil_div(M, 2 * TC_BM);
  args.L = n_layers;
  for (int l = 0; l < n_layers; ++l) {
    const bool last = l == n_layers - 1;
    args.K[l] = K[l];
    args.N[l] = N[l];
    args.bn[l] = last ? bn_last : N[l];
    args.ntile[l] = (int)ceil_div(N[l], args.bn[l]);
    args.bias[l] = bias[l];
    args.boff[l] = l == 0 ? 0 : args.boff[l - 1] + N[l - 1];
    USF_CHECK_ARG((ldw[l] % 8) == 0 && (N[l] % 16) == 0 && (args.bn[l] % 16) == 0 && args.bn[l] <= TC_MAX_BN,
                  "tc_mlp_coupling: bad layer %d", l);
    rc = make_tmap(&maps.w[l], Wb[l], N[l], K[l], ldw[l], args.bn[l] / 2);
    if (rc) return rc;
  }
  if (ep.mode == EPI_COUPLING_INV || ep.mode == EPI_COUPLING_FWD)
    USF_CHECK_ARG(bn_last == 2 * ep.C && (ep.C % 16) == 0 && (N[n_layers - 1] % bn_last) == 0 &&
                      (reinterpret_cast<uintptr_t>(ep.ub) & 31) == 0 && (ep.ldub % 16) == 0,
                  "tc_mlp_coupling: bad coupling tile");
  else
    USF_CHECK_ARG((ep.mode == EPI_ADD_INV || ep.mode == EPI_ADD_FWD) && bn_last == ep.C && ep.C <= 128 &&
                      (N[n_layers - 1] % bn_last) == 0 && (reinterpret_cast<uintptr_t>(ep.ub) & 31) == 0 && (ep.ldub % 16) == 0,
                  "tc_mlp_coupling: bad additive tile");
  args.ep = ep;
  args.reverse = g_tile_reverse;
  return launch_pairs(usf_tc_mlp_coupling_kernel, args.m_tiles, MLP_THREADS, MLP_SMEM_BYTES, stream, tmA, maps, args);
}

int tc_timeout_flag(int* out, int reset) {
  int v = 0;
  cudaError_t e = cudaMemcpyFromSymbol(&v, g_tc_timeout, sizeof(int));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyFromSymbol(g_tc_timeout)");
  if (out) *out = v;
  if (reset && v) {
    const int z = 0;
    e = cudaMemcpyToSymbol(g_tc_timeout, &z, sizeof(int));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyToSymbol(g_tc_timeout)");
  }
  return USF_OK;
}

}  // namespace usf
