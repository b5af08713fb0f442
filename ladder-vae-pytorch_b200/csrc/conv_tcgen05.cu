// bf16 implicit-GEMM convolution on the 5th-generation tensor cores (sm_100a only):
// TMA (cp.async.bulk.tensor) -> 128B-swizzled shared memory -> tcgen05.mma with the fp32
// accumulator in TMEM -> tcgen05.ld epilogue (bias, Dropout2d channel scale, residual).
//
// Covers the stride-1 "same" convolutions that carry ~97% of the model's FLOPs
// (lib/nn.py:83-87 3x3 64->64, lib/nn.py:118 1x1 64->128 gate, models/lvae_layers.py:350 1x1
// merge over two 64-channel inputs, lib/stochastic.py:25-26 3x3 64->64, lib/likelihoods.py:199
// 3x3 64->100) and, with flipped taps and transposed weights, their data gradients.
//
// GEMM view: D[128 pixels, N] += A_tap[128 pixels, 64 ch] * W_tap[N, 64 ch]^T, one k-block of 64
// channels per filter tap (or per input tensor for the merge).  A tile of 128 consecutive NHWC
// pixels is ONE 4-D TMA box {64 ch, bw, bh, bn}; shifting the box origin by the tap offset
// implements im2col, and TMA's out-of-bounds zero fill implements the zero padding (the batch is
// its own tensor dimension, so a shifted box never bleeds into the neighbouring image).
// All taps' weights stay resident in shared memory for the lifetime of a persistent CTA when they leave room for at least
// two activation stages ("resident").  Wider layers (3x3 128 -> 128 is 288 KB of weights) stream them instead: each
// pipeline stage then carries the A box of a k-block and the matching [Npad][64] weight tile, landing on one barrier
// ("streamed", plain epilogues only).  tc_weight_plan decides from the shape alone; lvae_conv2d_tc_plan exposes it.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA
// issuer, warps 2..9 = epilogue (TMEM lane quadrant = warp_id % 4, two warps per quadrant split the columns).  The accumulator is double
// buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
#include "common.cuh"
#include <cuda.h>
#include <string.h>
#include <mutex>

namespace {

constexpr int TC_THREADS = 320;        // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quadrant)
constexpr int TC_BM = 128;             // pixels per tile
constexpr int TC_BK = 64;              // channels per k-block (= one 128-byte swizzle row of bf16)
constexpr int TC_STAGE_BYTES = TC_BM * TC_BK * 2;   // 16 KB
constexpr int TC_MAX_KB = 36;          // k-blocks per tile: taps x input k-blocks

struct TcParams {
  const float* bias;        // [N] or null
  const float* out_scale;   // (B, N) or null
  const void* res;          // residual (M, N) same dtype as y, or null
  void* y;                  // (M, nsplit) when y2 != null else (M, N)
  void* y2;                 // optional second output for columns >= nsplit: (M, N - nsplit)
  int M_total, H, W, N, Npad, nsplit;
  int n_kb;                 // number of k-blocks (taps * inputs)
  int n_stages;
  int bw, bh, bn;           // TMA box (pixels) : bw*bh*bn == 128
  int out_f32;              // 1: y is fp32, 0: bf16
  int tmem_cols;
  // halo mode (3x3, W % 8 == 0, H % 16 == 0): ONE TMA box of 18 rows x 16 columns per 16x8-pixel tile; the nine
  // tap operands are the same shared-memory tile read through shifted UMMA descriptors (no per-tap re-fetch)
  int halo, stage_bytes, tiles_x, tiles_per_img;
  // H, W (hence tiles_x, tiles_per_img) are powers of two: the epilogue's per-tile index arithmetic is shifts and masks (the
  // 64-bit m / hw and the tile divisions cost several hundred cycles per tile on the exposed tail of every launch)
  int lg_w, lg_hw, lg_tx, lg_tpi;
  // reductions fused into the TMA-store epilogue (N == 64 only)
  double* stats_acc;        // += per-channel sum / sum of squares of the output as stored (next BatchNorm's statistics)
  const __nv_bfloat16* bnb_x;   // BatchNorm-backward reduction over this dgrad's output: BN input x (M,64)
  const float* bnb_save; const float* bnb_gamma; const float* bnb_beta;
  double* bnb_acc;          // += sum(g), sum(g * xhat), g = dy * act'(xhat*gamma+beta)
  int bnb_act;
  // gated-residual epilogue (1x1 gate conv, N == 128): out = act(h[:, :64]) * sigmoid(h[:, 64:]) + gate_x, stored through tmY2;
  // stats_acc (optional) then accumulates the statistics of out
  const __nv_bfloat16* gate_x;
  int gate_act;
  int gate_skip_h;          // eval mode: h = [a | g] is only staged for the gate pass, never stored (nothing runs backward)
  int tma_store;            // bf16 output, N % 64 == 0, no residual: epilogue stages the tile in smem and stores it with TMA
  // eval-mode BatchNorm + activation of the CONSUMER folded into this conv's epilogue (FUSE 4, N == 64, no_grad callers):
  // y = act((acc + bias) * s + (beta - mean * s)), s = gamma * rsqrt(var + eps) -- derived in the prologue from the running
  // statistics, so the separate BatchNorm-apply pass (one read + one write of the tensor, one launch) disappears
  const float* fold_gamma; const float* fold_beta; const float* fold_mean; const float* fold_var;
  float fold_eps;
  int fold_act;
  // ... and the eval-mode BatchNorm + activation in FRONT of this conv applied to its operand on the way in (FUSE 4, halo tiles):
  // five transform warps rewrite every landed halo tile in place, x -> act(x * s + t), before the MMA warp may read it, and leave
  // the zero fill of the out-of-image pixels alone (it is the convolution's padding of the ACTIVATED tensor).  The separate
  // BatchNorm-apply pass of the block input disappears: one launch and one read + write of the tensor less (lib/nn.py:78-81).
  const float* pre_gamma; const float* pre_beta; const float* pre_mean; const float* pre_var;
  float pre_eps;
  long long* dbg;           // optional per-tile clock64 trace of CTA 0 (profiling aid, normally null)
  int8_t dx[TC_MAX_KB], dy[TC_MAX_KB], src[TC_MAX_KB], coff[TC_MAX_KB];   // coff: channel offset / 64 inside the tensor
  // stride-2 convolutions (lvae_conv2d_tc_s2): the tile's pixel coordinates are multiplied by in_stride before the tap
  // offset is added (the input tensor map then traverses with the same element stride), and k-block kb reads weight
  // block wblk[kb] of the packed buffer (a parity class of a transposed convolution uses a subset of the nine taps)
  int in_stride, use_wblk;
  int8_t wblk[TC_MAX_KB];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(tm), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO), version 1
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);          // start address
  d |= (uint64_t)1 << 16;                            // LBO (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                  // SBO
  d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
  return d;
}
// same, with the 8-row groups sbo bytes apart and a start address that is only 128-byte aligned.  The base-offset field
// stays zero: the hardware swizzle is a function of the absolute shared-memory address
__device__ __forceinline__ uint64_t umma_desc_k_sw128_shifted(uint32_t saddr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// one elected lane of a fully converged warp (lets ptxas keep the MMA operands in uniform registers instead of
// wrapping every tcgen05.mma in a per-lane broadcast loop)
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Epilogue for 16 accumulator columns [c0, c0+16) of one output row: bias (shared memory), Dropout2d scale,
// residual, conversion, vectorised store.  All global reads go through the read-only path so that the
// compiler can batch them instead of ordering them against the stores.
template <bool OUT_F32>
__device__ __forceinline__ void epilogue16(const uint32_t* __restrict__ r, const float* __restrict__ sbias,
                                           const float* __restrict__ scale_row, const void* __restrict__ res_row,
                                           void* __restrict__ out_row, int c0, int cc, int nvalid, int ncols, int N) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) + sbias[c0 + j];
  if (scale_row) {
    if (c0 + 16 <= N && (N & 3) == 0) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float4 s4 = __ldg(reinterpret_cast<const float4*>(scale_row + c0) + q);
        v[4 * q] *= s4.x; v[4 * q + 1] *= s4.y; v[4 * q + 2] *= s4.z; v[4 * q + 3] *= s4.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)                  // static indexing keeps v[] in registers
        if (c0 + j < N) v[j] *= __ldg(scale_row + c0 + j);
    }
  }
  if (OUT_F32) {
    float* o = (float*)out_row + cc;
    const float* rr = res_row ? (const float*)res_row + cc : nullptr;
    if (nvalid == 16 && (ncols & 3) == 0) {
      if (rr) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 t = __ldg(reinterpret_cast<const float4*>(rr) + q);
          v[4 * q] += t.x; v[4 * q + 1] += t.y; v[4 * q + 2] += t.z; v[4 * q + 3] += t.w;
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(o)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j < nvalid) o[j] = v[j] + (rr ? __ldg(rr + j) : 0.f);
    }
  } else {
    __nv_bfloat16* o = (__nv_bfloat16*)out_row + cc;
    const __nv_bfloat16* rr = res_row ? (const __nv_bfloat16*)res_row + cc : nullptr;
    if (nvalid == 16 && (ncols & 7) == 0) {
      if (rr) {
        uint4 r0 = __ldg(reinterpret_cast<const uint4*>(rr)), r1 = __ldg(reinterpret_cast<const uint4*>(rr) + 1);
        const __nv_bfloat162* h0 = reinterpret_cast<const __nv_bfloat162*>(&r0);
        const __nv_bfloat162* h1 = reinterpret_cast<const __nv_bfloat162*>(&r1);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float2 f0 = __bfloat1622float2(h0[j]), f1 = __bfloat1622float2(h1[j]);
          v[2 * j] += f0.x; v[2 * j + 1] += f0.y; v[8 + 2 * j] += f1.x; v[8 + 2 * j + 1] += f1.y;
        }
      }
      uint4 w0, w1;
      __nv_bfloat162* g0 = reinterpret_cast<__nv_bfloat162*>(&w0);
      __nv_bfloat162* g1 = reinterpret_cast<__nv_bfloat162*>(&w1);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        g0[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        g1[j] = __floats2bfloat162_rn(v[8 + 2 * j], v[8 + 2 * j + 1]);
      }
      reinterpret_cast<uint4*>(o)[0] = w0;
      reinterpret_cast<uint4*>(o)[1] = w1;
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j < nvalid) o[j] = __float2bfloat16(v[j] + (rr ? __bfloat162float(rr[j]) : 0.f));
    }
  }
}

// FUSE: 0 plain epilogue, 1 output statistics (stats_acc), 2 BatchNorm-backward sums (bnb_*), 3 gated residual output, 4 eval-mode
// BatchNorm + activation of the consumer (fold_*)
// (+ its statistics).  A template parameter so that the plain kernel carries no accumulator registers (the 10-warp CTA
// caps ptxas at 168 registers per thread).
// Round-2 A/B on the B200 (profiles/ab_r02_summary.txt) retired three variants of this kernel that held parity but lost time:
// CTA pairs on cta_group::2 (576 vs 834 TFLOP/s at 32x32), a dynamic tile scheduler (+0.15 ms / step) and a warp-transposed
// fp32 epilogue (90 vs 51 us for the 64 -> 100 head).
// ACT (FUSE 2 / 3 only): the activation of the fused BatchNorm-backward / gate pass as a compile-time constant (ACT_ELU, the
// model default) or -1 = runtime value; a switch inside the unrolled second pass costs one jump table per element.
// SW: streamed weights (FUSE == 0, non-halo tiles only): no resident weight block, stage = A box + B tile.
template <int FUSE, int ACT = -1, bool SW = false>
__global__ void __launch_bounds__(FUSE == 4 ? TC_THREADS + 160 : TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmY,
               const __grid_constant__ CUtensorMap tmY2, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the 128B swizzle atoms
  // (offset arithmetic on the __shared__ array, not on a uintptr_t: the compiler keeps the shared address space)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int wbytes_kb = p.Npad * 128;                        // one k-block of weights
  uint8_t* sW = smem;                                        // n_kb * Npad * 128 (resident weights only)
  uint8_t* sA = sW + (SW ? 0 : ((p.n_kb * wbytes_kb + 1023) & ~1023));  // n_stages * stage_bytes
  const int stage_bytes = p.halo ? p.stage_bytes : (SW ? TC_STAGE_BYTES + wbytes_kb : TC_STAGE_BYTES);
  uint8_t* sOut = sA + p.n_stages * stage_bytes;             // (N/64) x 16 KB output staging (TMA-store epilogue only)
  uint64_t* bars = (uint64_t*)(sOut + (p.tma_store ? (p.Npad / 64 + (FUSE == 3 ? 1 : 0)) * TC_STAGE_BYTES : 0));
  // barrier layout: [0..S) full, [S..2S) empty, 2S: weights, 2S+1..2S+2: tmem_full[2], 2S+3..2S+4: tmem_empty[2]
  const int S = p.n_stages;
  // FUSE 4: [2S+5 .. 3S+5) "stage transformed" (operand-path BatchNorm), tmem slot behind them (S <= 8: still below bars + 32)
  uint32_t* tmem_slot = (uint32_t*)(bars + (FUSE == 4 ? 3 * S + 5 : 2 * S + 5));
  const bool pre_bn = FUSE == 4 && p.pre_gamma != nullptr && p.halo;
  float* sbias = (float*)(bars + 32);                         // Npad floats (<= 256), zero beyond N / when bias == null
  float* sred = sbias + 256;                                  // 2 statistics x 8 warps x 64 channels (fused reductions)
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.halo ? (p.M_total / (p.H * p.W)) * p.tiles_per_img : (p.M_total + TC_BM - 1) / TC_BM;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA0);
    prefetch_tmap(&tmA1);
    prefetch_tmap(&tmW);
    for (int i = 0; i < S; ++i) {
      mbar_init(BAR(i), 1);
      mbar_init(BAR(S + i), 1);
    }
    mbar_init(BAR(2 * S), 1);
    mbar_init(BAR(2 * S + 1), 1);
    mbar_init(BAR(2 * S + 2), 1);
    mbar_init(BAR(2 * S + 3), 8);                  // one arrive per epilogue warp
    mbar_init(BAR(2 * S + 4), 8);
    if (FUSE == 4) for (int i = 0; i < S; ++i) mbar_init(BAR(2 * S + 5 + i), 5);     // one arrive per transform warp
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && !SW) {
    __syncwarp();
    // weights were packed many kernels ago: fetch them before waiting on the previous kernel (PDL prologue)
    if (elect_one()) {
      mbar_expect_tx(BAR(2 * S), (uint32_t)(p.n_kb * wbytes_kb));
      for (int kb = 0; kb < p.n_kb; ++kb)
        tma_load_2d(smem_u32(sW + kb * wbytes_kb), &tmW, BAR(2 * S), 0, (p.use_wblk ? p.wblk[kb] : kb) * p.Npad);
    }
    __syncwarp();
  }
  if (FUSE == 4) {
    // per-channel affine of the folded BatchNorm (parameters and running statistics: written long before this launch)
    for (int i = threadIdx.x; i < 64; i += TC_THREADS) {
      const float sc = p.fold_gamma[i] * rsqrtf(p.fold_var[i] + p.fold_eps);
      sred[i] = sc;
      sbias[i] = fmaf(p.bias ? p.bias[i] : 0.f, sc, p.fold_beta[i] - p.fold_mean[i] * sc);
      if (pre_bn) {                                  // same arithmetic as bn_act_fwd2's eval prologue: bit-identical operand
        const float rstd = rsqrtf(p.pre_var[i] + p.pre_eps);
        const float ps = rstd * p.pre_gamma[i];
        sred[64 + i] = ps;
        sred[128 + i] = p.pre_beta[i] - p.pre_mean[i] * ps;
      }
    }
  } else {
    for (int i = threadIdx.x; i < p.Npad; i += TC_THREADS) sbias[i] = (p.bias && i < p.N) ? p.bias[i] : 0.f;
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();          // activations / residual / dropout mask come from the previous kernels
  pdl_launch();
  if (warp == 0) {
    // ===================== TMA producer (whole warp loops, one elected lane issues) =====================
    {
      int stage = 0;
      uint32_t phase = 0;
      const int hw = p.H * p.W;
      for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x) {
        if (p.halo) {
          int n0 = tile / p.tiles_per_img;
          int r = tile - n0 * p.tiles_per_img;
          int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
          mbar_wait(BAR(S + stage), phase ^ 1);
          if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[(tile / gridDim.x) * 8 + 6] = clock64();
          if (elect_one()) {
            mbar_expect_tx(BAR(stage), (uint32_t)stage_bytes);
            tma_load_4d(smem_u32(sA + stage * stage_bytes), &tmA0, BAR(stage), 0, tx * 8 - 1, ty * 16 - 1, n0);
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1; }
          continue;
        }
        int p0 = tile * TC_BM;
        int n0 = p0 / hw;
        int rem = p0 - n0 * hw;
        int h0 = rem / p.W;
        int w0 = rem - h0 * p.W;
        if (p.in_stride > 1) { h0 *= p.in_stride; w0 *= p.in_stride; }
        for (int kb = 0; kb < p.n_kb; ++kb) {
          mbar_wait(BAR(S + stage), phase ^ 1);
          if (elect_one()) {
            uint8_t* dst = sA + stage * (SW ? stage_bytes : TC_STAGE_BYTES);
            mbar_expect_tx(BAR(stage), SW ? (uint32_t)stage_bytes : (uint32_t)TC_STAGE_BYTES);
            tma_load_4d(smem_u32(dst), p.src[kb] ? &tmA1 : &tmA0, BAR(stage), 64 * p.coff[kb],
                        w0 + p.dx[kb], h0 + p.dy[kb], n0);
            // streamed weights: this k-block's [Npad][64] tile lands behind the A box, on the same barrier
            if (SW) tma_load_2d(smem_u32(dst + TC_STAGE_BYTES), &tmW, BAR(stage), 0, (p.use_wblk ? p.wblk[kb] : kb) * p.Npad);
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs the loop (converged); one elected lane issues tcgen05.mma / tcgen05.commit, so ptxas keeps
    // descriptors and the TMEM address in uniform registers.
    {
      // instruction descriptor: D fp32, A/B bf16, both K-major, M = 128, N = Npad
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.Npad >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      if (!SW) mbar_wait(BAR(2 * S), 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x, ++it) {
        const int buf = it & 1;
        const uint32_t use = (uint32_t)(it >> 1);
        mbar_wait(BAR(2 * S + 3 + buf), (use & 1) ^ 1);      // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + (uint32_t)(buf * p.Npad);
        if (p.halo) {
          if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[it * 8 + 0] = clock64();
          mbar_wait(BAR(pre_bn ? 2 * S + 5 + stage : stage), phase);     // landed (and, with the operand-path BatchNorm, transformed)
          tc_fence_after();
          if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[it * 8 + 1] = clock64();
          const uint32_t a_base = smem_u32(sA + stage * stage_bytes);
          if (elect_one()) {
            for (int kb = 0; kb < p.n_kb; ++kb) {
              // tap (dy,dx): the tile's first pixel sits at halo row 1+dy, halo column 1+dx; rows are 16 pixels (2048 B)
              const uint32_t a_start = a_base + (uint32_t)(((1 + p.dy[kb]) * 16 + (1 + p.dx[kb])) * 128);
              const uint64_t adesc = umma_desc_k_sw128_shifted(a_start, 2048);
              const uint64_t bdesc = umma_desc_k_sw128(smem_u32(sW + kb * wbytes_kb));
#pragma unroll
              for (int k = 0; k < TC_BK / 16; ++k) {
                umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
              }
            }
            umma_commit(BAR(S + stage));
            umma_commit(BAR(2 * S + 1 + buf));
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1; }
          if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[it * 8 + 2] = clock64();
          continue;
        }
        for (int kb = 0; kb < p.n_kb; ++kb) {
          mbar_wait(BAR(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_addr = smem_u32(sA + stage * (SW ? stage_bytes : TC_STAGE_BYTES));
            const uint64_t adesc = umma_desc_k_sw128(a_addr);
            const uint64_t bdesc = umma_desc_k_sw128(SW ? a_addr + TC_STAGE_BYTES : smem_u32(sW + kb * wbytes_kb));
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k) {
              // advance 16 bf16 = 32 bytes along K inside the swizzle atom: +2 in the (addr >> 4) field
              umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
            }
            umma_commit(BAR(S + stage));                       // frees the smem stage when these MMAs retire
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(BAR(2 * S + 1 + buf));    // accumulator ready for the epilogue
        __syncwarp();
      }
    }
  } else if (FUSE == 4 && warp >= 10) {
    // ===================== operand transform (5 warps): halo tile -> act(BatchNorm_eval(halo tile)) in place =====================
    if (pre_bn) {
      const int t = (int)threadIdx.x - TC_THREADS;               // 0..159
      const int cphys = t & 7, slot = t >> 3;                    // 16-byte chunk of a 128-byte pixel row; 20 pixel slots
      const int hx = slot % 10, hy0 = slot / 10;                 // the MMAs read halo columns 0..9 only; rows hy0, hy0 + 2, ...
      const int clog = cphys ^ (hx & 7);                         // 128B swizzle: chunk index ^= (row & 7), row = 16 hy + hx
      float ps[8], pt[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { ps[e] = sred[64 + clog * 8 + e]; pt[e] = sred[128 + clog * 8 + e]; }
      const int fact = ACT >= 0 ? ACT : p.fold_act;
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x) {
        const int r = tile & (p.tiles_per_img - 1);
        const int ty = r >> p.lg_tx, tx = r & (p.tiles_x - 1);
        const int x = tx * 8 - 1 + hx;
        const bool xin = x >= 0 && x < p.W;
        mbar_wait(BAR(stage), phase);                            // TMA landed (async-proxy writes visible after the wait)
        uint8_t* base = sA + stage * stage_bytes + hx * 128 + (cphys << 4);
#pragma unroll
        for (int j = 0; j < 9; ++j) {
          const int hy = hy0 + 2 * j;
          const int y = ty * 16 - 1 + hy;
          if (xin && y >= 0 && y < p.H) {                        // out-of-image pixels stay zero: padding of the activated tensor
            uint4* ptr = reinterpret_cast<uint4*>(base + hy * 2048);
            uint4 v = *ptr;
            uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float a = act_fwd_t<true>(fmaf(__uint_as_float(w[q] << 16), ps[2 * q], pt[2 * q]), fact);
              const float b = act_fwd_t<true>(fmaf(__uint_as_float(w[q] & 0xFFFF0000u), ps[2 * q + 1], pt[2 * q + 1]), fact);
              const __nv_bfloat162 ob = __floats2bfloat162_rn(a, b);
              w[q] = *reinterpret_cast<const uint32_t*>(&ob);
            }
            *ptr = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to tcgen05.mma
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(2 * S + 5 + stage));
        if (++stage == S) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= 2) {
    // ===================== epilogue (8 warps: quadrant x column half) =====================
    const int quad = warp & 3;                                 // TMEM lane quadrant this warp may read
    const int half = (warp - 2) >> 2;                          // which 32-column chunks (even / odd) this warp drains
    const int row = quad * 32 + lane;
    const int hw = p.H * p.W;
    // Fused reductions (FUSE != 0) run as a second, channel-major pass over the staged bf16 output tile: epilogue warp e
    // owns rows [16 e, 16 e + 16), lane l owns channels 2l and 2l+1, so the per-channel constants and the running sums
    // live in a handful of registers and no cross-lane traffic is needed until the CTA's last tile.
    const int ew = warp - 2;
    float ra0 = 0.f, ra1 = 0.f, rb0 = 0.f, rb1 = 0.f;              // sums A / B of channels 2l, 2l+1
    float kx0 = 0.f, kx1 = 0.f, kb0 = 0.f, kb1 = 0.f, kg0 = 0.f, kg1 = 0.f, kc0 = 0.f, kc1 = 0.f;
    if (FUSE == 2) {
      // xhat = x * kx + kb;  pre-activation = xhat * gamma + beta = x * kg + kc   (saved statistics / parameters: written
      // long before this kernel, safe to read ahead of pdl_wait's successor ordering)
      const float m0 = p.bnb_save[2 * lane], m1 = p.bnb_save[2 * lane + 1];
      const float r0 = p.bnb_save[64 + 2 * lane], r1 = p.bnb_save[64 + 2 * lane + 1];
      const float g0 = p.bnb_gamma[2 * lane], g1 = p.bnb_gamma[2 * lane + 1];
      kx0 = r0; kx1 = r1; kb0 = -m0 * r0; kb1 = -m1 * r1;
      kg0 = r0 * g0; kg1 = r1 * g1;
      kc0 = p.bnb_beta[2 * lane] - m0 * r0 * g0; kc1 = p.bnb_beta[2 * lane + 1] - m1 * r1 * g1;
    }
    // pixel index of staged row (16 ew + i) of a tile = row_base(tile) + (halo ? (i >> 3) * W + (i & 7) : i)
    auto row_base = [&](int tile) -> long long {
      if (p.halo) {
        int n0 = tile >> p.lg_tpi;
        int rr = tile & (p.tiles_per_img - 1);
        int ty = rr >> p.lg_tx, tx = rr & (p.tiles_x - 1);
        return (long long)((n0 * p.H + ty * 16 + ew * 2) * p.W + tx * 8);
      }
      return (long long)tile * TC_BM + ew * 16;
    };
    const int rstep = p.halo ? p.W - 8 : 0;                        // extra pixels skipped after 8 rows of the staged tile
    uint32_t xq[(FUSE == 2 || FUSE == 3) ? 16 : 1];                               // BatchNorm input / residual input of this tile (channels 2l, 2l+1)
    auto load_xq = [&](long long rb) {
      const uint32_t* xb = reinterpret_cast<const uint32_t*>((FUSE == 3 ? p.gate_x : p.bnb_x) + rb * 64) + lane;
#pragma unroll
      for (int i = 0; i < ((FUSE == 2 || FUSE == 3) ? 16 : 1); ++i) {
        const int off = i + (i >> 3) * rstep;
        xq[i] = rb + off < p.M_total ? __ldg(xb + off * 32) : 0u;
      }
    };
    int it = 0;
    for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      if (p.dbg && blockIdx.x == 0 && warp == 2 && lane == 0) p.dbg[it * 8 + 3] = clock64();
      long long m = (long long)tile * TC_BM + row;                 // (M_total = B*H*W fits an int)
      if (p.halo) {
        int n0 = tile >> p.lg_tpi;
        int r = tile & (p.tiles_per_img - 1);
        int ty = r >> p.lg_tx, tx = r & (p.tiles_x - 1);
        m = (long long)((n0 * p.H + ty * 16 + (row >> 3)) * p.W + tx * 8 + (row & 7));
      }
      const bool valid = m < p.M_total;
      const long long rbase = row_base(tile);
      if (FUSE == 2) load_xq(rbase);                               // BatchNorm input rows: fetched while the MMAs still run
      mbar_wait(BAR(2 * S + 1 + buf), use & 1);
      tc_fence_after();
      if (p.dbg && blockIdx.x == 0 && warp == 2 && lane == 0) p.dbg[it * 8 + 4] = clock64();
      const int b = valid ? ((int)m >> p.lg_hw) : 0;
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * p.Npad);
      const float* scale_row = p.out_scale ? p.out_scale + (long long)b * p.N : nullptr;
      if (FUSE != 0 || p.tma_store) {
        // ---- TMEM -> registers (bias, Dropout2d scale, bf16 pack), release the accumulator, stage in smem, TMA store ----
        constexpr int NCH = (FUSE == 1 || FUSE == 2 || FUSE == 4) ? 1 : 2;       // fused reductions: N = 64, one chunk per thread
        uint4 packed[NCH][4];
#pragma unroll
        for (int nch = 0; nch < NCH; ++nch) {                      // N <= 128 on this path: at most two chunks per thread
          const int c0 = 32 * half + 64 * nch;
          if (c0 >= p.Npad) break;
          uint32_t r[32];
          tmem_ld32_nowait(taddr + (uint32_t)c0, r);
          tmem_wait_ld();
          float f[32];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 b4 = *reinterpret_cast<const float4*>(sbias + c0 + 4 * q);
            if (FUSE == 4) {
              const float4 s4 = *reinterpret_cast<const float4*>(sred + c0 + 4 * q);
              const int fact = ACT >= 0 ? ACT : p.fold_act;
              f[4 * q] = act_fwd_t<true>(fmaf(__uint_as_float(r[4 * q]), s4.x, b4.x), fact);
              f[4 * q + 1] = act_fwd_t<true>(fmaf(__uint_as_float(r[4 * q + 1]), s4.y, b4.y), fact);
              f[4 * q + 2] = act_fwd_t<true>(fmaf(__uint_as_float(r[4 * q + 2]), s4.z, b4.z), fact);
              f[4 * q + 3] = act_fwd_t<true>(fmaf(__uint_as_float(r[4 * q + 3]), s4.w, b4.w), fact);
              continue;
            }
            f[4 * q] = __uint_as_float(r[4 * q]) + b4.x; f[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + b4.y;
            f[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + b4.z; f[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + b4.w;
            if (scale_row) {
              const float4 s4 = __ldg(reinterpret_cast<const float4*>(scale_row + c0 + 4 * q));
              f[4 * q] *= s4.x; f[4 * q + 1] *= s4.y; f[4 * q + 2] *= s4.z; f[4 * q + 3] *= s4.w;
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&packed[nch][q]);
#pragma unroll
            for (int e = 0; e < 4; ++e) h2[e] = __floats2bfloat162_rn(f[8 * q + 2 * e], f[8 * q + 2 * e + 1]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(2 * S + 3 + buf));          // accumulator free again: next-but-one tile may start
        if (FUSE == 3) load_xq(rbase);                               // residual input rows (in flight across the staging barriers)
        // the previous tile's TMA store must have finished reading the staging buffer
        if (threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
        for (int nch = 0; nch < NCH; ++nch) {
          const int c0 = 32 * half + 64 * nch;
          if (c0 >= p.Npad) break;
          uint8_t* blk = sOut + (c0 >> 6) * TC_STAGE_BYTES + row * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int chunk = ((c0 & 63) >> 3) + q;
            *reinterpret_cast<uint4*>(blk + ((chunk ^ (row & 7)) << 4)) = packed[nch][q];
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (threadIdx.x == 64) {
          int c1, c2, c3;
          if (p.halo) {
            int n0 = tile >> p.lg_tpi;
            int r2 = tile & (p.tiles_per_img - 1);
            c3 = n0; c2 = (r2 >> p.lg_tx) * 16; c1 = (r2 & (p.tiles_x - 1)) * 8;
          } else {
            int p0 = tile * TC_BM;
            c3 = p0 >> p.lg_hw;
            int rem = p0 & (hw - 1);
            c2 = rem >> p.lg_w; c1 = rem & (p.W - 1);
          }
          for (int j = 0; j < p.Npad / 64 && !(FUSE == 3 && p.gate_skip_h); ++j) {
            const bool second = p.y2 != nullptr && j * 64 >= p.nsplit;
            tma_store_4d(second ? &tmY2 : &tmY, smem_u32(sOut + j * TC_STAGE_BYTES), second ? j * 64 - p.nsplit : j * 64, c1, c2, c3);
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (FUSE == 3) {
          // gate pass over the staged h tile (a = block 0, gate = block 1; values as stored): out -> third staging block
          const int nrows = p.halo ? 128 : (int)min((long long)128, p.M_total - (long long)tile * TC_BM);
          uint8_t* sGate = sOut + 2 * TC_STAGE_BYTES;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int r = ew * 16 + i;
            const int pos = r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + (lane & 3) * 4;
            const uint32_t ua = *reinterpret_cast<const uint32_t*>(sOut + pos);
            const uint32_t ug = *reinterpret_cast<const uint32_t*>(sOut + TC_STAGE_BYTES + pos);
            const float a0 = __uint_as_float(ua << 16), a1 = __uint_as_float(ua & 0xFFFF0000u);
            const float s0 = __uint_as_float(ug << 16), s1 = __uint_as_float(ug & 0xFFFF0000u);
            const float x0 = __uint_as_float(xq[i] << 16), x1 = __uint_as_float(xq[i] & 0xFFFF0000u);
            const float o0 = fmaf(act_fwd_t<true>(a0, ACT >= 0 ? ACT : p.gate_act), sigmoid_tanh_approx(s0), x0);
            const float o1 = fmaf(act_fwd_t<true>(a1, ACT >= 0 ? ACT : p.gate_act), sigmoid_tanh_approx(s1), x1);
            const __nv_bfloat162 ob = __floats2bfloat162_rn(o0, o1);
            const uint32_t uo = *reinterpret_cast<const uint32_t*>(&ob);
            *reinterpret_cast<uint32_t*>(sGate + pos) = uo;
            if (r < nrows) {                                          // statistics of the output as stored
              const float q0 = __uint_as_float(uo << 16), q1 = __uint_as_float(uo & 0xFFFF0000u);
              ra0 += q0; ra1 += q1;
              rb0 = fmaf(q0, q0, rb0); rb1 = fmaf(q1, q1, rb1);
            }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (threadIdx.x == 64) {
            int c1, c2, c3;
            if (p.halo) {
              int n0 = tile >> p.lg_tpi;
              int r2 = tile & (p.tiles_per_img - 1);
              c3 = n0; c2 = (r2 >> p.lg_tx) * 16; c1 = (r2 & (p.tiles_x - 1)) * 8;
            } else {
              int p0 = tile * TC_BM;
              c3 = p0 >> p.lg_hw;
              int rem = p0 & (hw - 1);
              c2 = rem >> p.lg_w; c1 = rem & (p.W - 1);
            }
            tma_store_4d(&tmY2, smem_u32(sGate), 0, c1, c2, c3);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        } else if (FUSE == 1 || FUSE == 2) {
          // second pass over the staged tile (values as stored, bf16-rounded); the TMA store only reads it concurrently
          const int nrows = p.halo ? 128 : (int)min((long long)128, p.M_total - (long long)tile * TC_BM);   // rows past the end contribute nothing
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int r = ew * 16 + i;
            const bool rv = r < nrows;
            const uint32_t u = *reinterpret_cast<const uint32_t*>(sOut + r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + (lane & 3) * 4);
            const float y0 = rv ? __uint_as_float(u << 16) : 0.f, y1 = rv ? __uint_as_float(u & 0xFFFF0000u) : 0.f;
            if (FUSE == 1) {
              ra0 += y0; ra1 += y1;
              rb0 = fmaf(y0, y0, rb0); rb1 = fmaf(y1, y1, rb1);
            } else {
              // g = dy * act'(xhat * gamma + beta); accumulate sum(g) and sum(g * xhat) per channel
              const float x0 = __uint_as_float(xq[i] << 16), x1 = __uint_as_float(xq[i] & 0xFFFF0000u);
              const float h0 = fmaf(x0, kx0, kb0), h1 = fmaf(x1, kx1, kb1);
              const float t0 = fmaf(x0, kg0, kc0), t1 = fmaf(x1, kg1, kc1);
              const float g0 = y0 * act_bwd_t<true>(t0, ACT >= 0 ? ACT : p.bnb_act);
              const float g1 = y1 * act_bwd_t<true>(t1, ACT >= 0 ? ACT : p.bnb_act);
              ra0 += g0; ra1 += g1;
              rb0 = fmaf(g0, h0, rb0); rb1 = fmaf(g1, h1, rb1);
            }
          }
        }
        if (p.dbg && blockIdx.x == 0 && warp == 2 && lane == 0) p.dbg[it * 8 + 5] = clock64();
        continue;
      }
      for (int c0 = 32 * half; c0 < p.Npad; c0 += 64) {
        uint32_t r[32];
        const bool two = c0 + 32 <= p.Npad;
        if (two) tmem_ld32_nowait(taddr + (uint32_t)c0, r);      // warp-collective: all lanes participate
        else tmem_ld16_nowait(taddr + (uint32_t)c0, r);
        tmem_wait_ld();
        if (!valid) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c = c0 + 16 * h;
          if ((h == 1 && !two) || c >= p.N) break;
          const bool second = p.y2 != nullptr && c >= p.nsplit;
          const int ncols = p.y2 ? (second ? p.N - p.nsplit : p.nsplit) : p.N;
          const int cc = second ? c - p.nsplit : c;
          char* base = (char*)(second ? p.y2 : p.y);
          const int esz = p.out_f32 ? 4 : 2;
          void* out_row = base + (size_t)m * ncols * esz;
          const void* res_row = (p.res && !p.y2) ? (const char*)p.res + (size_t)m * ncols * esz : nullptr;
          const int nvalid = min(16, ncols - cc);
          if (p.out_f32) epilogue16<true>(r + 16 * h, sbias, scale_row, res_row, out_row, c, cc, nvalid, ncols, p.N);
          else epilogue16<false>(r + 16 * h, sbias, scale_row, res_row, out_row, c, cc, nvalid, ncols, p.N);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (p.dbg && blockIdx.x == 0 && warp == 2 && lane == 0) p.dbg[it * 8 + 5] = clock64();
      if (lane == 0) mbar_arrive(BAR(2 * S + 3 + buf));
    }
    if (FUSE != 0 && FUSE != 4) {
      // combine the eight row groups per channel: one double atomic per channel and statistic per CTA
      sred[(0 * 8 + ew) * 64 + 2 * lane] = ra0; sred[(0 * 8 + ew) * 64 + 2 * lane + 1] = ra1;
      sred[(1 * 8 + ew) * 64 + 2 * lane] = rb0; sred[(1 * 8 + ew) * 64 + 2 * lane + 1] = rb1;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const int t = threadIdx.x - 64;                              // 0..127 -> (statistic, channel)
      if (t < 128) {
        const int st = t >> 6, c = t & 63;
        float sum = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) sum += sred[(st * 8 + e) * 64 + c];
        double* acc = (FUSE == 2 ? p.bnb_acc : p.stats_acc);
        if (acc) atomicAdd(acc + (blockIdx.x & 7) * 128 + st * 64 + c, (double)sum);   // 8-way striped (see elementwise.cu)
      }
    }
  }
  if (p.tma_store && threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

long long* g_tc_dbg = nullptr;

int lg2_ceil(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}
void set_shifts(TcParams& p) {
  p.lg_w = lg2_ceil(p.W); p.lg_hw = lg2_ceil(p.H * p.W);
  p.lg_tx = lg2_ceil(p.tiles_x > 0 ? p.tiles_x : 1); p.lg_tpi = lg2_ceil(p.tiles_per_img > 0 ? p.tiles_per_img : 1);
}

int pow2_floor_le(int v, int cap) {
  int r = 1;
  while (r * 2 <= v && r * 2 <= cap) r *= 2;
  return r;
}

constexpr int TC_MAX_SMEM = 227 * 1024 - 1024 /*align*/ - 8192 /*barriers, bias, BatchNorm table, reduction scratch*/;

// Weight placement of a lvae_conv2d_tc launch, from the shape alone: 0 = rejected, 1 = resident, 2 = streamed.  Resident
// when the packed weights leave room for two 16 KB activation stages next to the largest output staging the shape can
// use (the TMA-store epilogue's, bf16 output with N = 64 / 128); every shape a 64-filter model launches is resident.
int tc_weight_plan(int Cin, int N, int ksize, int inputs, int H, int W, int out_f32) {
  if (!(Cin % 64 == 0 && Cin >= 64 && Cin <= 256 && (ksize == 1 || ksize == 3) && N >= 1 && N <= 256)) return 0;
  if (!(H > 0 && W > 0 && (W & (W - 1)) == 0 && (H & (H - 1)) == 0 && W <= 128)) return 0;
  const int n_kb = ksize * ksize * inputs * (Cin / 64);
  if (n_kb > TC_MAX_KB) return 0;
  const int Npad = (N + 15) / 16 * 16;
  const int out_stage = (!out_f32 && N % 64 == 0 && N <= 128) ? Npad / 64 * TC_STAGE_BYTES : 0;
  const int wbytes = ((n_kb * Npad * 128) + 1023) & ~1023;
  if ((TC_MAX_SMEM - wbytes - out_stage) / TC_STAGE_BYTES >= 2) return 1;
  if ((TC_MAX_SMEM - out_stage) / (TC_STAGE_BYTES + Npad * 128) >= 2) return 2;
  return 0;
}

}  // namespace

// x, x2: (B,H,W,Cin) bf16 NHWC, Cin a multiple of 64 (x2 optional: second input of a merge conv).
// wp: bf16 [n_kb][Npad][64] (k-block = tap-major, then input): see lvae_pack_weights modes 2/3.
// taps: ksize*ksize offsets; flip = 1 negates them (data gradient).  y: (B,H,W,N) bf16 or fp32;
// y2 != NULL splits the output columns at nsplit into two tensors (dgrad of a merge conv).
struct LvaeConvFuse {
  double* stats_acc;
  const void* bnb_x;
  const float* bnb_save;
  const float* bnb_gamma;
  const float* bnb_beta;
  double* bnb_acc;
  int bnb_act;
  const void* gate_x;
  void* gate_out;
  int gate_act;
  int gate_skip_h;
  const float* fold_gamma;
  const float* fold_beta;
  const float* fold_mean;
  const float* fold_var;
  float fold_eps;
  int fold_act;
  const float* pre_gamma;
  const float* pre_beta;
  const float* pre_mean;
  const float* pre_var;
  float pre_eps;
};

LVAE_API int lvae_conv2d_tc_ex(const void* x, const void* x2, const void* wp, const float* bias, const float* out_scale,
                               const void* res, void* y, void* y2, int nsplit, int B, int H, int W, int Cin, int N,
                               int ksize, int flip, int out_f32, const LvaeConvFuse* fuse, cudaStream_t stream);

LVAE_API int lvae_conv2d_tc(const void* x, const void* x2, const void* wp, const float* bias, const float* out_scale,
                            const void* res, void* y, void* y2, int nsplit, int B, int H, int W, int Cin, int N,
                            int ksize, int flip, int out_f32, cudaStream_t stream) {
  return lvae_conv2d_tc_ex(x, x2, wp, bias, out_scale, res, y, y2, nsplit, B, H, W, Cin, N, ksize, flip, out_f32, nullptr, stream);
}

// fuse (host struct, may be NULL): per-channel reductions computed in the epilogue, see LvaeConvFuse in include/lvae_b200.h.
// Only on the TMA-store path (bf16 output, N == 64, no residual); anything else is rejected.
LVAE_API int lvae_conv2d_tc_ex(const void* x, const void* x2, const void* wp, const float* bias, const float* out_scale,
                               const void* res, void* y, void* y2, int nsplit, int B, int H, int W, int Cin, int N,
                               int ksize, int flip, int out_f32, const LvaeConvFuse* fuse, cudaStream_t stream) {
  LVAE_REQUIRE(x && wp && (y || (fuse && fuse->gate_out && fuse->gate_skip_h)), "conv2d_tc: null pointer");
  LVAE_REQUIRE(Cin % 64 == 0 && Cin >= 64 && Cin <= 256 && (ksize == 1 || ksize == 3),
               "conv2d_tc: needs a multiple of 64 input channels per tensor and a 1x1 or 3x3 kernel");
  LVAE_REQUIRE(N >= 1 && N <= 256, "conv2d_tc: 1 <= N <= 256");
  LVAE_REQUIRE((W & (W - 1)) == 0 && (H & (H - 1)) == 0 && W <= 128, "conv2d_tc: H and W must be powers of two (W <= 128)");
  LVAE_REQUIRE(!(y2 && res), "conv2d_tc: residual and split output are exclusive");
  LVAE_REQUIRE(!y2 || (nsplit % 16 == 0 && nsplit > 0 && nsplit < N), "conv2d_tc: nsplit must be a multiple of 16 inside (0, N)");
  TcParams p{};
  p.bias = bias; p.out_scale = out_scale; p.res = res; p.y = y; p.y2 = y2; p.nsplit = nsplit;
  p.M_total = B * H * W; p.H = H; p.W = W; p.N = N; p.Npad = (N + 15) / 16 * 16;
  p.out_f32 = out_f32;
  p.dbg = g_tc_dbg;
  if (fuse) {
    p.stats_acc = fuse->stats_acc;
    p.bnb_x = (const __nv_bfloat16*)fuse->bnb_x; p.bnb_save = fuse->bnb_save; p.bnb_gamma = fuse->bnb_gamma;
    p.bnb_beta = fuse->bnb_beta; p.bnb_acc = fuse->bnb_acc; p.bnb_act = fuse->bnb_act;
    LVAE_REQUIRE(!p.bnb_acc || (p.bnb_x && p.bnb_save && p.bnb_gamma && p.bnb_beta), "conv2d_tc: incomplete BatchNorm-backward fusion arguments");
    LVAE_REQUIRE(!(p.bnb_acc && p.stats_acc), "conv2d_tc: output statistics and BatchNorm-backward sums cannot be fused into the same launch");
    if (fuse->gate_out) {
      LVAE_REQUIRE(fuse->gate_x && N == 128 && !y2 && !res && !out_f32 && !p.bnb_acc,
                   "conv2d_tc: the gated-residual epilogue needs N == 128, bf16 output, no residual / split");
      p.gate_x = (const __nv_bfloat16*)fuse->gate_x; p.gate_act = fuse->gate_act; p.gate_skip_h = fuse->gate_skip_h;
    }
    if (fuse->fold_gamma) {
      LVAE_REQUIRE(fuse->fold_beta && fuse->fold_mean && fuse->fold_var && N == 64 && !y2 && !res && !out_f32 && !out_scale &&
                   !p.bnb_acc && !p.stats_acc && !fuse->gate_out,
                   "conv2d_tc: the folded eval-mode BatchNorm needs N == 64, bf16 output and no other epilogue fusion");
      p.fold_gamma = fuse->fold_gamma; p.fold_beta = fuse->fold_beta; p.fold_mean = fuse->fold_mean; p.fold_var = fuse->fold_var;
      p.fold_eps = fuse->fold_eps; p.fold_act = fuse->fold_act;
      if (fuse->pre_gamma) {
        LVAE_REQUIRE(fuse->pre_beta && fuse->pre_mean && fuse->pre_var && !x2 && Cin == 64 && ksize == 3 && W % 8 == 0 && H % 16 == 0,
                     "conv2d_tc: the operand-path BatchNorm needs a single 64-channel input, a 3x3 kernel and halo tiles (W % 8 == 0, H % 16 == 0)");
        p.pre_gamma = fuse->pre_gamma; p.pre_beta = fuse->pre_beta; p.pre_mean = fuse->pre_mean; p.pre_var = fuse->pre_var;
        p.pre_eps = fuse->pre_eps;
      }
    }
  }
  const int inputs = x2 ? 2 : 1;
  const int taps = ksize * ksize;
  const int cblocks = Cin / 64;
  p.n_kb = taps * inputs * cblocks;
  LVAE_REQUIRE(p.n_kb <= TC_MAX_KB, "conv2d_tc: too many k-blocks");
  const int wplan = tc_weight_plan(Cin, N, ksize, inputs, H, W, out_f32);
  LVAE_REQUIRE(wplan != 0, "conv2d_tc: weights leave no room for the activation pipeline");
  const bool stream_w = wplan == 2;
  LVAE_REQUIRE(!stream_w || !fuse, "conv2d_tc: fused epilogues need resident weights");
  int kb = 0;
  for (int t = 0; t < taps; ++t) {
    int ky = t / ksize, kx = t % ksize;
    int oy = ky - ksize / 2, ox = kx - ksize / 2;
    if (flip) { oy = -oy; ox = -ox; }
    for (int s = 0; s < inputs; ++s)
      for (int c = 0; c < cblocks; ++c, ++kb) {
        p.dy[kb] = (int8_t)oy; p.dx[kb] = (int8_t)ox; p.src[kb] = (int8_t)s; p.coff[kb] = (int8_t)c;
      }
  }
  p.bw = W;                                  // full image rows (W <= 128)
  p.bh = pow2_floor_le(H, TC_BM / p.bw);
  p.bn = TC_BM / (p.bw * p.bh);
  p.tmem_cols = 32;
  while (p.tmem_cols < 2 * p.Npad) p.tmem_cols *= 2;
  LVAE_REQUIRE(p.tmem_cols <= 512, "conv2d_tc: accumulator does not fit TMEM");
  const int max_smem = TC_MAX_SMEM;
  const int wbytes = stream_w ? 0 : ((p.n_kb * p.Npad * 128) + 1023) & ~1023;
  p.tma_store = (!out_f32 && N % 64 == 0 && N <= 128 && !res && (!y2 || nsplit % 64 == 0)) ? 1 : 0;
  const int out_stage = p.tma_store ? (p.Npad / 64 + (p.gate_x ? 1 : 0)) * TC_STAGE_BYTES : 0;
  LVAE_REQUIRE(!p.gate_x || p.tma_store, "conv2d_tc: the gated-residual epilogue needs the TMA-store path");
  LVAE_REQUIRE(!p.fold_gamma || p.tma_store, "conv2d_tc: the folded BatchNorm epilogue needs the TMA-store path");
  LVAE_REQUIRE(!(p.stats_acc || p.bnb_acc) || (p.tma_store && (N == 64 || p.gate_x) && !y2),
               "conv2d_tc: fused reductions need the TMA-store path (bf16 output, N == 64, no residual, no split)");
  p.halo = (!stream_w && ksize == 3 && !x2 && Cin == 64 && W % 8 == 0 && H % 16 == 0 &&
            (max_smem - wbytes - out_stage) / (18 * 16 * 128) >= 2) ? 1 : 0;
  p.stage_bytes = 18 * 16 * 128;
  p.tiles_x = W / 8;
  p.tiles_per_img = (W / 8) * (H / 16);
  set_shifts(p);
  LVAE_REQUIRE(!p.pre_gamma || p.halo, "conv2d_tc: the operand-path BatchNorm needs the halo-tile path (no shared memory left for two halo stages)");
  const int a_stage = p.halo ? p.stage_bytes : (stream_w ? TC_STAGE_BYTES + p.Npad * 128 : TC_STAGE_BYTES);
  int stages = (max_smem - wbytes - out_stage) / a_stage;
  if (stages > 8) stages = 8;
  LVAE_REQUIRE(stages >= 2, "conv2d_tc: weights leave no room for the activation pipeline");
  p.n_stages = stages;
  const size_t smem = 1024 + (size_t)wbytes + (size_t)stages * a_stage + out_stage + 8192;

  EncodeTiledFn enc = get_encode();
  if (!enc) {
    lvae_set_error("conv2d_tc: cuTensorMapEncodeTiled unavailable");
    return LVAE_ERR_CUDA;
  }
  CUtensorMap tmA0, tmA1, tmW, tmY, tmY2;
  memset(&tmY, 0, sizeof(tmY));
  memset(&tmY2, 0, sizeof(tmY2));
  if (p.tma_store) {
    // output maps: same pixel box as the activation tiles (8 x 16 pixels in halo mode), 64 channels per box
    void* const gate_out = (fuse && fuse->gate_out) ? fuse->gate_out : nullptr;
    for (int which = (gate_out && p.gate_skip_h) ? 1 : 0; which < ((y2 || gate_out) ? 2 : 1); ++which) {
      const int ncols = gate_out ? (which ? 64 : N) : (y2 ? (which ? N - nsplit : nsplit) : N);
      cuuint64_t gdim[4] = {(cuuint64_t)ncols, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
      cuuint64_t gstr[3] = {(cuuint64_t)ncols * 2, (cuuint64_t)W * ncols * 2, (cuuint64_t)H * W * ncols * 2};
      cuuint32_t box[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bn};
      if (p.halo) { box[1] = 8; box[2] = 16; box[3] = 1; }
      cuuint32_t estr[4] = {1, 1, 1, 1};
      CUresult r = enc(which ? &tmY2 : &tmY, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, which ? (gate_out ? gate_out : y2) : y, gdim, gstr, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc: tensor map (y) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
    }
  }
  {
    cuuint64_t gdim[4] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t gstr[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bn};
    if (p.halo) { box[1] = 16; box[2] = 18; box[3] = 1; }
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tmA0, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)x, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc: tensor map (x) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
    r = enc(&tmA1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)(x2 ? x2 : x), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc: tensor map (x2) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
    cuuint64_t wdim[2] = {64, (cuuint64_t)p.n_kb * p.Npad};
    cuuint64_t wstr[1] = {128};
    cuuint32_t wbox[2] = {64, (cuuint32_t)p.Npad};
    cuuint32_t westr[2] = {1, 1};
    r = enc(&tmW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)wp, wdim, wstr, wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc: tensor map (w) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
  }
  static size_t attr_smem = 0;
  const int cap = 227 * 1024;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<2, ACT_ELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<3, ACT_ELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<4, ACT_ELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<0, -1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e != cudaSuccess) { lvae_set_error("conv2d_tc: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
    attr_smem = 227 * 1024;
  }
  const int n_tiles = p.halo ? B * p.tiles_per_img : (p.M_total + TC_BM - 1) / TC_BM;
  const int grid = n_tiles < lvae_num_sms() ? n_tiles : lvae_num_sms();
  if (p.fold_gamma && p.fold_act == ACT_ELU) lvae_launch(conv_tc_kernel<4, ACT_ELU>, grid, TC_THREADS + 160, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.fold_gamma) lvae_launch(conv_tc_kernel<4>, grid, TC_THREADS + 160, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.gate_x && p.gate_act == ACT_ELU) lvae_launch(conv_tc_kernel<3, ACT_ELU>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.gate_x) lvae_launch(conv_tc_kernel<3>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.stats_acc) lvae_launch(conv_tc_kernel<1>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.bnb_acc && p.bnb_act == ACT_ELU) lvae_launch(conv_tc_kernel<2, ACT_ELU>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (p.bnb_acc) lvae_launch(conv_tc_kernel<2>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else if (stream_w) lvae_launch(conv_tc_kernel<0, -1, true>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  else lvae_launch(conv_tc_kernel<0>, grid, TC_THREADS, smem, stream, tmA0, tmA1, tmW, tmY, tmY2, p);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("conv2d_tc");
  return LVAE_OK;
}

// Pure-host query: how lvae_conv2d_tc would hold the weights of this shape (0 rejected, 1 resident, 2 streamed).
LVAE_API int lvae_conv2d_tc_plan(int Cin, int N, int ksize, int two_inputs, int H, int W, int out_f32) {
  return tc_weight_plan(Cin, N, ksize, two_inputs ? 2 : 1, H, W, out_f32);
}

// Stride-2 3x3 convolutions of 64 -> 64 channels on the same kernel (bf16 in / out, TMA-store epilogue).
//   kind 0 "strided gather":  y[b,oy,ox,:] = bias + sum_t x[b, 2oy-1+ky, 2ox-1+kx, :] . Wt         x (B,2Ho,2Wo,64) -> y (B,Ho,Wo,N)
//           = Conv2d(stride 2, pad 1) forward, and the input gradient of ConvTranspose2d(stride 2, pad 1, output_padding 1)
//   kind 1 "transposed":      y[b,2iy-1+ky,2ix-1+kx,:] += x[b,iy,ix,:] . Wt                         x (B,Hi,Wi,64) -> y (B,2Hi,2Wi,N)
//           = ConvTranspose2d forward, and the input gradient of Conv2d(stride 2, pad 1).  Run as four launches, one per
//           output parity class (oy&1, ox&1): class (py,px) is a stride-1 convolution over the INPUT grid with the taps
//           {ky : ky = 1 if py == 0 else 0 or 2} x {kx likewise} (input offset +1 for k = 0, else 0), written through a
//           tensor map whose strides step two output pixels -- 1 + 2 + 2 + 4 = 9 tap-GEMMs in total, no zero work.
// wp: nine packed [Npad][64] weight blocks, block t = tap (ky,kx) = (t/3, t%3), rows = output channel, K = input channel
// (lvae_pack_weights mode 2 for Conv2d forward / ConvTranspose2d dgrad with the transposed-conv weight read as (O=ci, I=co);
// mode 3 for the other two).  Hg, Wg: the smaller of the two grids (Ho,Wo for kind 0; Hi,Wi for kind 1), powers of two.
LVAE_API int lvae_conv2d_tc_s2(const void* x, const void* wp, const float* bias, const float* out_scale, void* y, int B,
                               int Hg, int Wg, int N, int kind, cudaStream_t stream) {
  LVAE_REQUIRE(x && wp && y, "conv2d_tc_s2: null pointer");
  LVAE_REQUIRE(N == 64, "conv2d_tc_s2: 64 output channels");
  LVAE_REQUIRE((Wg & (Wg - 1)) == 0 && (Hg & (Hg - 1)) == 0 && Wg >= 1 && Wg <= 64 && Hg >= 1, "conv2d_tc_s2: grid must be powers of two, W <= 64");
  LVAE_REQUIRE(kind == 0 || kind == 1, "conv2d_tc_s2: bad kind");
  EncodeTiledFn enc = get_encode();
  if (!enc) { lvae_set_error("conv2d_tc_s2: cuTensorMapEncodeTiled unavailable"); return LVAE_ERR_CUDA; }
  const int Cin = 64, Hb = 2 * Hg, Wb = 2 * Wg;               // the bigger grid
  static size_t attr_smem = 0;
  if (!attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
    if (e != cudaSuccess) { lvae_set_error("conv2d_tc_s2: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
    attr_smem = 227 * 1024;
  }
  for (int cls = 0; cls < (kind == 0 ? 1 : 4); ++cls) {
    TcParams p{};
    p.bias = bias; p.out_scale = out_scale; p.y = y;
    p.M_total = B * Hg * Wg; p.H = Hg; p.W = Wg; p.N = N; p.Npad = 64;
    p.dbg = nullptr;
    p.use_wblk = 1;
    p.in_stride = kind == 0 ? 2 : 1;
    int kb = 0;
    const int py = cls >> 1, px = cls & 1;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        int oy, ox;
        if (kind == 0) { oy = ky - 1; ox = kx - 1; }
        else {
          if ((py == 0) != (ky == 1) || (px == 0) != (kx == 1)) continue;       // this tap never reaches the class
          oy = ky == 0 ? 1 : 0; ox = kx == 0 ? 1 : 0;
        }
        p.dy[kb] = (int8_t)oy; p.dx[kb] = (int8_t)ox; p.src[kb] = 0; p.coff[kb] = 0; p.wblk[kb] = (int8_t)(ky * 3 + kx);
        ++kb;
      }
    p.n_kb = kb;
    p.bw = Wg;
    p.bh = pow2_floor_le(Hg, TC_BM / p.bw);
    p.bn = TC_BM / (p.bw * p.bh);
    p.tmem_cols = 128;
    p.tma_store = 1;
    p.halo = 0;
    p.stage_bytes = TC_STAGE_BYTES;
    const int wbytes = ((p.n_kb * p.Npad * 128) + 1023) & ~1023;
    p.n_stages = 8;
    const size_t smem = 1024 + (size_t)wbytes + (size_t)p.n_stages * TC_STAGE_BYTES + TC_STAGE_BYTES + 8192;
    CUtensorMap tmA, tmW, tmY, tmY2;
    memset(&tmY2, 0, sizeof(tmY2));
    {
      // input: for kind 0 the (bigger) input grid is traversed with element stride 2, so a box of 2*bw x 2*bh input
      // pixels delivers the bw x bh pixels one filter tap needs for a tile of output pixels
      const int Hi = kind == 0 ? Hb : Hg, Wi = kind == 0 ? Wb : Wg, st = kind == 0 ? 2 : 1;
      cuuint64_t gdim[4] = {(cuuint64_t)Cin, (cuuint64_t)Wi, (cuuint64_t)Hi, (cuuint64_t)B};
      cuuint64_t gstr[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Wi * Cin * 2, (cuuint64_t)Hi * Wi * Cin * 2};
      cuuint32_t box[4] = {64, (cuuint32_t)(p.bw * st), (cuuint32_t)(p.bh * st), (cuuint32_t)p.bn};
      cuuint32_t estr[4] = {1, (cuuint32_t)st, (cuuint32_t)st, 1};
      CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)x, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc_s2: tensor map (x) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
      // output: kind 0 the plain (B,Hg,Wg,N) tensor; kind 1 the parity class (py,px) of the (B,2Hg,2Wg,N) tensor
      const size_t Wo = kind == 0 ? Wg : Wb, Ho = kind == 0 ? Hg : Hb, step = kind == 0 ? 1 : 2;
      char* ybase = (char*)y + (kind == 0 ? 0 : ((size_t)py * Wo + px) * N * 2);
      cuuint64_t odim[4] = {(cuuint64_t)N, (cuuint64_t)Wg, (cuuint64_t)Hg, (cuuint64_t)B};
      cuuint64_t ostr[3] = {(cuuint64_t)(step * N * 2), (cuuint64_t)(step * Wo * N * 2), (cuuint64_t)(Ho * Wo * N * 2)};
      cuuint32_t obox[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bn};
      cuuint32_t one[4] = {1, 1, 1, 1};
      r = enc(&tmY, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)ybase, odim, ostr, obox, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc_s2: tensor map (y) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
      cuuint64_t wdim[2] = {64, (cuuint64_t)9 * p.Npad};
      cuuint64_t wstr[1] = {128};
      cuuint32_t wbox[2] = {64, (cuuint32_t)p.Npad};
      cuuint32_t westr[2] = {1, 1};
      r = enc(&tmW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)wp, wdim, wstr, wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) { lvae_set_error("conv2d_tc_s2: tensor map (w) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
    }
    const int n_tiles = (p.M_total + TC_BM - 1) / TC_BM;
    const int grid = n_tiles < lvae_num_sms() ? n_tiles : lvae_num_sms();
    set_shifts(p);
    lvae_launch(conv_tc_kernel<0>, grid, TC_THREADS, smem, stream, tmA, tmA, tmW, tmY, tmY2, p);
    LVAE_COUNT_LAUNCH();
    LVAE_CHECK_LAUNCH("conv2d_tc_s2");
  }
  return LVAE_OK;
}

// profiling aid: device buffer (>= 8 * tiles-per-CTA int64) that CTA 0 of the following conv2d_tc launches fills with
// clock64 stamps per tile: [0] MMA thread ready, [1] operands landed, [2] MMAs issued, [3] epilogue waiting,
// [4] accumulator ready, [5] epilogue done, [6] producer got a free stage.  NULL switches it off.
LVAE_API void lvae_conv2d_tc_debug(long long* dev_buf) { g_tc_dbg = dev_buf; }
