// The tail of a gated residual block as ONE kernel (default since the round-2 A/B on the B200: 17.41 -> 16.71 ms per step):
//     c2  = (conv3x3(a2) + bias2) * mask2                      second 3x3 convolution of lib/nn.py:83-87 (+ its Dropout2d)
//     h   = conv1x1(c2) + bias_g        = [a | g], 128 channels   GateLayer2d's convolution, lib/nn.py:118
//     out = act(a) * sigmoid(g) + x                              gate and residual add, lib/nn.py:121-126,99
//     (+ per-channel sum / sum of squares of `out` for the next block's BatchNorm)
// The 1x1 gate convolution is tile-local: its A operand is exactly the bf16, 128B-swizzled tile that the 3x3 convolution's
// epilogue stages in shared memory for its TMA store, so the second GEMM (M = 128 pixels, N = 128, K = 64: four tcgen05.mma)
// reads it in place -- no second launch, no re-read of c2 from HBM / L2, no second prologue.  Per tile:
//     TMA -> smem -> 36 MMAs -> TMEM acc1 -> epilogue phase 1 (bias, mask, bf16, stage c2, TMA store) -> 4 MMAs on the staged
//     tile -> TMEM acc2 -> epilogue phase 2 (bias, stage h, TMA store; gate pass over the staged h; stage out, TMA store).
// The MMA warp issues the 3x3 MMAs of tile i+1 before the gate MMAs of tile i, so the tensor pipe stays busy while the
// epilogue warps stage tile i.  Same warp roles, descriptors, halo tiles and epilogue arithmetic as conv_tcgen05.cu
// (which keeps serving every other convolution).
#include "common.cuh"
#include <cuda.h>
#include <string.h>

namespace {

// warp 0 TMA, warp 1 MMA, warps 2 .. 2 + EW - 1 epilogue.  The ELU gate runs with EW = 16: four warps per TMEM lane quadrant,
// 16 accumulator columns per thread (any other activation: EW = 8).  The epilogue of this kernel is a serial chain per tile
// (c2 -> gate GEMM -> gate -> store) that the clock64 trace (profiles/trace_conv_gate.py) shows to be latency-bound, not
// issue-bound: with 8 warps (two per scheduler) a tile took ~4900 cycles at B = 1000 against ~2300 for its MMAs.
constexpr int CG_BM = 128;
constexpr int CG_TILE_BYTES = CG_BM * 64 * 2;      // 16 KB: one 128-pixel x 64-channel bf16 tile
constexpr int CG_HALO_BYTES = 18 * 16 * 128;       // 36 KB
constexpr int CG_TAPS = 9;

struct CgParams {
  const float* bias2;       // [64] or null
  const float* scale2;      // (B,64) Dropout2d mask of the 3x3 convolution, or null
  const float* bias_g;      // [128] or null
  const __nv_bfloat16* x_res;   // block input (M,64): residual
  double* stats_acc;        // 8-way striped (sum, sum of squares) of out, or null
  int M_total, H, W;
  int n_stages, halo, stage_bytes, tiles_x, tiles_per_img;
  int lg_w, lg_hw, lg_tx, lg_tpi;   // H, W (hence tiles_x, tiles_per_img) are powers of two: per-tile index arithmetic is shifts --
                            // the 64-bit m / hw and the tile divisions cost ~800 cycles per tile on the epilogue's critical path
  int bw, bh, bn;           // per-tap TMA box (non-halo): bw*bh*bn == 128
  int gate_act;
  int store_c2h;            // 1: c2 and h are stored (a backward pass will read them); 0: eval, only out leaves the SM
  long long* dbg;           // optional clock64 trace of CTA 0, 16 stamps per tile (lvae_conv_gate_tc_debug; normally null)
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
// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups sbo bytes apart
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr, uint32_t sbo_bytes = 1024) {
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
template <int N> __device__ __forceinline__ void tmem_ldN_nowait(uint32_t taddr, uint32_t* r) {
  if (N == 32) tmem_ld32_nowait(taddr, r);
  else tmem_ld16_nowait(taddr, r);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// N (16 / 32) accumulator columns [c0, c0 + N) of this thread's row: + bias, * Dropout2d scale, packed to N / 8 16-byte bf16 chunks
template <int N>
__device__ __forceinline__ void packN(const uint32_t* r, const float* sb, const float* scale_row, int c0, uint4* packed) {
  float f[N];
#pragma unroll
  for (int q = 0; q < N / 4; ++q) {
    const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + 4 * q);
    f[4 * q] = __uint_as_float(r[4 * q]) + b4.x; f[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + b4.y;
    f[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + b4.z; f[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + b4.w;
    if (scale_row) {
      const float4 s4 = __ldg(reinterpret_cast<const float4*>(scale_row + c0 + 4 * q));
      f[4 * q] *= s4.x; f[4 * q + 1] *= s4.y; f[4 * q + 2] *= s4.z; f[4 * q + 3] *= s4.w;
    }
  }
#pragma unroll
  for (int q = 0; q < N / 8; ++q) {
    __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&packed[q]);
#pragma unroll
    for (int e = 0; e < 4; ++e) h2[e] = __floats2bfloat162_rn(f[8 * q + 2 * e], f[8 * q + 2 * e + 1]);
  }
}

// ACT: the gate activation as a compile-time constant (ACT_ELU, the model default) or -1 = read p.gate_act.  A runtime switch
// inside the unrolled gate pass compiled to one jump table (LDC + BRX) per element: 34 indirect branches per tile-thread that
// also kept the 16 iterations from overlapping (ncu, B = 1000: 1950 instructions per tile-thread, IPC 0.35 per scheduler).
template <int ACT, int EW>
#define CG_STAMP(slot) do { if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[it * 16 + (slot)] = clock64(); } while (0)
__global__ void __launch_bounds__(64 + 32 * EW, 1)
conv_gate_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmWg, const __grid_constant__ CUtensorMap tmC2,
                    const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmOut, const CgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sW2 = smem;                                   // 9 x [64][64] bf16 = 72 KB
  uint8_t* sWg = sW2 + CG_TAPS * 64 * 128;               // [128][64] bf16 = 16 KB
  uint8_t* sA = sWg + 128 * 128;                         // n_stages x stage_bytes
  const int stage_bytes = p.halo ? CG_HALO_BYTES : CG_TILE_BYTES;
  uint8_t* sC2 = sA + p.n_stages * stage_bytes;          // staged c2 tile = A operand of the gate GEMM; later the staged out tile
  uint8_t* sH = sC2 + CG_TILE_BYTES;                     // staged h tile: [a | g], two 64-channel blocks
  uint64_t* bars = (uint64_t*)(sH + 2 * CG_TILE_BYTES);
  // barriers: [0..S) full, [S..2S) empty, 2S weights, 2S+1..2 acc1_full[2], 2S+3..4 acc1_empty[2], 2S+5..6 c2_staged[2],
  //           2S+7..8 acc2_full[2], 2S+9..10 acc2_empty[2]  (the second of each gate-side pair: eval mode with two epilogue groups)
  const int S = p.n_stages;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * S + 12);
  float* sbias = (float*)(bars + 32);                    // [0,64): bias2, [64,192): bias_g
  float* sred = sbias + 192;                             // 2 x 8 x 64 partial statistics
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const int B_W = 2 * S, B_A1F = 2 * S + 1, B_A1E = 2 * S + 3, B_C2 = 2 * S + 5, B_A2F = 2 * S + 7, B_A2E = 2 * S + 9;
  // Eval mode (nothing but `out` leaves the SM) with 16 epilogue warps: TWO GROUPS of eight warps take alternate tiles, each
  // with its own staging buffer, gate accumulator and barriers, so that two of the per-tile chains
  //   acc1 -> c2 staged -> gate GEMM -> gate -> out staged -> TMA store      (~4500 cycles, all dependent latencies)
  // are in flight against ~2300 cycles of MMAs per tile: the kernel becomes tensor-pipe-bound instead of chain-bound.
  const bool fast = !p.store_c2h && !p.stats_acc;
  const int G = (fast && EW == 16) ? 2 : 1;
  const uint32_t tmem_cols = G == 2 ? 512u : 256u;

  constexpr int CG_THREADS = 64 + 32 * EW;
  constexpr int CPT = 256 / EW;              // accumulator columns per epilogue thread and 64-column block (32 / 16)
  constexpr int RPW = 128 / EW;              // staged rows per epilogue warp in the channel-major gate pass (16 / 8)
  constexpr int NQ = CPT / 8;                // 16-byte bf16 chunks per thread and block
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gact = ACT >= 0 ? ACT : p.gate_act;
  const int n_tiles = p.halo ? (p.M_total / (p.H * p.W)) * p.tiles_per_img : (p.M_total + CG_BM - 1) / CG_BM;
  const int hw = p.H * p.W;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW2);
    prefetch_tmap(&tmWg);
    for (int i = 0; i < S; ++i) {
      mbar_init(BAR(i), 1);
      mbar_init(BAR(S + i), 1);
    }
    mbar_init(BAR(B_W), 1);
    mbar_init(BAR(B_A1F), 1);
    mbar_init(BAR(B_A1F + 1), 1);
    mbar_init(BAR(B_A1E), EW / G);     // one arrive per epilogue warp (of the group that owns the tile)
    mbar_init(BAR(B_A1E + 1), EW / G);
    for (int g = 0; g < 2; ++g) {
      mbar_init(BAR(B_C2 + g), 1);     // the group's elected thread, after the staging barrier
      mbar_init(BAR(B_A2F + g), 1);
      mbar_init(BAR(B_A2E + g), EW / G);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    __syncwarp();
    // both weight sets were packed many kernels ago: fetch them before waiting on the previous kernel (PDL prologue)
    if (elect_one()) {
      mbar_expect_tx(BAR(B_W), (uint32_t)(CG_TAPS * 64 * 128 + 128 * 128));
      for (int t = 0; t < CG_TAPS; ++t) tma_load_2d(smem_u32(sW2 + t * 64 * 128), &tmW2, BAR(B_W), 0, t * 64);
      tma_load_2d(smem_u32(sWg), &tmWg, BAR(B_W), 0, 0);
    }
    __syncwarp();
  }
  for (int i = threadIdx.x; i < 192; i += CG_THREADS)
    sbias[i] = i < 64 ? (p.bias2 ? p.bias2[i] : 0.f) : (p.bias_g ? p.bias_g[i - 64] : 0.f);
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;      // columns [0,64) / [64,128): acc1[0] / acc1[1]; [128,256): acc2[0]; [256,384): acc2[1]
  pdl_wait();
  pdl_launch();

  if (warp == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      if (p.halo) {
        const int n0 = tile / p.tiles_per_img;
        const int r = tile - n0 * p.tiles_per_img;
        const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
        mbar_wait(BAR(S + stage), phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(stage), (uint32_t)CG_HALO_BYTES);
          tma_load_4d(smem_u32(sA + stage * stage_bytes), &tmA, BAR(stage), 0, tx * 8 - 1, ty * 16 - 1, n0);
        }
        __syncwarp();
        if (++stage == S) { stage = 0; phase ^= 1; }
        continue;
      }
      const int p0 = tile * CG_BM;
      const int n0 = p0 / hw;
      const int rem = p0 - n0 * hw;
      const int h0 = rem / p.W;
      const int w0 = rem - h0 * p.W;
      for (int t = 0; t < CG_TAPS; ++t) {
        mbar_wait(BAR(S + stage), phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(stage), CG_TILE_BYTES);
          tma_load_4d(smem_u32(sA + stage * CG_TILE_BYTES), &tmA, BAR(stage), 0, w0 + (t % 3) - 1, h0 + (t / 3) - 1, n0);
        }
        __syncwarp();
        if (++stage == S) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc3 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(CG_BM >> 4) << 24);
    const uint32_t idescg = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(CG_BM >> 4) << 24);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    mbar_wait(BAR(B_W), 0);
    tc_fence_after();
    // gate GEMM of tile j (the j-th tile of this CTA): A = the staged c2 tile, B = the gate weights, D = acc2
    auto gate_phase = [&](int j) {
      const int g = G == 2 ? (j & 1) : 0;                    // epilogue group of tile j and its own tile count
      const uint32_t par = (uint32_t)((G == 2 ? (j >> 1) : j) & 1);
      mbar_wait(BAR(B_A2E + g), par ^ 1);                    // epilogue drained this gate accumulator
      mbar_wait(BAR(B_C2 + g), par);                         // c2 of tile j is staged (and fenced for the async proxy)
      tc_fence_after();
      if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[j * 16 + 10] = clock64();
      if (elect_one()) {
        const uint64_t adesc = umma_desc_k_sw128(smem_u32(sC2 + g * CG_TILE_BYTES));
        const uint64_t bdesc = umma_desc_k_sw128(smem_u32(sWg));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem_u + 128u + (uint32_t)(g * 128), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idescg, (uint32_t)(k != 0));
        umma_commit(BAR(B_A2F + g));
      }
      __syncwarp();
    };
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      mbar_wait(BAR(B_A1E + buf), (use & 1) ^ 1);            // epilogue drained this 3x3 accumulator
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + (uint32_t)(buf * 64);
      CG_STAMP(8);
      if (p.halo) {
        mbar_wait(BAR(stage), phase);
        tc_fence_after();
        CG_STAMP(9);
        const uint32_t a_base = smem_u32(sA + stage * stage_bytes);
        if (elect_one()) {
          for (int t = 0; t < CG_TAPS; ++t) {
            // tap (dy,dx) = (t/3 - 1, t%3 - 1): the tile's first pixel sits at halo row 1+dy, halo column 1+dx
            const uint32_t a_start = a_base + (uint32_t)(((t / 3) * 16 + (t % 3)) * 128);
            const uint64_t adesc = umma_desc_k_sw128(a_start, 2048);
            const uint64_t bdesc = umma_desc_k_sw128(smem_u32(sW2 + t * 64 * 128));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc3, (uint32_t)((t | k) != 0));
          }
          umma_commit(BAR(S + stage));
          umma_commit(BAR(B_A1F + buf));
        }
        __syncwarp();
        if (++stage == S) { stage = 0; phase ^= 1; }
      } else {
        for (int t = 0; t < CG_TAPS; ++t) {
          mbar_wait(BAR(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = umma_desc_k_sw128(smem_u32(sA + stage * CG_TILE_BYTES));
            const uint64_t bdesc = umma_desc_k_sw128(smem_u32(sW2 + t * 64 * 128));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc3, (uint32_t)((t | k) != 0));
            umma_commit(BAR(S + stage));
          }
          __syncwarp();
          if (++stage == S) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(BAR(B_A1F + buf));
        __syncwarp();
      }
      if (it > 0) gate_phase(it - 1);      // behind the 3x3 MMAs of this tile: the epilogue had their whole duration to stage tile it-1
    }
    if (it > 0) gate_phase(it - 1);
  } else {
    // ===================== epilogue (EW warps: TMEM lane quadrant x column part) =====================
    const int quad = warp & 3;
    const int part = (warp - 2) >> 2;                          // which CPT columns of every 64-column block
    const int row = quad * 32 + lane;
    const int ew = warp - 2;
    float ra0 = 0.f, ra1 = 0.f, rb0 = 0.f, rb1 = 0.f;          // statistics of out, channels 2l and 2l+1
    const int rstep = p.halo ? p.W - 8 : 0;
#define CG_EPI_BAR() asm volatile("bar.sync 1, %0;" ::"n"(32 * EW) : "memory")
    if (fast) {
      // ---------------- eval mode (the IW evaluator's sample passes) ----------------
      // Group g = eight warps (TMEM lane quadrant x column half, 32 accumulator columns per thread) owns the CTA's tiles
      // it = g, g + G, ...  The gate is evaluated straight from the accumulator registers -- a thread's loads are channels
      // [32 half, 32 half + 32) of `a` and of `g` for its own pixel -- values rounded to bf16 exactly where the training path
      // rounds them (so `out` is bit-identical to it), and `out` is staged in the buffer that held c2 (the gate GEMM is done).
      const int g = G == 2 ? (ew >> 3) : 0;
      const int half = (ew & 7) >> 2;
      uint8_t* sStage = sC2 + g * CG_TILE_BYTES;
      const bool elected = threadIdx.x == 64 + g * 256;
      const float* ba = sbias + 64 + 32 * half;
      const float* bg = sbias + 128 + 32 * half;
      const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
      auto group_bar = [&]() {
        if (G == 2) asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
        else CG_EPI_BAR();
      };
      int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        if (G == 2 && (it & 1) != g) continue;
        const int buf = it & 1;
        const uint32_t par1 = (uint32_t)((it >> 1) & 1);                       // this acc1 buffer's use count
        const uint32_t par2 = (uint32_t)((G == 2 ? (it >> 1) : it) & 1);       // the group's own tile count
        int m = tile * CG_BM + row;
        int c1, c2, c3;
        if (p.halo) {
          const int n0 = tile >> p.lg_tpi;
          const int r = tile & (p.tiles_per_img - 1);
          const int ty = r >> p.lg_tx, tx = r & (p.tiles_x - 1);
          m = (n0 * p.H + ty * 16 + (row >> 3)) * p.W + tx * 8 + (row & 7);
          c3 = n0; c2 = ty * 16; c1 = tx * 8;
        } else {
          const int p0 = tile * CG_BM;
          c3 = p0 >> p.lg_hw;
          const int rem = p0 & (hw - 1);
          c2 = rem >> p.lg_w; c1 = rem & (p.W - 1);
        }
        const bool valid = m < p.M_total;
        const float* scale_row = p.scale2 ? p.scale2 + (long long)(valid ? (m >> p.lg_hw) : 0) * 64 : nullptr;
        if (ew == 0 || ew == 8) CG_STAMP(0);
        uint4 xr[4];                                              // this thread's half row of the residual: requested first
#pragma unroll
        for (int q = 0; q < 4; ++q)
          xr[q] = valid ? __ldg(reinterpret_cast<const uint4*>(p.x_res + (long long)m * 64 + 32 * half) + q) : make_uint4(0u, 0u, 0u, 0u);
        // phase 1: c2 = (acc1 + bias2) * mask2 -> bf16 -> the group's staging buffer
        mbar_wait(BAR(B_A1F + buf), par1);
        tc_fence_after();
        if (ew == 0 || ew == 8) CG_STAMP(1);
        {
          uint4 pc[4];
          uint32_t r[32];
          tmem_ld32_nowait(lane_addr + (uint32_t)(buf * 64 + 32 * half), r);
          tmem_wait_ld();
          packN<32>(r, sbias, scale_row, 32 * half, pc);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(BAR(B_A1E + buf));           // the 3x3 accumulator is free for the tile after next
          if (elected) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the group's previous `out` store has left the buffer
          group_bar();
          uint8_t* blk = sStage + row * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(blk + (((4 * half + q) ^ (row & 7)) << 4)) = pc[q];
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        group_bar();
        if (ew == 0 || ew == 8) CG_STAMP(3);
        if (elected) mbar_arrive(BAR(B_C2 + g));                  // the MMA warp may run the gate GEMM on the staged tile
        // phase 2: out = act(a) * sigmoid(g) + x from the gate accumulator, 16 columns at a time
        mbar_wait(BAR(B_A2F + g), par2);
        tc_fence_after();
        if (ew == 0 || ew == 8) CG_STAMP(4);
        uint4 po[4];
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
          uint32_t ra[16], rg[16];
          tmem_ld16_nowait(lane_addr + (uint32_t)(128 + g * 128 + 32 * half + 16 * hq), ra);
          tmem_ld16_nowait(lane_addr + (uint32_t)(128 + g * 128 + 64 + 32 * half + 16 * hq), rg);
          tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const uint32_t* xw = reinterpret_cast<const uint32_t*>(&xr[2 * hq + q]);
            uint32_t* ow = reinterpret_cast<uint32_t*>(&po[2 * hq + q]);
            const float4 ba0 = *reinterpret_cast<const float4*>(ba + 16 * hq + 8 * q), ba1 = *reinterpret_cast<const float4*>(ba + 16 * hq + 8 * q + 4);
            const float4 bg0 = *reinterpret_cast<const float4*>(bg + 16 * hq + 8 * q), bg1 = *reinterpret_cast<const float4*>(bg + 16 * hq + 8 * q + 4);
            const float bav[8] = {ba0.x, ba0.y, ba0.z, ba0.w, ba1.x, ba1.y, ba1.z, ba1.w};
            const float bgv[8] = {bg0.x, bg0.y, bg0.z, bg0.w, bg1.x, bg1.y, bg1.z, bg1.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = 8 * q + 2 * e;
              const __nv_bfloat162 ab = __floats2bfloat162_rn(__uint_as_float(ra[c]) + bav[2 * e], __uint_as_float(ra[c + 1]) + bav[2 * e + 1]);
              const __nv_bfloat162 gb = __floats2bfloat162_rn(__uint_as_float(rg[c]) + bgv[2 * e], __uint_as_float(rg[c + 1]) + bgv[2 * e + 1]);
              const float2 af = __bfloat1622float2(ab), gf = __bfloat1622float2(gb);
              const float x0 = __uint_as_float(xw[e] << 16), x1 = __uint_as_float(xw[e] & 0xFFFF0000u);
              const float o0 = fmaf(act_fwd_t<true>(af.x, gact), sigmoid_tanh_approx(gf.x), x0);
              const float o1 = fmaf(act_fwd_t<true>(af.y, gact), sigmoid_tanh_approx(gf.y), x1);
              const __nv_bfloat162 ob = __floats2bfloat162_rn(o0, o1);
              ow[e] = *reinterpret_cast<const uint32_t*>(&ob);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(B_A2E + g));               // the gate accumulator is free for the group's next tile
        if (ew == 0 || ew == 8) CG_STAMP(5);
        {
          uint8_t* blk = sStage + row * 128;                      // c2 was consumed: acc2_full means the gate MMAs have completed
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(blk + (((4 * half + q) ^ (row & 7)) << 4)) = po[q];
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        group_bar();
        if (elected) {
          tma_store_4d(&tmOut, smem_u32(sStage), 0, c1, c2, c3);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (ew == 0 || ew == 8) CG_STAMP(6);
      }
      if (elected) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else {
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      // pixel of this thread's accumulator row; first pixel of the RPW staged rows this warp owns in the gate pass
      int m = tile * CG_BM + row;                               // (M_total = B*H*W fits an int)
      int rbase = tile * CG_BM + ew * RPW;
      int c1, c2, c3;                                           // TMA-store coordinates of the tile
      if (p.halo) {
        const int n0 = tile >> p.lg_tpi;
        const int r = tile & (p.tiles_per_img - 1);
        const int ty = r >> p.lg_tx, tx = r & (p.tiles_x - 1);
        m = (n0 * p.H + ty * 16 + (row >> 3)) * p.W + tx * 8 + (row & 7);
        rbase = (n0 * p.H + ty * 16 + ((ew * RPW) >> 3)) * p.W + tx * 8;
        c3 = n0; c2 = ty * 16; c1 = tx * 8;
      } else {
        const int p0 = tile * CG_BM;
        c3 = p0 >> p.lg_hw;
        const int rem = p0 & (hw - 1);
        c2 = rem >> p.lg_w; c1 = rem & (p.W - 1);
      }
      const bool valid = m < p.M_total;
      const int b = valid ? (m >> p.lg_hw) : 0;
      const float* scale_row = p.scale2 ? p.scale2 + (long long)b * 64 : nullptr;
      const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);

      if (warp == 2) CG_STAMP(0);
      // ---------------- phase 1: c2 = (acc1 + bias2) * mask2 -> bf16 -> staged tile (+ TMA store) ----------------
      mbar_wait(BAR(B_A1F + buf), use & 1);
      tc_fence_after();
      if (warp == 2) CG_STAMP(1);
      uint4 pc[NQ];
      {
        uint32_t r[CPT];
        tmem_ldN_nowait<CPT>(lane_addr + (uint32_t)(buf * 64 + CPT * part), r);
        tmem_wait_ld();
        packN<CPT>(r, sbias, scale_row, CPT * part, pc);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(B_A1E + buf));             // the 3x3 accumulator is free for the tile after next
      if (warp == 2) CG_STAMP(2);
      // every TMA store of the previous tile (c2, h, out) has finished reading the staging buffers
      if (threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      CG_EPI_BAR();
      {
        uint8_t* blk = sC2 + row * 128;
#pragma unroll
        for (int q = 0; q < NQ; ++q) *reinterpret_cast<uint4*>(blk + (((NQ * part + q) ^ (row & 7)) << 4)) = pc[q];
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to TMA and tcgen05.mma
      CG_EPI_BAR();
      if (warp == 2) CG_STAMP(3);
      if (threadIdx.x == 64) {
        mbar_arrive(BAR(B_C2));                                  // the MMA warp may run the gate GEMM on the staged tile
        if (p.store_c2h) {
          tma_store_4d(&tmC2, smem_u32(sC2), 0, c1, c2, c3);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
      // residual rows for the gate pass: in flight while the gate GEMM runs
      uint32_t xq[RPW];
      {
        const uint32_t* xb = reinterpret_cast<const uint32_t*>(p.x_res + (long long)rbase * 64) + lane;
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
          const int off = i + (i >> 3) * rstep;
          xq[i] = rbase + off < p.M_total ? __ldg(xb + off * 32) : 0u;
        }
      }

      // ---------------- phase 2: h = acc2 + bias_g -> bf16 -> staged (+ TMA store); gate pass; out -> staged -> TMA store ------
      mbar_wait(BAR(B_A2F), (uint32_t)(it & 1));
      tc_fence_after();
      if (warp == 2) CG_STAMP(4);
      // (sH is free: the previous tile's h store finished reading it before this tile's phase 1 passed its first barrier)
#pragma unroll
      for (int nch = 0; nch < 2; ++nch) {
        uint32_t r[CPT];
        uint4 ph[NQ];
        tmem_ldN_nowait<CPT>(lane_addr + (uint32_t)(128 + CPT * part + 64 * nch), r);
        tmem_wait_ld();
        packN<CPT>(r, sbias + 64, nullptr, CPT * part + 64 * nch, ph);
        uint8_t* blk = sH + nch * CG_TILE_BYTES + row * 128;
#pragma unroll
        for (int q = 0; q < NQ; ++q) *reinterpret_cast<uint4*>(blk + (((NQ * part + q) ^ (row & 7)) << 4)) = ph[q];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(B_A2E));                    // acc2 is free for the next tile's gate GEMM
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      CG_EPI_BAR();
      if (threadIdx.x == 64) {
        if (p.store_c2h) {
          tma_store_4d(&tmH, smem_u32(sH), 0, c1, c2, c3);
          tma_store_4d(&tmH, smem_u32(sH + CG_TILE_BYTES), 64, c1, c2, c3);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          // the c2 store (the older group) must have finished reading sC2 before the gate pass overwrites it with `out`
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        }
      }
      CG_EPI_BAR();
      {
        const int nrows = p.halo ? 128 : min(128, p.M_total - tile * CG_BM);
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
          const int r = ew * RPW + i;
          const int pos = r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + (lane & 3) * 4;
          const uint32_t ua = *reinterpret_cast<const uint32_t*>(sH + pos);
          const uint32_t ug = *reinterpret_cast<const uint32_t*>(sH + CG_TILE_BYTES + pos);
          const float a0 = __uint_as_float(ua << 16), a1 = __uint_as_float(ua & 0xFFFF0000u);
          const float s0 = __uint_as_float(ug << 16), s1 = __uint_as_float(ug & 0xFFFF0000u);
          const float x0 = __uint_as_float(xq[i] << 16), x1 = __uint_as_float(xq[i] & 0xFFFF0000u);
          const float o0 = fmaf(act_fwd_t<true>(a0, gact), sigmoid_tanh_approx(s0), x0);
          const float o1 = fmaf(act_fwd_t<true>(a1, gact), sigmoid_tanh_approx(s1), x1);
          const __nv_bfloat162 ob = __floats2bfloat162_rn(o0, o1);
          const uint32_t uo = *reinterpret_cast<const uint32_t*>(&ob);
          *reinterpret_cast<uint32_t*>(sC2 + pos) = uo;
          if (r < nrows) {                                       // statistics of the output as stored
            const float q0 = __uint_as_float(uo << 16), q1 = __uint_as_float(uo & 0xFFFF0000u);
            ra0 += q0; ra1 += q1;
            rb0 = fmaf(q0, q0, rb0); rb1 = fmaf(q1, q1, rb1);
          }
        }
      }
      if (warp == 2) CG_STAMP(5);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      CG_EPI_BAR();
      if (threadIdx.x == 64) {
        tma_store_4d(&tmOut, smem_u32(sC2), 0, c1, c2, c3);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (warp == 2) CG_STAMP(6);
    }
    }   // training path
    if (p.stats_acc) {
      // combine the EW row groups per channel in a fixed order (deterministic): eight slots, the warps beyond the eighth add
      // into the slot of warp ew - 8 after the first eight have written theirs
      if (ew < 8) {
        sred[(0 * 8 + ew) * 64 + 2 * lane] = ra0; sred[(0 * 8 + ew) * 64 + 2 * lane + 1] = ra1;
        sred[(1 * 8 + ew) * 64 + 2 * lane] = rb0; sred[(1 * 8 + ew) * 64 + 2 * lane + 1] = rb1;
      }
      CG_EPI_BAR();
      if (EW > 8) {
        if (ew >= 8) {
          sred[(0 * 8 + ew - 8) * 64 + 2 * lane] += ra0; sred[(0 * 8 + ew - 8) * 64 + 2 * lane + 1] += ra1;
          sred[(1 * 8 + ew - 8) * 64 + 2 * lane] += rb0; sred[(1 * 8 + ew - 8) * 64 + 2 * lane + 1] += rb1;
        }
        CG_EPI_BAR();
      }
      const int t = threadIdx.x - 64;
      if (t < 128) {
        const int st = t >> 6, c = t & 63;
        float sum = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) sum += sred[(st * 8 + e) * 64 + c];
        atomicAdd(p.stats_acc + (blockIdx.x & 7) * 128 + st * 64 + c, (double)sum);    // 8-way striped (see elementwise.cu)
      }
    }
#undef CG_EPI_BAR
  }
  if (threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_cg() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

int pow2_floor_le_cg(int v, int cap) {
  int r = 1;
  while (r * 2 <= v && r * 2 <= cap) r *= 2;
  return r;
}

long long* g_cg_dbg = nullptr;

}  // namespace

// profiling aid: CTA 0 of subsequent lvae_conv_gate_tc launches records clock64 stamps (16 per tile) into dev_buf (NULL = off)
LVAE_API void lvae_conv_gate_tc_debug(long long* dev_buf) { g_cg_dbg = dev_buf; }

// a2, x_res, c2, out: (B,H,W,64) bf16 NHWC; h: (B,H,W,128) bf16.  w2p: nine packed [64][64] blocks (tap-major, rows = output
// channel, lvae_pack_weights mode 2); wgp: one packed [128][64] block.  scale2: (B,64) or NULL.  c2 and h may both be NULL
// (eval: nothing runs backward).  stats_acc: 8-way striped (8,2,64) doubles or NULL.  H, W powers of two, W <= 128.
LVAE_API int lvae_conv_gate_tc(const void* a2, const void* w2p, const float* bias2, const float* scale2, const void* wgp,
                               const float* bias_g, const void* x_res, void* c2, void* h, void* out, double* stats_acc, int B,
                               int H, int W, int gate_act, cudaStream_t stream) {
  LVAE_REQUIRE(a2 && w2p && wgp && x_res && out, "conv_gate_tc: null pointer");
  LVAE_REQUIRE((c2 == nullptr) == (h == nullptr), "conv_gate_tc: c2 and h are stored together or not at all");
  LVAE_REQUIRE(B > 0 && (W & (W - 1)) == 0 && (H & (H - 1)) == 0 && W >= 1 && W <= 128 && H >= 1,
               "conv_gate_tc: H and W must be powers of two (W <= 128)");
  EncodeTiledFn enc = get_encode_cg();
  if (!enc) { lvae_set_error("conv_gate_tc: cuTensorMapEncodeTiled unavailable"); return LVAE_ERR_CUDA; }
  CgParams p{};
  p.bias2 = bias2; p.scale2 = scale2; p.bias_g = bias_g; p.x_res = (const __nv_bfloat16*)x_res; p.stats_acc = stats_acc;
  p.M_total = B * H * W; p.H = H; p.W = W;
  p.gate_act = gate_act;
  p.store_c2h = c2 ? 1 : 0;
  p.dbg = g_cg_dbg;
  p.halo = (W % 8 == 0 && H % 16 == 0) ? 1 : 0;
  p.stage_bytes = p.halo ? CG_HALO_BYTES : CG_TILE_BYTES;
  p.tiles_x = W / 8;
  p.tiles_per_img = (W / 8) * (H / 16);
  auto lg2 = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
  p.lg_w = lg2(W); p.lg_hw = lg2(H * W); p.lg_tx = lg2(p.tiles_x > 0 ? p.tiles_x : 1);
  p.lg_tpi = lg2(p.tiles_per_img > 0 ? p.tiles_per_img : 1);
  p.bw = W;
  p.bh = pow2_floor_le_cg(H, CG_BM / p.bw);
  p.bn = CG_BM / (p.bw * p.bh);
  const int fixed = 1024 + CG_TAPS * 64 * 128 + 128 * 128 + 3 * CG_TILE_BYTES + 8192;
  int stages = (227 * 1024 - fixed) / p.stage_bytes;
  if (stages > 8) stages = 8;
  LVAE_REQUIRE(stages >= 2, "conv_gate_tc: no room for the activation pipeline");
  p.n_stages = stages;
  const size_t smem = (size_t)fixed + (size_t)stages * p.stage_bytes;

  CUtensorMap tmA, tmW2, tmWg, tmC2, tmH, tmOut;
  memset(&tmC2, 0, sizeof(tmC2));
  memset(&tmH, 0, sizeof(tmH));
  const cuuint32_t one[4] = {1, 1, 1, 1};
  auto enc_act = [&](CUtensorMap* tm, void* ptr, int ncols, bool load) -> CUresult {
    cuuint64_t gdim[4] = {(cuuint64_t)ncols, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t gstr[3] = {(cuuint64_t)ncols * 2, (cuuint64_t)W * ncols * 2, (cuuint64_t)H * W * ncols * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bn};
    if (p.halo) {
      if (load) { box[1] = 16; box[2] = 18; box[3] = 1; }
      else { box[1] = 8; box[2] = 16; box[3] = 1; }
    }
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ptr, gdim, gstr, box, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  };
  CUresult r = enc_act(&tmA, (void*)a2, 64, true);
  if (r == CUDA_SUCCESS) r = enc_act(&tmOut, out, 64, false);
  if (r == CUDA_SUCCESS && c2) r = enc_act(&tmC2, c2, 64, false);
  if (r == CUDA_SUCCESS && h) r = enc_act(&tmH, h, 128, false);
  if (r != CUDA_SUCCESS) { lvae_set_error("conv_gate_tc: tensor map (activation) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
  {
    cuuint64_t wstr[1] = {128};
    cuuint32_t westr[2] = {1, 1};
    cuuint64_t wdim2[2] = {64, (cuuint64_t)CG_TAPS * 64};
    cuuint32_t wbox2[2] = {64, 64};
    r = enc(&tmW2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)w2p, wdim2, wstr, wbox2, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    cuuint64_t wdimg[2] = {64, 128};
    cuuint32_t wboxg[2] = {64, 128};
    if (r == CUDA_SUCCESS)
      r = enc(&tmWg, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)wgp, wdimg, wstr, wboxg, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { lvae_set_error("conv_gate_tc: tensor map (weights) encode failed: %d", (int)r); return LVAE_ERR_CUDA; }
  }
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_gate_tc_kernel<ACT_ELU, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_gate_tc_kernel<-1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
    if (e != cudaSuccess) { lvae_set_error("conv_gate_tc: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
    attr = true;
  }
  const int n_tiles = p.halo ? B * p.tiles_per_img : (p.M_total + CG_BM - 1) / CG_BM;
  const int grid = n_tiles < lvae_num_sms() ? n_tiles : lvae_num_sms();
  if (gate_act == ACT_ELU) lvae_launch(conv_gate_tc_kernel<ACT_ELU, 16>, grid, 64 + 32 * 16, smem, stream, tmA, tmW2, tmWg, tmC2, tmH, tmOut, p);
  else lvae_launch(conv_gate_tc_kernel<-1, 8>, grid, 64 + 32 * 8, smem, stream, tmA, tmW2, tmWg, tmC2, tmH, tmOut, p);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("conv_gate_tc");
  return LVAE_OK;
}
