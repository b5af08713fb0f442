// bf16 weight-gradient GEMM on the 5th-generation tensor cores (sm_100a):
//     dW[tap][ci][co] = sum_pixels X[pixel + offset(tap)][ci] * dY[pixel][co]
// for the stride-1 "same" convolutions (3x3 64->64, 1x1 64->128 gate, 1x1 merge over two inputs).
//
// The reduction dimension is the pixel index, so both operands are "MN-major": a TMA tile of 128
// pixels x 64 channels (128-byte swizzled rows) is, read column-wise, a 64 x 128 operand whose K
// runs over the rows.  One tcgen05.mma (M = 128, N = co, K = 16 pixels) consumes TWO activation
// tiles stacked along M (two filter taps, or a tap and an all-ones tile whose accumulator rows are
// the bias gradient), so a 3x3 convolution needs five accumulators of 64 TMEM columns each.
// Every CTA reduces its share of the pixel tiles into TMEM, then adds its fp32 partial into the PACKED gradient
// Gp[(pair, row)][co] with TMA reduce-stores (cp.reduce.async.bulk.tensor ... .add: the additions happen in L2, there is
// no per-CTA workspace and no reduction pass).  lvae_wgrad_unpack[_batched] re-lays Gp into the (O, I, kh, kw) gradient.
// Shifted 4-D TMA boxes implement im2col, out-of-bounds zero fill implements the padding.
#include "common.cuh"
#include <cuda.h>
#include <string.h>

namespace {

constexpr int WG_THREADS_TC = 192;
constexpr int WG_TILE = 128;                 // pixels per tile (K of the GEMM)
constexpr int WG_BLK_BYTES = WG_TILE * 64 * 2;   // 16 KB
constexpr int WG_MAX_PAIRS = 5;
constexpr int WG_PAIR_SLOTS = 4;
constexpr int WG_B_SLOTS = 2;
constexpr int WG_HALO_BYTES = 18 * 16 * 128;                         // 36 KB
constexpr int WG_HALO_STAGE_BYTES = WG_HALO_BYTES + WG_BLK_BYTES;    // + the dY tile
constexpr int WG_HALO_STAGES = 3;

struct WgParams {
  int M_total, H, W;
  int n_pairs;               // accumulators
  int n_bblk;                // dY channel blocks of 64 (1 or 2)  -> N = 64 * n_bblk
  int tmem_cols;
  int tiles_per_cta;
  int dy_c0;                 // first dY channel of this launch (dY may be wider than N: split launches)
  int x_c0;                  // first channel of the 64-channel X window (X, X2 may be wider than 64: split launches)
  // halo mode (3x3, one input, N = 64, W % 8 == 0, H % 16 == 0): pixel tiles are 16 rows x 8 columns and ONE TMA box of
  // 18 rows x 16 columns serves all nine taps (shifted MN-major descriptors, SBO = one 16-pixel image row = 2048 B)
  int halo, tiles_x, tiles_per_img;
  // stride-2 convolutions (lvae_conv2d_wgrad_tc_s2*): the shifted operand lives on the grid of twice the size and its tensor
  // map traverses it with element stride 2; a tile's pixel coordinates are multiplied by in_stride before the tap offset is added
  int in_stride;

  // A-block table: 2 per pair.  src: 0 = x, 1 = x2, 2 = ones tile, 3 = unused (zero rows, never read back)
  int8_t a_src[2 * WG_MAX_PAIRS], a_dx[2 * WG_MAX_PAIRS], a_dy[2 * WG_MAX_PAIRS];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
// MN-major, 128B-swizzled operand: 64 MN elements per 128-byte row, 8 K-rows per 1024-byte atom (SBO),
// next block of 64 MN elements LBO bytes further.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes = 1024) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
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
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__global__ void __launch_bounds__(WG_THREADS_TC, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmX2,
                const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmGp, const WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // keeps the shared address space
  uint8_t* sPair = smem;                                                   // WG_PAIR_SLOTS x 32 KB
  uint8_t* sB = sPair + WG_PAIR_SLOTS * 2 * WG_BLK_BYTES;                  // WG_B_SLOTS x n_bblk x 16 KB
  // halo mode re-uses the same region as WG_HALO_STAGES x (36 KB halo tile + 16 KB dY tile); the ones tile sits above both
  uint8_t* sOnes = p.halo ? smem + WG_HALO_STAGES * WG_HALO_STAGE_BYTES
                          : sB + WG_B_SLOTS * p.n_bblk * WG_BLK_BYTES;     // 16 KB of bf16 1.0
  uint64_t* bars = (uint64_t*)(sOnes + WG_BLK_BYTES);
  // barriers: [0,4) pair full, [4,8) pair empty, [8,10) b full, [10,12) b empty, 12: accumulators done
  uint32_t* tmem_slot = (uint32_t*)(bars + 16);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = p.halo ? (p.M_total / (p.H * p.W)) * p.tiles_per_img : (p.M_total + WG_TILE - 1) / WG_TILE;
  const int tile_beg = blockIdx.x * p.tiles_per_cta;
  const int tile_end = min(n_tiles, tile_beg + p.tiles_per_cta);
  const int N = 64 * p.n_bblk;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 13; ++i) mbar_init(BAR(i), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // all-ones tile (any swizzle of a constant tile is the same tile)
  for (int i = threadIdx.x; i < WG_BLK_BYTES / 4; i += WG_THREADS_TC) ((uint32_t*)sOnes)[i] = 0x3F803F80u;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core (async proxy)
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch();

  if (warp == 0) {
    if (p.halo) {
      // ===================== TMA producer, halo mode: one halo box + one dY box per tile =====================
      int st = 0;
      uint32_t ph = 0;
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        const int n0 = tile / p.tiles_per_img;
        const int r = tile - n0 * p.tiles_per_img;
        const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
        mbar_wait(BAR(4 + st), ph ^ 1);
        if (elect_one()) {
          uint8_t* stage = smem + st * WG_HALO_STAGE_BYTES;
          mbar_expect_tx(BAR(st), (uint32_t)WG_HALO_STAGE_BYTES);
          tma_load_4d(smem_u32(stage), &tmX, BAR(st), p.x_c0, tx * 8 - 1, ty * 16 - 1, n0);
          tma_load_4d(smem_u32(stage + WG_HALO_BYTES), &tmDY, BAR(st), p.dy_c0, tx * 8, ty * 16, n0);
        }
        __syncwarp();
        if (++st == WG_HALO_STAGES) { st = 0; ph ^= 1; }
      }
    } else {
      // ===================== TMA producer (whole warp loops, one elected lane issues) =====================
      const int hw = p.H * p.W;
      int ps = 0, bs = 0;
      uint32_t pph = 0, bph = 0;
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        int p0 = tile * WG_TILE;
        int n0 = p0 / hw;
        int rem = p0 - n0 * hw;
        int h0 = rem / p.W;
        int w0 = rem - h0 * p.W;
        mbar_wait(BAR(10 + bs), bph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(8 + bs), (uint32_t)(p.n_bblk * WG_BLK_BYTES));
          for (int j = 0; j < p.n_bblk; ++j)
            tma_load_4d(smem_u32(sB + (bs * p.n_bblk + j) * WG_BLK_BYTES), &tmDY, BAR(8 + bs), p.dy_c0 + 64 * j, w0, h0, n0);
        }
        __syncwarp();
        if (++bs == WG_B_SLOTS) { bs = 0; bph ^= 1; }
        for (int pr = 0; pr < p.n_pairs; ++pr) {
          mbar_wait(BAR(4 + ps), pph ^ 1);
          if (elect_one()) {
            int nload = 0;
            for (int h = 0; h < 2; ++h) nload += p.a_src[2 * pr + h] < 2 ? 1 : 0;
            mbar_expect_tx(BAR(ps), (uint32_t)(nload * WG_BLK_BYTES));
            for (int h = 0; h < 2; ++h) {
              int src = p.a_src[2 * pr + h];
              if (src < 2)
                tma_load_4d(smem_u32(sPair + (ps * 2 + h) * WG_BLK_BYTES), src ? &tmX2 : &tmX, BAR(ps), p.x_c0,
                            w0 * p.in_stride + p.a_dx[2 * pr + h], h0 * p.in_stride + p.a_dy[2 * pr + h], n0);
            }
          }
          __syncwarp();
          if (++ps == WG_PAIR_SLOTS) { ps = 0; pph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer (whole warp loops, one elected lane issues) =====================
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      // D fp32, A/B bf16, both MN-major, M = 128, N = 64 * n_bblk
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                             ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      int ps = 0, bs = 0;
      uint32_t pph = 0, bph = 0;
      if (p.halo) {
        int st = 0;
        uint32_t ph = 0;
        const uint32_t ones = smem_u32(sOnes);
        for (int tile = tile_beg; tile < tile_end; ++tile) {
          mbar_wait(BAR(st), ph);
          tc_fence_after();
          const uint32_t h_addr = smem_u32(smem + st * WG_HALO_STAGE_BYTES);
          const uint32_t b_addr = h_addr + WG_HALO_BYTES;
          if (elect_one()) {
            for (int pr = 0; pr < p.n_pairs; ++pr) {
              // block (dy,dx): the tile's first pixel sits at halo row 1+dy, column 1+dx; halo rows are 16 pixels (2048 B)
              const uint32_t a0 = h_addr + (uint32_t)(((1 + p.a_dy[2 * pr]) * 16 + (1 + p.a_dx[2 * pr])) * 128);
              const bool second_ones = p.a_src[2 * pr + 1] == 2;
              const uint32_t a1 = h_addr + (uint32_t)(((1 + p.a_dy[2 * pr + 1]) * 16 + (1 + p.a_dx[2 * pr + 1])) * 128);
              const uint32_t d_tmem = tmem_u + (uint32_t)(pr * N);
#pragma unroll
              for (int k = 0; k < WG_TILE / 16; ++k) {
                // K-step k = output rows 2k, 2k+1 of the tile = two 8-pixel groups one halo row (2048 B) apart
                const uint32_t ak = a0 + k * 4096;
                const uint32_t lbo = second_ones ? ones - ak : a1 - a0;
                umma_bf16(d_tmem, umma_desc_mn_sw128(ak, lbo, 2048), umma_desc_mn_sw128(b_addr + k * 2048, WG_BLK_BYTES),
                          idesc, (uint32_t)((tile != tile_beg) || k != 0));
              }
            }
            umma_commit(BAR(4 + st));
          }
          __syncwarp();
          if (++st == WG_HALO_STAGES) { st = 0; ph ^= 1; }
        }
        if (elect_one()) umma_commit(BAR(12));
        __syncwarp();
      } else {
      for (int tile = tile_beg; tile < tile_end; ++tile) {
        mbar_wait(BAR(8 + bs), bph);
        tc_fence_after();
        const uint32_t b_addr = smem_u32(sB + bs * p.n_bblk * WG_BLK_BYTES);
        for (int pr = 0; pr < p.n_pairs; ++pr) {
          mbar_wait(BAR(ps), pph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sPair + ps * 2 * WG_BLK_BYTES);
          // second 64-row block: the slot's own second half, or the constant ones tile
          const uint32_t a2 = p.a_src[2 * pr + 1] == 2 ? smem_u32(sOnes) : a_addr + WG_BLK_BYTES;
          const uint32_t lbo_a = a2 - a_addr;
          const uint32_t d_tmem = tmem_u + (uint32_t)(pr * N);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < WG_TILE / 16; ++k) {
              // 16 pixels = two 8-row swizzle atoms = 2048 bytes along K; the ones tile is constant, so the
              // same LBO works for it at every k (a_k + LBO stays inside its 16 KB)
              umma_bf16(d_tmem, umma_desc_mn_sw128(a_addr + k * 2048, lbo_a), umma_desc_mn_sw128(b_addr + k * 2048, WG_BLK_BYTES),
                        idesc, (uint32_t)((tile != tile_beg) || k != 0));
            }
            umma_commit(BAR(4 + ps));
          }
          __syncwarp();
          if (++ps == WG_PAIR_SLOTS) { ps = 0; pph ^= 1; }
        }
        if (elect_one()) umma_commit(BAR(10 + bs));
        __syncwarp();
        if (++bs == WG_B_SLOTS) { bs = 0; bph ^= 1; }
      }
      if (elect_one()) umma_commit(BAR(12));
      __syncwarp();
      }
    }
  } else {
    // ===================== epilogue: TMEM -> registers -> swizzled staging tile -> TMA reduce-add into Gp ==========
    // The staging tiles (2 x 16 KB: 128 rows x 32 fp32 columns, 128B-swizzled) alias the operand pipeline, which is idle
    // once the last MMA has completed.
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const bool leader = threadIdx.x == 64;
    mbar_wait(BAR(12), 0);
    tc_fence_after();
    if (tile_beg < tile_end) {                         // a CTA without work has nothing to add
      int nbuf = 0;
      for (int pr = 0; pr < p.n_pairs; ++pr) {
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(pr * N);
        for (int c0 = 0; c0 < N; c0 += 32, ++nbuf) {
          uint8_t* stg = smem + (nbuf & 1) * WG_BLK_BYTES;
          uint32_t r[32];
          tmem_ld32(taddr + (uint32_t)c0, r);
          if (leader) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store two tiles back has read its buffer
          asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(stg + row * 128 + ((q ^ (row & 7)) << 4)) = make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (leader) {
            asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(&tmGp), "r"(smem_u32(stg)), "r"(c0), "r"(pr * 128) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// Packed gradient Gp -> torch-layout gradient.  Block blk (= pair*2 + half) of Gp holds 64 rows x N columns of kind
//   tap t, input-channel block s:   dw[(co*I_real + 64 s + ci)*taps + t] += Gp[blk*64 + ci][co]
//   ones:                            dbias[co] += Gp[blk*64][co]
// One descriptor per convolution (host-built, lvae_wgrad_unpack_desc); the batched kernel walks a device table of them.
struct UnpackDesc {
  const float* gp; float* dw; float* dbias;
  int n_pairs, N, taps, I_real, N_real, clear;
  int8_t kind[2 * WG_MAX_PAIRS];     // 0 tap block, 1 ones, 2 unused
  int8_t tap[2 * WG_MAX_PAIRS], ci0_blk[2 * WG_MAX_PAIRS];
  // X window of a split launch, in 64-channel blocks: the packed rows of input s hold dw input channels
  // s * xC + x_c0 + [0, 64).  Both zero (xC = 64, x_c0 = 0) for the single-window launches the engine batches.
  int8_t x_c0_blk, xC_blk;
};
static_assert(sizeof(UnpackDesc) == 80, "UnpackDesc layout is mirrored by engine.py");

constexpr int UNPACK_CO = 16;         // output channels per CTA (64-byte segments of Gp rows); each writes 16 contiguous (I_real * taps) runs of dw

// A CTA gathers Gp[*][co0..co0+3] for every (tap, ci) into shared memory laid out like dw, then adds contiguous runs.
// With clear != 0 it also zeroes what it consumed, so Gp is ready for the next step.
__device__ __forceinline__ void unpack_body(const UnpackDesc& d, float (*tile)[9 * 64 + 1]) {
  const int co0 = blockIdx.x * UNPACK_CO;
  if (co0 >= d.N_real) return;
  const int run = d.I_real * d.taps;                       // floats per output channel in dw
  float* gp = const_cast<float*>(d.gp);
  const int n_items = d.n_pairs * 128 * (UNPACK_CO / 4);
  const bool clear = (d.clear & 1) != 0, overwrite = (d.clear & 2) != 0;
  const bool windowed = d.x_c0_blk != 0 || d.xC_blk != 0;
  const int xC = 64 * (d.xC_blk ? d.xC_blk : 1), x_c0 = 64 * d.x_c0_blk;
  // four independent 16-byte loads in flight per thread
  for (int base = threadIdx.x; base < n_items; base += 4 * blockDim.x) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = base + u * blockDim.x;
      if (idx < n_items) v[u] = *reinterpret_cast<const float4*>(gp + (size_t)(idx / (UNPACK_CO / 4)) * d.N + co0 + 4 * (idx % (UNPACK_CO / 4)));
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = base + u * blockDim.x;
      if (idx >= n_items) break;
      const int i = idx / (UNPACK_CO / 4), part = idx % (UNPACK_CO / 4);        // Gp row, float4 within the 64-byte segment
      const int blk = i >> 6, ci = i & 63;
      const int kind = d.kind[blk];
      if (clear) *reinterpret_cast<float4*>(gp + (size_t)i * d.N + co0 + 4 * part) = make_float4(0.f, 0.f, 0.f, 0.f);
      const float vv[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
      if (kind == 0) {
        const int cin = d.ci0_blk[blk] * 64 + ci;                  // row of the packed gradient: input block, channel
        if ((windowed ? d.ci0_blk[blk] * xC + x_c0 + ci : cin) < d.I_real) {
          const int o = cin * d.taps + d.tap[blk];
#pragma unroll
          for (int e = 0; e < 4; ++e) tile[4 * part + e][o] = vv[e];
        }
      } else if (kind == 1 && ci == 0 && d.dbias) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (co0 + 4 * part + e < d.N_real) {
            if (overwrite) d.dbias[co0 + 4 * part + e] = vv[e];
            else d.dbias[co0 + 4 * part + e] += vv[e];
          }
      }
    }
  }
  __syncthreads();
  // contiguous runs of dw: (co0 + j) * run .. + run; all UNPACK_CO runs of this CTA are adjacent in memory
  const int nco = min(UNPACK_CO, d.N_real - co0);
  float* dst = d.dw + (size_t)co0 * run;
  const int total = nco * run;
  if (windowed) {
    // the tile holds 64 input channels per input, dw rows span all I_real of them: scatter each window into its place
    int inputs = 0;
    for (int b = 0; b < 2 * WG_MAX_PAIRS; ++b)
      if (d.kind[b] == 0 && d.ci0_blk[b] + 1 > inputs) inputs = d.ci0_blk[b] + 1;
    const int lrun = inputs * 64 * d.taps;                       // tile entries per output channel
    for (int o = threadIdx.x; o < nco * lrun; o += blockDim.x) {
      const int j = o / lrun, lo = o - j * lrun;
      const int cl = lo / d.taps, t = lo - cl * d.taps;
      const int cin = (cl >> 6) * xC + x_c0 + (cl & 63);
      if (cin >= d.I_real) continue;
      float* q = dst + (size_t)j * run + cin * d.taps + t;
      *q = overwrite ? tile[j][lo] : *q + tile[j][lo];
    }
    return;
  }
  if (overwrite) {
    for (int o = threadIdx.x; o < total; o += blockDim.x) dst[o] = tile[o / run][o % run];
  } else {
    for (int base = threadIdx.x; base < total; base += 4 * blockDim.x) {
      float old[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { const int o = base + u * blockDim.x; if (o < total) old[u] = dst[o]; }
#pragma unroll
      for (int u = 0; u < 4; ++u) { const int o = base + u * blockDim.x; if (o < total) dst[o] = old[u] + tile[o / run][o % run]; }
    }
  }
}

// grid (ceil(max N_real / 16), n_desc): one descriptor of the device table per blockIdx.y
__global__ void __launch_bounds__(256) wgrad_unpack_kernel(const UnpackDesc* __restrict__ table) {
  pdl_wait();
  pdl_launch();
  __shared__ UnpackDesc d;
  __shared__ float tile[UNPACK_CO][9 * 64 + 1];
  if (threadIdx.x < sizeof(UnpackDesc) / 4)
    reinterpret_cast<uint32_t*>(&d)[threadIdx.x] = reinterpret_cast<const uint32_t*>(table + blockIdx.y)[threadIdx.x];
  __syncthreads();
  unpack_body(d, tile);
}
// single convolution, descriptor passed by value
__global__ void __launch_bounds__(256) wgrad_unpack_one_kernel(const UnpackDesc dpar) {
  pdl_wait();
  pdl_launch();
  __shared__ UnpackDesc d;
  __shared__ float tile[UNPACK_CO][9 * 64 + 1];
  if (threadIdx.x == 0) d = dpar;
  __syncthreads();
  unpack_body(d, tile);
}

void fill_unpack_desc(UnpackDesc* d, const float* gp, float* dw, float* dbias, int N, int ksize, int inputs, int I_real,
                      int N_real, int clear, int xC = 64, int x_c0 = 0) {
  memset(d, 0, sizeof(*d));
  const int taps = ksize * ksize;
  int nblk = 0;
  for (int t = 0; t < taps; ++t)
    for (int s = 0; s < inputs && nblk < 2 * WG_MAX_PAIRS - 1; ++s, ++nblk) { d->kind[nblk] = 0; d->tap[nblk] = (int8_t)t; d->ci0_blk[nblk] = (int8_t)s; }
  if (nblk % 2 == 0 && nblk < 2 * WG_MAX_PAIRS - 1) { d->kind[nblk] = 2; ++nblk; }
  d->kind[nblk] = 1; ++nblk;
  d->gp = gp; d->dw = dw; d->dbias = dbias; d->n_pairs = nblk / 2; d->N = N; d->taps = taps;
  d->I_real = I_real > 0 ? I_real : 64 * inputs; d->N_real = N_real > 0 ? N_real : N; d->clear = clear;
  if (xC != 64 || x_c0 != 0) {
    d->x_c0_blk = (int8_t)(x_c0 / 64); d->xC_blk = (int8_t)(xC / 64);
    if (I_real <= 0) d->I_real = xC * inputs;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn wg_get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

int make_act_map(EncodeTiledFn enc, CUtensorMap* tm, const void* ptr, int B, int H, int W, int C, int bw, int bh, int bn, int st = 1) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)(bw * st), (cuuint32_t)(bh * st), (cuuint32_t)bn};
  cuuint32_t estr[4] = {1, (cuuint32_t)st, (cuuint32_t)st, 1};
  return (int)enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

}  // namespace

static bool wgrad_shape_ok(int N, int ksize, int inputs) {
  if (!(N == 64 || N == 128) || !(ksize == 1 || ksize == 3) || inputs < 1 || inputs > 2) return false;
  const int nblk = ksize * ksize * inputs;
  const int n_pairs = (nblk + 1 + (nblk % 2 == 0 ? 1 : 0)) / 2;
  return n_pairs <= WG_MAX_PAIRS && n_pairs * N <= 512;
}

// I_real / N_real (0 = all) select the rows / columns of Gp the unpack reads: more than the packed gradient holds would read
// (and with the clear bit zero) memory past each Gp row, or copy never-written shared memory into dw.
static bool wgrad_real_ok(int N, int inputs, int I_real, int N_real) {
  return I_real >= 0 && I_real <= 64 * inputs && N_real >= 0 && N_real <= N;
}

// Floats in the packed gradient Gp of one convolution (0 if the shape is unsupported): pairs x 128 rows x N columns.
LVAE_API long long lvae_wgrad_tc_packed_size(int N, int ksize, int two_inputs) {
  const int inputs = two_inputs ? 2 : 1;
  if (!wgrad_shape_ok(N, ksize, inputs)) return 0;
  const int nblk = ksize * ksize * inputs;
  return (long long)((nblk + 1 + (nblk % 2 == 0 ? 1 : 0)) / 2) * 128 * N;
}
// kept for callers of the previous interface: the workspace of lvae_conv2d_wgrad_tc is one packed gradient
LVAE_API long long lvae_wgrad_tc_workspace(int B, int H, int W, int N, int ksize, int two_inputs) {
  (void)B; (void)H; (void)W;
  return lvae_wgrad_tc_packed_size(N, ksize, two_inputs);
}

// Gp += wgrad.  x, x2: (B,H,W,64) bf16 (x2 optional); dY: (B,H,W,dyC) bf16 (dyC = 0 means N), already multiplied by any
// Dropout2d mask; this launch uses its channels [dy_c0, dy_c0 + N), N in {64, 128}.  gp: lvae_wgrad_tc_packed_size floats.
static int wgrad_tc_acc_impl(const void* x, const void* x2, const void* dy, float* gp, int B, int H, int W, int N,
                             int ksize, int dyC, int dy_c0, int in_stride, cudaStream_t stream, int xC = 64, int x_c0 = 0);

LVAE_API int lvae_conv2d_wgrad_tc_acc(const void* x, const void* x2, const void* dy, float* gp, int B, int H, int W, int N,
                                      int ksize, int dyC, int dy_c0, cudaStream_t stream) {
  return wgrad_tc_acc_impl(x, x2, dy, gp, B, H, W, N, ksize, dyC, dy_c0, 1, stream);
}

// Stride-2 3x3 convolutions 64 -> 64 (models/lvae_layers.py:261-276), Gp += sum over the (B,Hg,Wg) grid of
//   xs[b, 2gy-1+ky, 2gx-1+kx, row] * c[b, gy, gx, col]      xs: (B,2Hg,2Wg,64) bf16, c: (B,Hg,Wg,64) bf16
// Conv2d(stride 2, pad 1): xs = the input, c = dY -> rows = input channel, columns = output channel, ones row = bias gradient.
// ConvTranspose2d(stride 2, pad 1, output_padding 1): xs = dY, c = the input -> rows = OUTPUT channel, columns = input
// channel, which is the (Cin, Cout, 3, 3) layout of its weight under the same unpack formula (the ones row is then unused).
LVAE_API int lvae_conv2d_wgrad_tc_s2_acc(const void* xs, const void* c, float* gp, int B, int Hg, int Wg, cudaStream_t stream) {
  return wgrad_tc_acc_impl(xs, nullptr, c, gp, B, Hg, Wg, 64, 3, 64, 0, 2, stream);
}

static int wgrad_tc_acc_impl(const void* x, const void* x2, const void* dy, float* gp, int B, int H, int W, int N,
                             int ksize, int dyC, int dy_c0, int in_stride, cudaStream_t stream, int xC, int x_c0) {
  LVAE_REQUIRE(x && dy && gp, "conv2d_wgrad_tc: null pointer");
  LVAE_REQUIRE((N == 64 || N == 128) && (ksize == 1 || ksize == 3), "conv2d_wgrad_tc: N must be 64 or 128, ksize 1 or 3");
  LVAE_REQUIRE(B > 0 && H > 0 && W > 0 && (W & (W - 1)) == 0 && (H & (H - 1)) == 0 && W <= 128,
               "conv2d_wgrad_tc: H and W must be powers of two (W <= 128), B positive");
  if (dyC <= 0) dyC = N;
  LVAE_REQUIRE(dy_c0 >= 0 && dy_c0 % 64 == 0 && dy_c0 + N <= dyC, "conv2d_wgrad_tc: bad dY channel window");
  LVAE_REQUIRE(x_c0 >= 0, "conv2d_wgrad_tc: negative X channel window");
  LVAE_REQUIRE(x_c0 % 64 == 0, "conv2d_wgrad_tc: X channel window not 64-aligned");
  LVAE_REQUIRE(xC % 64 == 0 && xC <= 256 && x_c0 + 64 <= xC, "conv2d_wgrad_tc: X channel window past the %d input channels", xC);
  EncodeTiledFn enc = wg_get_encode();
  if (!enc) { lvae_set_error("conv2d_wgrad_tc: cuTensorMapEncodeTiled unavailable"); return LVAE_ERR_CUDA; }
  const int inputs = x2 ? 2 : 1, taps = ksize * ksize;
  LVAE_REQUIRE(wgrad_shape_ok(N, ksize, inputs), "conv2d_wgrad_tc: too many operand blocks (3x3 over two inputs is not supported)");
  WgParams p{};
  int nblk = 0;
  for (int t = 0; t < taps; ++t) {
    int oy = t / ksize - ksize / 2, ox = t % ksize - ksize / 2;
    for (int s = 0; s < inputs; ++s, ++nblk) { p.a_src[nblk] = (int8_t)s; p.a_dx[nblk] = (int8_t)ox; p.a_dy[nblk] = (int8_t)oy; }
  }
  // the ones block must be the SECOND half of a pair (its half of the descriptor is not advanced along K)
  if (nblk % 2 == 0) { p.a_src[nblk] = 0; p.a_dx[nblk] = 0; p.a_dy[nblk] = 0; ++nblk; }
  p.a_src[nblk] = 2; ++nblk;
  p.n_pairs = nblk / 2;
  p.n_bblk = N / 64;
  p.tmem_cols = 32;
  while (p.tmem_cols < p.n_pairs * N) p.tmem_cols *= 2;
  p.M_total = B * H * W; p.H = H; p.W = W;
  p.in_stride = in_stride;
  p.halo = (in_stride == 1 && ksize == 3 && !x2 && N == 64 && W % 8 == 0 && H % 16 == 0) ? 1 : 0;
  p.tiles_x = W / 8;
  p.tiles_per_img = (W / 8) * (H / 16);
  const int n_tiles = p.halo ? B * p.tiles_per_img : (p.M_total + WG_TILE - 1) / WG_TILE;
  // Few, fat CTAs: every CTA pays one pass of reduce-stores over the whole packed gradient (160 KB for a 3x3 conv), so the
  // SM-time of the launch is minimised by giving each CTA several pixel tiles; the kernel runs on a side stream, its latency
  // does not matter, and the SMs it leaves alone serve the main stream's convolutions (8: sweep in profiles/tail_kernels_r02.txt).
  constexpr int WG_TILES_PER_CTA = 8;
  int grid = (n_tiles + WG_TILES_PER_CTA - 1) / WG_TILES_PER_CTA;
  if (grid > lvae_num_sms()) grid = lvae_num_sms();
  if (grid < 1) grid = 1;
  p.tiles_per_cta = (n_tiles + grid - 1) / grid;
  grid = (n_tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  int bw = W;
  int bh = 1;
  while (bh * 2 <= H && bh * 2 * bw <= WG_TILE) bh *= 2;
  int bn = WG_TILE / (bw * bh);
  if (p.halo) { bw = 8; bh = 16; bn = 1; }
  CUtensorMap tmX, tmX2, tmDY, tmGp;
  p.x_c0 = x_c0;
  int r = p.halo ? make_act_map(enc, &tmX, x, B, H, W, xC, 16, 18, 1)
                 : make_act_map(enc, &tmX, x, B, H * in_stride, W * in_stride, xC, bw, bh, bn, in_stride);
  if (!r) r = make_act_map(enc, &tmX2, x2 ? x2 : x, B, H, W, xC, bw, bh, bn);
  p.dy_c0 = dy_c0;
  if (!r) r = make_act_map(enc, &tmDY, dy, B, H, W, dyC, bw, bh, bn);
  if (!r) {
    // Gp as a 2-D fp32 tensor (rows = pairs x 128, columns = N); the reduce-store box is 128 rows x 32 columns (128 B)
    cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)p.n_pairs * 128};
    cuuint64_t gstr[1] = {(cuuint64_t)N * 4};
    cuuint32_t box[2] = {32, 128};
    cuuint32_t estr[2] = {1, 1};
    r = (int)enc(&tmGp, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)gp, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r) { lvae_set_error("conv2d_wgrad_tc: tensor map encode failed: %d", r); return LVAE_ERR_CUDA; }
  const size_t smem = p.halo ? 1024 + (size_t)WG_HALO_STAGES * WG_HALO_STAGE_BYTES + WG_BLK_BYTES + 256
                             : 1024 + (size_t)WG_PAIR_SLOTS * 2 * WG_BLK_BYTES + (size_t)WG_B_SLOTS * p.n_bblk * WG_BLK_BYTES + WG_BLK_BYTES + 256;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { lvae_set_error("conv2d_wgrad_tc: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
    attr = true;
  }
  lvae_launch(wgrad_tc_kernel, grid, WG_THREADS_TC, smem, stream, tmX, tmX2, tmDY, tmGp, p);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("conv2d_wgrad_tc");
  return LVAE_OK;
}

// Bytes of one unpack descriptor and its construction on the host (the engine keeps a device table of them).
LVAE_API int lvae_wgrad_unpack_desc_size(void) { return (int)sizeof(UnpackDesc); }
LVAE_API int lvae_wgrad_unpack_desc(void* desc_host, const float* gp, float* dw, float* dbias, int N, int ksize, int two_inputs,
                                    int I_real, int N_real, int clear) {
  LVAE_REQUIRE(desc_host && gp && dw, "wgrad_unpack_desc: null pointer");
  LVAE_REQUIRE(wgrad_shape_ok(N, ksize, two_inputs ? 2 : 1), "wgrad_unpack_desc: unsupported shape");
  LVAE_REQUIRE(wgrad_real_ok(N, two_inputs ? 2 : 1, I_real, N_real),
               "wgrad_unpack_desc: I_real %d / N_real %d outside 0..%d / 0..%d", I_real, N_real, two_inputs ? 128 : 64, N);
  fill_unpack_desc((UnpackDesc*)desc_host, gp, dw, dbias, N, ksize, two_inputs ? 2 : 1, I_real, N_real, clear);
  return LVAE_OK;
}
// dw / dbias += unpack(Gp) for n descriptors in device memory (max_n_real: largest N_real among them)
LVAE_API int lvae_wgrad_unpack_batched(const void* desc_dev, int n, int max_n_real, cudaStream_t stream) {
  LVAE_REQUIRE(desc_dev && n > 0 && max_n_real > 0, "wgrad_unpack_batched: bad args");
  lvae_launch(wgrad_unpack_kernel, dim3(cdiv(max_n_real, UNPACK_CO), n), 256, 0, stream, (const UnpackDesc*)desc_dev);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("wgrad_unpack");
  return LVAE_OK;
}

// One-call form of the stride-2 gradient: dw (64, 64, 3, 3) fp32 += unpack(Gp) (see lvae_conv2d_wgrad_tc_s2_acc for the two operand
// orders), dbias [64] += column sums of c, or NULL.  ws: lvae_wgrad_tc_packed_size(64, 3, 0) floats, overwritten.
LVAE_API int lvae_conv2d_wgrad_tc_s2(const void* xs, const void* c, float* dw, float* dbias, float* ws, int B, int Hg, int Wg,
                                     cudaStream_t stream) {
  LVAE_REQUIRE(xs && c && dw && ws, "conv2d_wgrad_tc_s2: null pointer");
  const long long n = lvae_wgrad_tc_packed_size(64, 3, 0);
  cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)n * 4, stream);
  if (e != cudaSuccess) { lvae_set_error("conv2d_wgrad_tc_s2: memset failed: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
  int rc = lvae_conv2d_wgrad_tc_s2_acc(xs, c, ws, B, Hg, Wg, stream);
  if (rc) return rc;
  UnpackDesc d;
  fill_unpack_desc(&d, ws, dw, dbias, 64, 3, 1, 64, 64, 0);
  lvae_launch(wgrad_unpack_one_kernel, dim3(cdiv(d.N_real, UNPACK_CO), 1), 256, 0, stream, d);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("wgrad_unpack");
  return LVAE_OK;
}

// One-call form: dw (N_real, I_real, k, k) fp32 += wgrad, dbias [N_real] += column sums (or NULL).  x may carry zero-padded
// channels beyond I_real (0 = none), dY beyond N_real (0 = none).  ws: lvae_wgrad_tc_workspace floats, overwritten.
LVAE_API int lvae_conv2d_wgrad_tc_ex(const void* x, const void* x2, const void* dy, float* dw, float* dbias, float* ws,
                                     int B, int H, int W, int N, int ksize, int I_real, int N_real, int dyC, int dy_c0,
                                     int xC, int x_c0, cudaStream_t stream);

LVAE_API int lvae_conv2d_wgrad_tc(const void* x, const void* x2, const void* dy, float* dw, float* dbias, float* ws,
                                  int B, int H, int W, int N, int ksize, int I_real, int N_real, int dyC, int dy_c0,
                                  cudaStream_t stream) {
  return lvae_conv2d_wgrad_tc_ex(x, x2, dy, dw, dbias, ws, B, H, W, N, ksize, I_real, N_real, dyC, dy_c0, 0, 0, stream);
}

// The same over the 64-channel X window [x_c0, x_c0 + 64) of inputs with xC channels each (0 = 64): dw is (N_real, I_real,
// k, k) with I_real = xC per input (0) or fewer, and this launch adds the window's columns of it.  The bias gradient comes
// with every launch: pass dbias to exactly one launch per dY window.
LVAE_API int lvae_conv2d_wgrad_tc_ex(const void* x, const void* x2, const void* dy, float* dw, float* dbias, float* ws,
                                     int B, int H, int W, int N, int ksize, int I_real, int N_real, int dyC, int dy_c0,
                                     int xC, int x_c0, cudaStream_t stream) {
  LVAE_REQUIRE(x && dy && dw && ws, "conv2d_wgrad_tc: null pointer");
  const long long n = lvae_wgrad_tc_packed_size(N, ksize, x2 != nullptr);
  LVAE_REQUIRE(n > 0, "conv2d_wgrad_tc: unsupported shape");
  if (xC <= 0) xC = 64;
  const int inputs = x2 ? 2 : 1;
  LVAE_REQUIRE(I_real >= 0 && I_real <= xC * inputs && N_real >= 0 && N_real <= N,
               "conv2d_wgrad_tc: I_real %d / N_real %d outside 0..%d / 0..%d", I_real, N_real, xC * inputs, N);
  LVAE_REQUIRE(x_c0 >= 0, "conv2d_wgrad_tc: negative X channel window");
  LVAE_REQUIRE(x_c0 % 64 == 0, "conv2d_wgrad_tc: X channel window not 64-aligned");
  LVAE_REQUIRE(xC % 64 == 0 && xC <= 256 && x_c0 + 64 <= xC, "conv2d_wgrad_tc: X channel window past the %d input channels", xC);
  cudaError_t e = cudaMemsetAsync(ws, 0, (size_t)n * 4, stream);
  if (e != cudaSuccess) { lvae_set_error("conv2d_wgrad_tc: memset failed: %s", cudaGetErrorString(e)); return LVAE_ERR_CUDA; }
  int rc = wgrad_tc_acc_impl(x, x2, dy, ws, B, H, W, N, ksize, dyC, dy_c0, 1, stream, xC, x_c0);
  if (rc) return rc;
  UnpackDesc d;
  fill_unpack_desc(&d, ws, dw, dbias, N, ksize, inputs, I_real, N_real, 0, xC, x_c0);
  lvae_launch(wgrad_unpack_one_kernel, dim3(cdiv(d.N_real, UNPACK_CO), 1), 256, 0, stream, d);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("wgrad_unpack");
  return LVAE_OK;
}
