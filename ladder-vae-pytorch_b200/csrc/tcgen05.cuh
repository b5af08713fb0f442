// The Blackwell (sm_100a) primitives of the tensor-core kernels: mbarriers, TMA (cp.async.bulk.tensor), bulk-group
// completion, tcgen05 MMA / TMEM and the shared-memory and instruction descriptors, plus the host-side tensor-map encoders.
// One copy for conv_tcgen05.cu, conv_gate_tcgen05.cu and wgrad_tcgen05.cu: the descriptor bit layouts live here only.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace {

// ---- shared memory, mbarriers, fences ----
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
// makes the mbarrier.init of this thread visible to the other threads and to the async proxy (TMA, tcgen05.commit)
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the async proxy (TMA stores, tcgen05.mma operands)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// named barrier ID over THREADS threads (a multiple of 32), immediate operands
template <int ID, int THREADS> __device__ __forceinline__ void named_bar_sync() {
  asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(THREADS) : "memory");
}

// ---- TMA ----
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
// global tile += shared tile (fp32 addition in L2)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* tm, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(tm), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
// bulk groups of the issuing thread's TMA stores / reduce-stores
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N groups still pending (complete: their global writes are done)
template <int N> __device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// at most N groups still reading their shared-memory source (the buffer may be overwritten)
template <int N> __device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ---- TMEM ----
// Warp-collective: writes the base address of ncols (a power of two >= 32) columns to the shared-memory word at slot.
// The operands are const references: a by-value copy changes nvcc's virtual-register order in conv_gate_tc_kernel.
__device__ __forceinline__ void tmem_alloc(const uint32_t& slot, const uint32_t& ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(const uint32_t& taddr, const uint32_t& ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 32 / 16 consecutive 32-bit columns; the registers are valid after tmem_wait_ld()
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
// order tcgen05 operations against a thread synchronisation (barrier, mbarrier wait) before / after it
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- MMA ----
// D[tmem] (+)= A * B, kind::f16 (bf16 operands, fp32 accumulator per idesc); accumulate == 0 overwrites D
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives once on the mbarrier when every tcgen05.mma this thread issued before it has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
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

// ---- descriptors ----
// Shared-memory operand descriptor, both forms 128B-swizzled (bits 61-63 = 2) and version 1 (bit 46, Blackwell):
//   bits 0-13 start address >> 4, bits 16-29 leading byte offset >> 4, bits 32-45 stride byte offset >> 4.
// Advancing K by 16 bf16 (32 bytes) inside a swizzle atom is +2 on the descriptor.
// K-major: rows of 128 B (64 bf16 of K), 8-row groups sbo bytes apart; LBO is unused (1).  The start address may be only
// 128-byte aligned (shifted halo taps); the base-offset field stays zero because the hardware swizzle is a function of the
// absolute shared-memory address.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr, uint32_t sbo_bytes = 1024) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major: 64 MN elements per 128-byte row, 8 K-rows per 1024-byte atom (SBO), next block of 64 MN elements LBO bytes further.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes = 1024) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor of tcgen05.mma.kind::f16, D fp32, A and B bf16, dense, no negation:
//   bits 4-5 D type (1 = f32), 7-9 A type (1 = bf16), 10-12 B type (1 = bf16), 15 A MN-major, 16 B MN-major,
//   17-22 N >> 3, 24-28 M >> 4.
__host__ __device__ __forceinline__ constexpr uint32_t umma_idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// ---- host: tensor maps ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled from the driver, or null
inline EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// NHWC bf16 tensor (B, H, W, C) as a 4-D map with boxes of 64 channels x bw x bh x bn pixels, 128B-swizzled, zero fill out of
// bounds.  st > 1 traverses W and H with that element stride: the box then spans st * bw x st * bh pixels and delivers bw x bh.
inline CUresult make_act_map(EncodeTiledFn enc, CUtensorMap* tm, const void* ptr, int B, int H, int W, int C, int bw, int bh,
                             int bn, int st = 1) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)(bw * st), (cuuint32_t)(bh * st), (cuuint32_t)bn};
  cuuint32_t estr[4] = {1, (cuuint32_t)st, (cuuint32_t)st, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// Packed bf16 weights [rows][64] (one 128-byte swizzle row each) as a 2-D map with boxes of box_rows rows.
inline CUresult make_weight_map(EncodeTiledFn enc, CUtensorMap* tm, const void* ptr, int rows, int box_rows) {
  cuuint64_t dim[2] = {64, (cuuint64_t)rows};
  cuuint64_t str[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)ptr, dim, str, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// ---- host: powers of two ----
// largest power of two r <= v with r <= cap (1 if v < 2)
inline int pow2_floor_le(int v, int cap) {
  int r = 1;
  while (r * 2 <= v && r * 2 <= cap) r *= 2;
  return r;
}
// smallest l with 2^l >= v
inline int lg2_ceil(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

}  // namespace
