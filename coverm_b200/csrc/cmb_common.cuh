// Shared constants and PTX helpers of the libcoverm_b200 kernels (included inside an anonymous namespace).
#pragma once


constexpr uint32_t SPAN = 32;                   // elements per thread span; contig alignment
constexpr uint32_t K2_THREADS = 8192 / SPAN;
constexpr uint32_t CHUNK = SPAN * K2_THREADS;   // 8192 elements = 32 KB
constexpr uint32_t CHUNK_BYTES = CHUNK * 4;
constexpr uint32_t CHUNK_SPANS = K2_THREADS;    // spans per chunk
constexpr uint32_t ROW_ELEMS = 32;              // TMA row: 32 x i32 = 128 B
constexpr uint32_t CHUNK_ROWS = CHUNK / ROW_ELEMS;  // 256
#ifndef CMB_K2_STAGES
#define CMB_K2_STAGES 2
#endif
constexpr uint32_t K2_STAGES = CMB_K2_STAGES;
constexpr uint32_t K2_WARPS = K2_THREADS / 32;  // 16
#ifndef CMB_HIST_SLOTS
#define CMB_HIST_SLOTS 8
#endif
#ifndef CMB_K2_MINBLOCKS
#define CMB_K2_MINBLOCKS 3
#endif
constexpr uint32_t HIST_SLOTS = CMB_HIST_SLOTS;             // contigs per chunk with a shared-memory histogram
constexpr uint32_t HIST_BINS = 128;             // direct-mapped bins per slot: bin = depth % 128, word = tag|count
constexpr uint32_t HIST_TOTAL = HIST_SLOTS * HIST_BINS;  // 2048
constexpr uint32_t HIST_CNT_BITS = 14;          // a chunk holds 8192 = 2^13 positions, so a count fits 14 bits
constexpr uint32_t HIST_MAX_DEPTH = ((1u << (32 - HIST_CNT_BITS)) - 2) * HIST_BINS;  // deeper runs use the overflow list
constexpr uint32_t OVF_NIL = 0xffffffffu;
constexpr uint32_t K1_THREADS = 256;
constexpr uint32_t ROWFLAG_OVF = 1u;            // cmb_contig_stats.reserved: some records are in the overflow list

// error_flags bits (device)
constexpr uint32_t ERR_UNSORTED = 1u, ERR_NM = 2u, ERR_BOUNDS = 4u, ERR_CAPACITY = 8u, ERR_TID = 16u, ERR_INTERNAL = 32u;

#define FULL 0xffffffffu

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// TMA: 2-D tiled bulk tensor load global -> shared, completion on an mbarrier.
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tmap, int32_t x, int32_t y, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(bar)
      : "memory");
}

__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
  return v;
}

