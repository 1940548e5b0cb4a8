// libcoverm_b200 — device side: hand-written sm_100a kernels + the C ABI of include/coverm_b200.h.
//
// Data layout in HBM (one cmb_ctx = one GPU = one contig shard):
//   arena        i32[arena_elems]   all contigs' `ups_and_downs` (contig.rs:144-145) back to back; every contig
//                                   starts on a 32-element span boundary (SPAN), the arena is a whole number of
//                                   8192-element chunks (CHUNK).  4 B per reference base.
//   off_span     u32[n_local+1]     padded contig offsets in span units; len u32[n_local]
//   chunk_first  u32[n_chunks+1]    contig containing the first span of each chunk
//   tail_sum     i32[n_chunks]      K1: sum of the deltas of the contig that continues past the chunk end
//   carry_in     i32[n_chunks]      K1b: running depth at the first element of each chunk
//   rows         cmb_contig_stats[n_contigs]
//   rec / warp_table / ovf          K2 -> K3 histogram records
//
// Kernels (all HBM-bound integer work, no tensor cores):
//   K1  k1_filter_accumulate  one thread per record: FlagFilter + ReferenceSortedBamFilter predicates
//                             (lib.rs:59-79, filter.rs:243-336), per-contig read counters (contig.rs:157-211),
//                             +1/-1 delta REDs into the arena (contig.rs:166-202), chunk tail sums.
//   K1b k1b_chunk_carry       segmented scan of the per-chunk tail sums -> carry_in (so K2 needs no look-back).
//   K2  k2_scan_reduce        persistent CTAs, TMA (cp.async.bulk.tensor, 128B swizzle) + mbarrier ring of 32 KB
//                             chunks, blocked 32-element spans per thread, warp-shuffle segmented scan, then every
//                             O(L) reduction of EST:366-502 in one pass: sum/covered over the end-trimmed window,
//                             covered over the full contig, window depth histogram into a shared-memory table that
//                             is flushed as (depth,count) records; optionally re-zeroes the arena as it goes.
//   K3  k3_finalize           per contig: merge the records, trimmed-mean walk (EST:598-642) and the variance sums
//                             (EST:790-805) in integers; optional CSR histogram output.
//   KD* kd_inflate ...        device-side BAM decode behind cmb_submit_bgzf (cmb_decode.cuh): BGZF inflate, record chain,
//                             tuple extraction -- the compressed file crosses PCIe instead of tuples.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <nccl.h>
#include <nvtx3/nvToolsExt.h>
#include <strings.h>
#include <unistd.h>
#include <zlib.h>

#include "../../include/coverm_b200.h"

// NVTX ranges around the entry points and the stages of the device decode (visible in Nsight Systems / `ncu --nvtx`; no-ops
// without a tool attached: nvtx3 is header-only and resolves its injection library lazily).
struct NvtxRange {
  bool open = true;
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  void end() {
    if (open) {
      nvtxRangePop();
      open = false;
    }
  }
  ~NvtxRange() { end(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

namespace {
#include "cmb_common.cuh"
#include "cmb_k1.cuh"
#include "cmb_k1b.cuh"
#include "cmb_k2.cuh"
#include "cmb_k3.cuh"
#include "cmb_decode.cuh"
#include "cmb_decode_g8.cuh"
#include "cmb_decode_t1.cuh"
#include "cmb_pairs.cuh"
#include "cmb_filter.cuh"

// rows[i].hist_offset += base for the rows that carry histogram pairs (cmb_allgather_stats: local -> global pair offsets)
__global__ void __launch_bounds__(256) k_rebase_hist_offsets(cmb_contig_stats* rows, uint32_t n, uint64_t base) {
  const uint32_t i = blockIdx.x * 256 + threadIdx.x;
  if (i < n && rows[i].hist_count) rows[i].hist_offset += base;
}

// ------------------------------------------------------------------------------------------------ host context
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

std::string g_create_error;

// Ranks that live in ONE process (cmb_comm_init_local) meet here before every collective: a rank must not be inside a CUDA call
// that synchronises across devices (cudaHostAlloc, cudaMalloc, cudaFree ...) while another rank's NCCL kernel is already
// waiting for it -- that is the classic single-process multi-GPU deadlock.  All allocation happens before the barrier, only
// stream-ordered work after it.
struct LocalBarrier {
  std::mutex m;
  std::condition_variable cv;
  int n = 0, waiting = 0;
  uint64_t generation = 0;
  void arrive_and_wait() {
    std::unique_lock<std::mutex> lk(m);
    const uint64_t g = generation;
    if (++waiting == n) {
      waiting = 0;
      ++generation;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != g; });
    }
  }
};

struct DevBatch {  // device mirror of one staging batch
  void* slab = nullptr;
  cmb_read_batch ptr{};
};

}  // namespace

struct cmb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  cmb_device_cfg cfg{};
  int sm_count = 0;
  // staging
  std::vector<void*> host_slab;
  std::vector<cmb_read_batch> host_batch;
  std::vector<DevBatch> dev_batch;
  std::vector<cudaEvent_t> batch_done;
  std::vector<bool> batch_busy;
  uint32_t n_acquired = 0;   // staging batches handed out and not yet submitted (FIFO)
  uint32_t next_batch = 0;   // next staging slot to hand out
  // reference
  uint32_t n_contigs = 0, tid_begin = 0, tid_end = 0, n_local = 0;
  uint64_t arena_elems = 0;
  uint32_t n_chunks = 0;
  int32_t* d_arena = nullptr;
  uint32_t *d_off_span = nullptr, *d_len = nullptr, *d_chunk_first = nullptr;
  int32_t *d_tail_sum = nullptr, *d_carry_in = nullptr;
  int2* d_block_agg = nullptr;
  cmb_contig_stats* d_rows = nullptr;
  uint32_t* d_counters = nullptr;  // [0] error flags, [1] unused, [2] rec_count, [3] ovf_count, [4..5] pair_count (u64),
                                   // [6..7] kept tid range of the exclusive records (K1Args::kept_range)
  uint32_t kept_range[2] = {0, 0};  // host copy after cmb_end_sample*
  // multi-GPU (cmb_comm_*): one NCCL communicator per ctx, collectives on the ctx stream
  ncclComm_t comm = nullptr;
  int comm_rank = 0, comm_size = 1;
  std::shared_ptr<LocalBarrier> local_barrier;  // set when all ranks of the communicator live in this process
  uint8_t* d_xchg = nullptr;  // staging of cmb_comm_allgather
  size_t xchg_cap = 0;
  cmb_hist_pair* d_pairs_all = nullptr;  // concatenated histogram pairs of all ranks (cmb_allgather_stats)
  uint64_t pairs_all_capacity = 0;
  uint2* d_rec = nullptr;
  uint32_t rec_capacity = 0;
  uint2* d_warp_table = nullptr;
  uint4* d_ovf = nullptr;
  uint32_t* d_ovf_head = nullptr;
  uint32_t ovf_capacity = 0;
  cmb_hist_pair* d_pairs = nullptr;
  uint64_t pair_capacity = 0;
  int2* d_block_minmax = nullptr;
  int2* d_block_xrange = nullptr;  // same capacity as d_block_minmax
  bool have_xrange = false;
  uint32_t block_minmax_capacity = 0, block_minmax_used = 0;
  // gene mode (cmb_set_genes): segments are genes; records carry contig tids
  bool gene_mode = false;
  uint32_t n_ref_contigs = 0;  // contigs of the BAM header (== n_contigs outside gene mode)
  uint32_t *d_gene_first = nullptr, *d_gene_start = nullptr, *d_gene_end = nullptr, *d_gene_maxlen = nullptr, *d_contig_len32 = nullptr;
  uint8_t* d_contig_seen = nullptr;
  CUtensorMap tmap{};
  bool arena_dirty = true;  // cmb_begin_sample must zero the arena: only a completed K2 leaves it clean
  // params
  cmb_params params{};
  cmb_filter_mode mode{};
  bool have_params = false, in_sample = false, ended = false;
  // timing
  cudaEvent_t ev[8]{};
  cmb_sample_timing timing{};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> k1_events;
  uint32_t k1_events_used = 0;
  uint64_t n_records = 0, n_intervals = 0;
  // device-side decode (cmb_submit_bgzf); every buffer is grow-only and reused across samples
  struct Decode {
    uint8_t* d_comp = nullptr;
    size_t comp_cap = 0;
    uint8_t* d_inflated = nullptr;
    size_t infl_cap = 0;
    uint64_t *d_coff = nullptr, *d_ustart = nullptr, *d_guess = nullptr, *d_exit = nullptr, *d_rec_base = nullptr, *d_cig_base = nullptr;
    uint32_t *d_clen = nullptr, *d_isize = nullptr, *d_status = nullptr, *d_nrec = nullptr, *d_ncig = nullptr, *d_dirty = nullptr;
    size_t blocks_cap = 0;
    uint8_t* d_t1_scratch = nullptr;  // kd_inflate_t1: code-length scratch, 160 B per block
    uint32_t* d_tickets = nullptr;  // [0] block ticket, [1 + w] arrival flag: window w has been copied
    size_t tickets_cap = 0;
    uint32_t* d_block_window = nullptr;
    size_t block_window_cap = 0;
    uint32_t* h_ones = nullptr;  // pinned source of the arrival flags
    uint32_t* d_cnt = nullptr;  // [0] inflate failures [1] decode error bits [2] chain changed [4..5] n_primary [6..9] totals
    uint64_t* d_rec_off = nullptr;
    size_t rec_cap = 0;
    void* d_tuple_slab = nullptr;
    size_t tuple_slab_bytes = 0;
    uint32_t last_n_rec = 0, last_n_cig = 0;  // tuples of the last successful cmb_submit_bgzf (cmb_last_bgzf_batch)
    bool last_valid = false;
    // mate matching (cmb_pairs.cuh)
    uint64_t* d_pair_key = nullptr;
    int32_t* d_pair_mate = nullptr;
    uint32_t* d_pair_next = nullptr;
    size_t pair_rec_cap = 0;
    unsigned long long* d_pair_tag = nullptr;
    uint32_t* d_pair_head = nullptr;
    size_t pair_table_cap = 0;
    const int32_t* last_mate = nullptr;
    uint32_t last_excl_n = 0xffffffffu;
    const uint8_t* last_infl_base = nullptr;  // biased base of the inflated stream of the last decode
    // coverm filter
    unsigned long long* d_filter_anchor = nullptr;
    uint8_t* d_filter_role = nullptr;
    size_t filter_rec_cap = 0;
    uint8_t* d_filter_out = nullptr;
    size_t filter_out_cap = 0;
    uint64_t filter_bytes = 0;
    bool filter_planned = false;
    std::vector<void*> pinned;
    std::vector<cudaStream_t> streams;
    std::vector<cudaEvent_t> slot_events, done_events;
    cudaEvent_t ev[6]{};
    bool have_events = false;
  } dec;
};

namespace {

int fail(cmb_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  else g_create_error = buf;
  return code;
}

#define CU_TRY(ctx, expr)                                                                                   \
  do {                                                                                                      \
    cudaError_t e_ = (expr);                                                                                \
    if (e_ != cudaSuccess) return fail(ctx, e_ == cudaErrorMemoryAllocation ? CMB_E_NOMEM : CMB_E_CUDA,      \
                                       "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

size_t batch_slab_bytes(uint32_t nr, uint32_t ni, size_t* offs) {
  // column order: tid,pos,nm,l_seq,aligned,del,ins,iv_begin(nr+1),iv_start(ni),iv_len(ni),flag(u16),mapq(u8),nm_state(u8)
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t r = o;
    o += (bytes + 255) & ~(size_t)255;
    return r;
  };
  offs[0] = take(4ull * nr);        // tid
  offs[1] = take(4ull * nr);        // pos
  offs[2] = take(4ull * nr);        // nm
  offs[3] = take(4ull * nr);        // l_seq
  offs[4] = take(4ull * nr);        // aligned
  offs[5] = take(4ull * nr);        // del
  offs[6] = take(4ull * nr);        // ins
  offs[7] = take(4ull * (nr + 1));  // iv_begin
  offs[8] = take(4ull * ni);        // iv_start
  offs[9] = take(4ull * ni);        // iv_len
  offs[10] = take(2ull * nr);       // flag
  offs[11] = take(1ull * nr);       // mapq
  offs[12] = take(1ull * nr);       // nm_state
  return o;
}

void carve_batch(void* slab, uint32_t nr, uint32_t ni, cmb_read_batch* b) {
  size_t offs[13];
  batch_slab_bytes(nr, ni, offs);
  uint8_t* p = (uint8_t*)slab;
  b->capacity_records = nr;
  b->capacity_intervals = ni;
  b->tid = (int32_t*)(p + offs[0]);
  b->pos = (int32_t*)(p + offs[1]);
  b->nm = (uint32_t*)(p + offs[2]);
  b->l_seq = (uint32_t*)(p + offs[3]);
  b->aligned = (uint32_t*)(p + offs[4]);
  b->del = (uint32_t*)(p + offs[5]);
  b->ins = (uint32_t*)(p + offs[6]);
  b->iv_begin = (uint32_t*)(p + offs[7]);
  b->iv_start = (int32_t*)(p + offs[8]);
  b->iv_len = (int32_t*)(p + offs[9]);
  b->flag = (uint16_t*)(p + offs[10]);
  b->mapq = (uint8_t*)(p + offs[11]);
  b->nm_state = (uint8_t*)(p + offs[12]);
}

void free_reference(cmb_ctx* c) {
  cudaFree(c->d_arena);
  cudaFree(c->d_off_span);
  cudaFree(c->d_len);
  cudaFree(c->d_chunk_first);
  cudaFree(c->d_tail_sum);
  cudaFree(c->d_carry_in);
  cudaFree(c->d_block_agg);
  c->d_block_agg = nullptr;
  cudaFree(c->d_rows);
  cudaFree(c->d_rec);
  cudaFree(c->d_warp_table);
  cudaFree(c->d_ovf);
  cudaFree(c->d_ovf_head);
  c->d_ovf_head = nullptr;
  cudaFree(c->d_pairs);
  cudaFree(c->d_gene_first); cudaFree(c->d_gene_start); cudaFree(c->d_gene_end); cudaFree(c->d_gene_maxlen); cudaFree(c->d_contig_len32);
  cudaFree(c->d_contig_seen);
  c->d_gene_first = c->d_gene_start = c->d_gene_end = c->d_gene_maxlen = c->d_contig_len32 = nullptr;
  c->d_contig_seen = nullptr;
  c->gene_mode = false;
  c->d_arena = nullptr;
  c->d_off_span = c->d_len = c->d_chunk_first = nullptr;
  c->d_tail_sum = c->d_carry_in = nullptr;
  c->d_rows = nullptr;
  c->d_rec = nullptr;
  c->d_warp_table = nullptr;
  c->d_ovf = nullptr;
  c->d_pairs = nullptr;
  c->pair_capacity = 0;
}

int launch_k1(cmb_ctx* c, const cmb_read_batch& b, uint32_t n_records, uint32_t n_intervals, uint32_t excl_n = 0xffffffffu,
              const int32_t* mate = nullptr) {
  if (n_records == 0) return CMB_OK;
  const uint32_t blocks = (n_records + K1_THREADS - 1) / K1_THREADS;
  if (c->block_minmax_used + blocks > c->block_minmax_capacity) {
    // grow (rare): allocate a larger array and copy what is there
    uint32_t ncap = std::max(c->block_minmax_capacity * 2, c->block_minmax_used + blocks + 4096);
    int2 *nd = nullptr, *nx = nullptr;
    CU_TRY(c, cudaMalloc(&nd, sizeof(int2) * (size_t)ncap));
    CU_TRY(c, cudaMalloc(&nx, sizeof(int2) * (size_t)ncap));
    if (c->block_minmax_used) {
      CU_TRY(c, cudaMemcpyAsync(nd, c->d_block_minmax, sizeof(int2) * (size_t)c->block_minmax_used, cudaMemcpyDeviceToDevice, c->stream));
      CU_TRY(c, cudaMemcpyAsync(nx, c->d_block_xrange, sizeof(int2) * (size_t)c->block_minmax_used, cudaMemcpyDeviceToDevice, c->stream));
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_block_minmax);
    cudaFree(c->d_block_xrange);
    c->d_block_minmax = nd;
    c->d_block_xrange = nx;
    c->block_minmax_capacity = ncap;
  }
  K1Args a{};
  a.tid = b.tid; a.pos = b.pos; a.flag = b.flag; a.mapq = b.mapq; a.nm_state = b.nm_state; a.nm = b.nm;
  a.l_seq = b.l_seq; a.aligned = b.aligned; a.del = b.del; a.ins = b.ins; a.iv_begin = b.iv_begin;
  a.iv_start = b.iv_start; a.iv_len = b.iv_len;
  a.n = n_records;
  a.off_span = c->d_off_span; a.len = c->d_len;
  a.n_contigs = c->gene_mode ? c->n_ref_contigs : c->n_contigs; a.tid_begin = c->tid_begin; a.tid_end = c->tid_end;
  if (c->gene_mode) {
    a.gene_first = c->d_gene_first; a.gene_start = c->d_gene_start; a.gene_end = c->d_gene_end; a.gene_maxlen = c->d_gene_maxlen;
    a.contig_len = c->d_contig_len32; a.contig_seen = c->d_contig_seen; a.kept_primary = (unsigned long long*)(c->d_counters + 8);
  }
  a.arena = c->d_arena; a.tail_sum = c->d_tail_sum; a.rows = c->d_rows;
  a.block_minmax = c->d_block_minmax + c->block_minmax_used;
  a.error_flags = c->d_counters + 0;
  a.block_xrange = c->comm_size > 1 || excl_n != 0xffffffffu ? c->d_block_xrange + c->block_minmax_used : nullptr;
  a.excl_n = excl_n;
  if (a.block_xrange) c->have_xrange = true;
  a.mate = mate;
  a.p = c->params;
  a.filter_single = c->mode.filter_single_reads;
  a.filter_pairs = c->mode.filter_pairs;
  if (c->k1_events_used == c->k1_events.size()) {
    cudaEvent_t e0, e1;
    CU_TRY(c, cudaEventCreate(&e0));
    CU_TRY(c, cudaEventCreate(&e1));
    c->k1_events.emplace_back(e0, e1);
  }
  auto& ev = c->k1_events[c->k1_events_used++];
  CU_TRY(c, cudaEventRecord(ev.first, c->stream));
  k1_filter_accumulate<<<blocks, K1_THREADS, 0, c->stream>>>(a);
  CU_TRY(c, cudaGetLastError());
  CU_TRY(c, cudaEventRecord(ev.second, c->stream));
  c->block_minmax_used += blocks;
  c->n_records += n_records;
  c->n_intervals += n_intervals;
  c->timing.k1_launches += 1;
  return CMB_OK;
}

template <bool HIST>
int launch_k2_variant(cmb_ctx* c, const K2Args& a) {
  auto kern = k2_scan_reduce<HIST>;
  constexpr uint32_t smem_bytes = HIST ? K2_SMEM_BYTES_HIST : K2_SMEM_BYTES_NOHIST;
  CU_TRY(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  int occ = 0;
  CU_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, (int)K2_THREADS, smem_bytes));
  if (occ < 1) return fail(c, CMB_E_CUDA, "k2_scan_reduce does not fit on an SM");
  const uint32_t grid = std::min<uint32_t>(c->n_chunks, (uint32_t)(occ * c->sm_count));
  kern<<<grid, K2_THREADS, smem_bytes, c->stream>>>(c->tmap, a);
  CU_TRY(c, cudaGetLastError());
  return CMB_OK;
}

int run_end_of_sample(cmb_ctx* c) {
  const bool hist = c->params.want & (CMB_WANT_HIST | CMB_WANT_HIST_CSR);
  const bool csr = c->params.want & CMB_WANT_HIST_CSR;
  const uint32_t excl = (uint32_t)std::min<uint64_t>(c->params.contig_end_exclusion, 0x7fffffffu);
  CU_TRY(c, cudaEventRecord(c->ev[2], c->stream));
  if (c->block_minmax_used) {
    k1c_check_sorted<<<1, 1024, 0, c->stream>>>(c->d_block_minmax, c->block_minmax_used, c->d_counters + 0,
                                                c->have_xrange ? c->d_block_xrange : nullptr, c->d_counters + 6);
    CU_TRY(c, cudaGetLastError());
  }
  {
    const uint32_t blocks = (c->n_chunks + K1B_BLOCK - 1) / K1B_BLOCK;
    k1b_local<<<blocks, K1B_THREADS, 0, c->stream>>>(c->d_tail_sum, c->d_chunk_first, c->d_off_span, c->n_chunks, c->d_carry_in, c->d_block_agg);
    CU_TRY(c, cudaGetLastError());
    k1b_apply<<<blocks, K1B_THREADS, 0, c->stream>>>(c->d_tail_sum, c->d_block_agg, c->n_chunks, c->d_carry_in);
    CU_TRY(c, cudaGetLastError());
  }
  K2Args a{};
  a.off_span = c->d_off_span; a.len = c->d_len; a.chunk_first = c->d_chunk_first; a.carry_in = c->d_carry_in;
  a.rows = c->d_rows; a.tid_begin = c->tid_begin; a.n_local = c->n_local; a.n_chunks = c->n_chunks; a.excl = excl;
  a.arena = c->d_arena;
  a.rec = c->d_rec; a.rec_capacity = c->rec_capacity; a.rec_count = c->d_counters + 2;
  a.warp_table = c->d_warp_table; a.ovf = c->d_ovf; a.ovf_head = c->d_ovf_head; a.ovf_capacity = c->ovf_capacity; a.ovf_count = c->d_counters + 3;
  a.error_flags = c->d_counters + 0;
  if (hist) CU_TRY(c, cudaMemsetAsync(c->d_ovf_head, 0xff, 4ull * c->n_chunks, c->stream));
  CU_TRY(c, cudaEventRecord(c->ev[3], c->stream));
  const int rc = hist ? launch_k2_variant<true>(c, a) : launch_k2_variant<false>(c, a);
  if (rc) return rc;
  c->timing.k2_launches = 1;
  c->arena_dirty = false;  // K2 re-zeroed every delta it read
  CU_TRY(c, cudaEventRecord(c->ev[4], c->stream));
  if (hist) {
    K3Args k{};
    k.off_span = c->d_off_span; k.len = c->d_len; k.chunk_first = c->d_chunk_first; k.rows = c->d_rows;
    k.tid_begin = c->tid_begin; k.n_local = c->n_local; k.excl = excl;
    k.trim_min = c->params.trim_min; k.trim_max = c->params.trim_max;
    k.rec = c->d_rec; k.warp_table = c->d_warp_table; k.ovf = c->d_ovf; k.ovf_head = c->d_ovf_head;
    k.ovf_capacity = c->ovf_capacity;
    k.pairs = c->d_pairs; k.pair_count = (unsigned long long*)(c->d_counters + 4); k.pair_capacity = c->pair_capacity;
    k.want_csr = csr; k.all_rows = c->gene_mode ? 1u : 0u; k.error_flags = c->d_counters + 0;
    const uint32_t grid = (c->n_local + K3_WARPS - 1) / K3_WARPS;  // one warp per contig
    k3_finalize<<<grid, K3_THREADS, 0, c->stream>>>(k);
    CU_TRY(c, cudaGetLastError());
    c->timing.k3_launches = 1;
  }
  CU_TRY(c, cudaEventRecord(c->ev[5], c->stream));
  return CMB_OK;
}

int collect_errors_and_timing(cmb_ctx* c, uint32_t* counters_out) {
  uint32_t h[8];
  CU_TRY(c, cudaMemcpyAsync(h, c->d_counters, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaEventRecord(c->ev[6], c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  memcpy(counters_out, h, 6 * sizeof(uint32_t));
  c->kept_range[0] = h[6];
  c->kept_range[1] = h[7];
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); c->timing.ms_zero = ms;
  cudaEventElapsedTime(&ms, c->ev[3], c->ev[4]); c->timing.ms_scan = ms;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->timing.ms_finalize = ms;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[6]); c->timing.ms_total = ms;
  float acc = 0;
  for (uint32_t i = 0; i < c->k1_events_used; ++i) {
    cudaEventElapsedTime(&ms, c->k1_events[i].first, c->k1_events[i].second);
    acc += ms;
  }
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);  // k1c + k1b
  c->timing.ms_accumulate = acc + ms;
  c->timing.arena_elems = c->arena_elems;
  c->timing.n_records = c->n_records;
  c->timing.n_intervals = c->n_intervals;
  const uint32_t e = h[0];
  if (e) c->arena_dirty = true;
  if (e & ERR_UNSORTED)
    return fail(c, CMB_E_UNSORTED, "BAM file appears to be unsorted. Input BAM files must be sorted by reference (i.e. by samtools sort)");
  if (e & ERR_NM)
    return fail(c, CMB_E_NM, "Mapping record encountered that does not have an 'NM' auxiliary tag in the SAM/BAM format. This is required to work out some coverage statistics");
  if (e & (ERR_BOUNDS | ERR_TID)) return fail(c, CMB_E_BOUNDS, "index out of bounds: an aligned block starts beyond the end of its reference sequence");
  if (e & ERR_CAPACITY) return fail(c, CMB_E_CAPACITY, "device histogram record buffer overflowed");
  if (e & ERR_INTERNAL) return fail(c, CMB_E_CUDA, "internal error: negative running depth (inconsistent delta arena)");
  return CMB_OK;
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

int cmb_abi_version(void) { return CMB_ABI_VERSION; }

const char* cmb_last_error(const cmb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int cmb_create(const cmb_device_cfg* cfg, cmb_ctx** out) {
  NvtxRange nvtx_fn("cmb_create");
  if (!cfg || !out) return fail(nullptr, CMB_E_ARG, "cmb_create: null argument");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, CMB_E_CUDA, "cmb_create: no usable CUDA device (%s); libcoverm_b200 has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= n_dev) return fail(nullptr, CMB_E_ARG, "cmb_create: device %d out of range", cfg->device);
  cmb_ctx* c = new cmb_ctx();
  c->device = cfg->device;
  c->cfg = *cfg;
  if (c->cfg.batch_records == 0) c->cfg.batch_records = 1u << 20;
  if (c->cfg.batch_intervals == 0) c->cfg.batch_intervals = c->cfg.batch_records + c->cfg.batch_records / 2;
  if (c->cfg.n_staging < 2) c->cfg.n_staging = 2;
  auto bail = [&](int code) {
    g_create_error = c->err;
    cmb_destroy(c);
    return code;
  };
#define CREATE_TRY(expr)                                                                           \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      fail(c, CMB_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_));                         \
      return bail(e_ == cudaErrorMemoryAllocation ? CMB_E_NOMEM : CMB_E_CUDA);                     \
    }                                                                                              \
  } while (0)
  CREATE_TRY(cudaSetDevice(c->device));
  cudaDeviceProp prop;
  CREATE_TRY(cudaGetDeviceProperties(&prop, c->device));
  if (prop.major < 10) {
    fail(c, CMB_E_CUDA, "cmb_create: device %d is sm_%d%d; this library is built for sm_100a only", c->device, prop.major, prop.minor);
    return bail(CMB_E_CUDA);
  }
  c->sm_count = prop.multiProcessorCount;
  CREATE_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  for (auto& ev : c->ev) CREATE_TRY(cudaEventCreate(&ev));
  size_t offs[13];
  const size_t slab = batch_slab_bytes(c->cfg.batch_records, c->cfg.batch_intervals, offs);
  for (uint32_t i = 0; i < c->cfg.n_staging; ++i) {
    void* h = nullptr;
    CREATE_TRY(cudaHostAlloc(&h, slab, cudaHostAllocDefault));
    c->host_slab.push_back(h);
    cmb_read_batch hb;
    carve_batch(h, c->cfg.batch_records, c->cfg.batch_intervals, &hb);
    c->host_batch.push_back(hb);
    DevBatch db;
    CREATE_TRY(cudaMalloc(&db.slab, slab));
    carve_batch(db.slab, c->cfg.batch_records, c->cfg.batch_intervals, &db.ptr);
    c->dev_batch.push_back(db);
    cudaEvent_t ev;
    CREATE_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    c->batch_done.push_back(ev);
    c->batch_busy.push_back(false);
  }
  CREATE_TRY(cudaMalloc(&c->d_counters, 64));
  CREATE_TRY(cudaMemset(c->d_counters, 0, 64));
  c->block_minmax_capacity = 1u << 16;
  CREATE_TRY(cudaMalloc(&c->d_block_minmax, sizeof(int2) * (size_t)c->block_minmax_capacity));
  CREATE_TRY(cudaMalloc(&c->d_block_xrange, sizeof(int2) * (size_t)c->block_minmax_capacity));
  *out = c;
  return CMB_OK;
}

void cmb_destroy(cmb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  free_reference(c);
  for (auto h : c->host_slab) cudaFreeHost(h);
  for (auto& d : c->dev_batch) cudaFree(d.slab);
  for (auto e : c->batch_done) cudaEventDestroy(e);
  for (auto& e : c->k1_events) {
    cudaEventDestroy(e.first);
    cudaEventDestroy(e.second);
  }
  for (auto e : c->ev)
    if (e) cudaEventDestroy(e);
  cudaFree(c->d_counters);
  cudaFree(c->d_block_minmax);
  cudaFree(c->d_block_xrange);
  cmb_comm_destroy(c);
  cudaFree(c->d_xchg);
  cudaFree(c->d_pairs_all);
  {
    auto& d = c->dec;
    cudaFree(d.d_comp); cudaFree(d.d_inflated); cudaFree(d.d_coff); cudaFree(d.d_ustart); cudaFree(d.d_guess); cudaFree(d.d_exit);
    cudaFree(d.d_rec_base); cudaFree(d.d_cig_base); cudaFree(d.d_clen); cudaFree(d.d_isize); cudaFree(d.d_status); cudaFree(d.d_nrec);
    cudaFree(d.d_filter_anchor); cudaFree(d.d_filter_role); cudaFree(d.d_filter_out);
    cudaFree(d.d_pair_key); cudaFree(d.d_pair_mate); cudaFree(d.d_pair_next); cudaFree(d.d_pair_tag); cudaFree(d.d_pair_head);
    cudaFree(d.d_ncig); cudaFree(d.d_dirty); cudaFree(d.d_tickets); cudaFree(d.d_t1_scratch); cudaFree(d.d_block_window); if (d.h_ones) cudaFreeHost(d.h_ones); cudaFree(d.d_cnt); cudaFree(d.d_rec_off); cudaFree(d.d_tuple_slab);
    for (auto p : d.pinned) cudaFreeHost(p);
    for (auto st : d.streams) cudaStreamDestroy(st);
    for (auto e : d.slot_events) cudaEventDestroy(e);
    for (auto e : d.done_events) cudaEventDestroy(e);
    if (d.have_events)
      for (auto e : d.ev) cudaEventDestroy(e);
  }
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int cmb_set_genes(cmb_ctx* c, uint32_t n_contigs, const uint64_t* contig_len, uint32_t n_genes, const cmb_gene* genes) {
  if (!c || (!contig_len && n_contigs) || (!genes && n_genes)) return fail(c, CMB_E_ARG, "cmb_set_genes: null argument");
  if (c->in_sample) return fail(c, CMB_E_ARG, "cmb_set_genes: a sample is in progress");
  std::vector<uint64_t> seg_len(std::max<uint32_t>(1, n_genes), 1);
  std::vector<uint32_t> first((size_t)n_contigs + 1, 0), gs(std::max<uint32_t>(1, n_genes)), ge(std::max<uint32_t>(1, n_genes)), maxlen(std::max<uint32_t>(1, n_contigs), 0), clen(std::max<uint32_t>(1, n_contigs), 0);
  for (uint32_t t = 0; t < n_contigs; ++t) {
    if (contig_len[t] > 0x7fffffffull) return fail(c, CMB_E_ARG, "cmb_set_genes: contig %u longer than 2^31-1", t);
    clen[t] = (uint32_t)contig_len[t];
  }
  for (uint32_t g = 0; g < n_genes; ++g) {
    const cmb_gene& x = genes[g];
    if (x.tid >= n_contigs || x.start >= x.end || x.end > contig_len[x.tid]) return fail(c, CMB_E_ARG, "cmb_set_genes: gene %u is not a range of its contig", g);
    if (g && (genes[g - 1].tid > x.tid || (genes[g - 1].tid == x.tid && genes[g - 1].start > x.start)))
      return fail(c, CMB_E_ARG, "cmb_set_genes: genes must be sorted by (tid, start)");
    seg_len[g] = x.end - x.start;
    gs[g] = x.start;
    ge[g] = x.end;
    first[x.tid + 1] += 1;
    maxlen[x.tid] = std::max(maxlen[x.tid], x.end - x.start);
  }
  for (uint32_t t = 0; t < n_contigs; ++t) first[t + 1] += first[t];
  // the arena, rows and histogram buffers are laid out over the genes exactly as over contigs (a placeholder segment keeps an
  // empty gene set well-formed)
  const uint32_t n_seg = std::max<uint32_t>(1, n_genes);
  int rc = cmb_set_reference(c, n_seg, seg_len.data(), 0, n_seg);
  if (rc) return rc;
  c->gene_mode = true;
  c->n_ref_contigs = n_contigs;
  CU_TRY(c, cudaMalloc(&c->d_gene_first, 4ull * (n_contigs + 1)));
  CU_TRY(c, cudaMalloc(&c->d_gene_start, 4ull * n_seg));
  CU_TRY(c, cudaMalloc(&c->d_gene_end, 4ull * n_seg));
  CU_TRY(c, cudaMalloc(&c->d_gene_maxlen, 4ull * std::max<uint32_t>(1, n_contigs)));
  CU_TRY(c, cudaMalloc(&c->d_contig_len32, 4ull * std::max<uint32_t>(1, n_contigs)));
  CU_TRY(c, cudaMalloc(&c->d_contig_seen, std::max<size_t>(1, n_contigs)));
  CU_TRY(c, cudaMemcpyAsync(c->d_gene_first, first.data(), 4ull * (n_contigs + 1), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_gene_start, gs.data(), 4ull * n_seg, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_gene_end, ge.data(), 4ull * n_seg, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_gene_maxlen, maxlen.data(), 4ull * std::max<uint32_t>(1, n_contigs), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_contig_len32, clen.data(), 4ull * std::max<uint32_t>(1, n_contigs), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  return CMB_OK;
}

int cmb_fetch_gene_extras(cmb_ctx* c, uint8_t* contig_seen, uint64_t* n_kept_primary) {
  if (!c || !contig_seen || !n_kept_primary) return fail(c, CMB_E_ARG, "cmb_fetch_gene_extras: null argument");
  if (!c->gene_mode || !c->ended) return fail(c, CMB_E_ARG, "cmb_fetch_gene_extras: no ended sample in gene mode");
  CU_TRY(c, cudaSetDevice(c->device));
  unsigned long long kp = 0;
  if (c->n_ref_contigs) CU_TRY(c, cudaMemcpyAsync(contig_seen, c->d_contig_seen, c->n_ref_contigs, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaMemcpyAsync(&kp, c->d_counters + 8, 8, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  *n_kept_primary = kp;
  return CMB_OK;
}

int cmb_set_reference(cmb_ctx* c, uint32_t n_contigs, const uint64_t* contig_len, uint32_t tid_begin, uint32_t tid_end) {
  if (!c || !contig_len || tid_begin > tid_end || tid_end > n_contigs) return fail(c, CMB_E_ARG, "cmb_set_reference: bad arguments");
  if (c->in_sample) return fail(c, CMB_E_ARG, "cmb_set_reference: a sample is in progress");
  CU_TRY(c, cudaSetDevice(c->device));
  free_reference(c);
  c->n_contigs = n_contigs;
  c->n_ref_contigs = n_contigs;
  c->tid_begin = tid_begin;
  c->tid_end = tid_end;
  c->n_local = tid_end - tid_begin;
  std::vector<uint32_t> off_span(c->n_local + 1), len(c->n_local);
  uint64_t spans = 0;
  for (uint32_t i = 0; i < c->n_local; ++i) {
    const uint64_t L = contig_len[tid_begin + i];
    if (L > 0x7fffffffull) return fail(c, CMB_E_ARG, "cmb_set_reference: contig %u longer than 2^31-1", tid_begin + i);
    off_span[i] = (uint32_t)spans;
    len[i] = (uint32_t)L;
    spans += std::max<uint64_t>(1, (L + SPAN - 1) / SPAN);
    if (spans > 0xfffffff0ull) return fail(c, CMB_E_ARG, "cmb_set_reference: shard larger than 2^36 bases; use more shards");
  }
  off_span[c->n_local] = (uint32_t)spans;
  const uint64_t chunks = std::max<uint64_t>(1, (spans + CHUNK_SPANS - 1) / CHUNK_SPANS);
  c->n_chunks = (uint32_t)chunks;
  c->arena_elems = chunks * CHUNK;
  std::vector<uint32_t> chunk_first(c->n_chunks + 1);
  {
    uint32_t ci = 0;
    for (uint32_t k = 0; k < c->n_chunks; ++k) {
      const uint64_t s = (uint64_t)k * CHUNK_SPANS;
      while (ci + 1 < c->n_local && off_span[ci + 1] <= s) ++ci;
      chunk_first[k] = ci;
    }
    chunk_first[c->n_chunks] = c->n_local ? c->n_local - 1 : 0;
  }
  if (c->n_local == 0) {  // empty shard: nothing to allocate beyond the rows
    CU_TRY(c, cudaMalloc(&c->d_rows, sizeof(cmb_contig_stats) * std::max<size_t>(1, n_contigs)));
    return CMB_OK;
  }
  CU_TRY(c, cudaMalloc(&c->d_arena, c->arena_elems * 4));
  CU_TRY(c, cudaMalloc(&c->d_off_span, 4ull * (c->n_local + 1)));
  CU_TRY(c, cudaMalloc(&c->d_len, 4ull * c->n_local));
  CU_TRY(c, cudaMalloc(&c->d_chunk_first, 4ull * (c->n_chunks + 1)));
  CU_TRY(c, cudaMalloc(&c->d_tail_sum, 4ull * c->n_chunks));
  CU_TRY(c, cudaMalloc(&c->d_carry_in, 4ull * c->n_chunks));
  CU_TRY(c, cudaMalloc(&c->d_block_agg, sizeof(int2) * ((size_t)c->n_chunks / K1B_BLOCK + 1)));
  CU_TRY(c, cudaMalloc(&c->d_rows, sizeof(cmb_contig_stats) * (size_t)n_contigs));
  CU_TRY(c, cudaMemcpyAsync(c->d_off_span, off_span.data(), 4ull * (c->n_local + 1), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_len, len.data(), 4ull * c->n_local, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(c->d_chunk_first, chunk_first.data(), 4ull * (c->n_chunks + 1), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  // histogram record buffers: one 8 B record per 8 arena elements is far above anything a real sample produces
  c->rec_capacity = (uint32_t)std::min<uint64_t>(0xfffffff0ull, std::max<uint64_t>(1u << 20, c->arena_elems / 8));
  c->ovf_capacity = (uint32_t)std::min<uint64_t>(1u << 26, std::max<uint64_t>(1u << 20, c->arena_elems / 64));
  if (getenv("CMB_TEST_SMALL_HIST")) {  // testing aid: buffers that overflow at once (cmb_grow_buffers path)
    c->rec_capacity = 256;
    c->ovf_capacity = 64;
  }
  CU_TRY(c, cudaMalloc(&c->d_rec, 8ull * c->rec_capacity));
  CU_TRY(c, cudaMalloc(&c->d_warp_table, 8ull * c->n_chunks * HIST_SLOTS));
  CU_TRY(c, cudaMalloc(&c->d_ovf, 16ull * c->ovf_capacity));
  CU_TRY(c, cudaMalloc(&c->d_ovf_head, 4ull * c->n_chunks));
  c->arena_dirty = true;
  // TMA descriptor: the arena as [rows][32] i32, box = one chunk (256 rows x 128 B), 128B swizzle
  PFN_encodeTiled encode = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CU_TRY(c, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&encode, cudaEnableDefault, &qres));
  if (!encode || qres != cudaDriverEntryPointSuccess) return fail(c, CMB_E_CUDA, "cuTensorMapEncodeTiled not available in this driver");
  cuuint64_t gdim[2] = {ROW_ELEMS, c->arena_elems / ROW_ELEMS};
  cuuint64_t gstride[1] = {ROW_ELEMS * 4};
  cuuint32_t box[2] = {ROW_ELEMS, CHUNK_ROWS};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(&c->tmap, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, c->d_arena, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, CMB_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return CMB_OK;
}

int cmb_set_params(cmb_ctx* c, const cmb_params* p, cmb_filter_mode* mode_out) {
  if (!c || !p) return fail(c, CMB_E_ARG, "cmb_set_params: null argument");
  if (c->in_sample) return fail(c, CMB_E_ARG, "cmb_set_params: a sample is in progress");
  c->params = *p;
  // filter.rs:48-61
  const bool single_initial = p->min_aligned_length_single > 0 || p->min_percent_identity_single > 0.0f || p->min_aligned_percent_single > 0.0f;
  const bool pairs_initial = p->min_aligned_length_pair > 0 || p->min_percent_identity_pair > 0.0f || p->min_aligned_percent_pair > 0.0f;
  const bool fs = single_initial || (!pairs_initial && p->min_mapq != 255);
  const bool fp = pairs_initial || ((!fs || !p->include_improper_pairs) && p->min_mapq != 255);
  c->mode.filter_single_reads = p->filtering ? fs : 0;
  c->mode.filter_pairs = p->filtering ? fp : 0;
  if (mode_out) *mode_out = c->mode;
  c->have_params = true;
  return CMB_OK;
}

int cmb_begin_sample(cmb_ctx* c) {
  NvtxRange nvtx_fn("cmb_begin_sample");
  if (!c) return CMB_E_ARG;
  if (!c->d_rows || !c->have_params) return fail(c, CMB_E_ARG, "cmb_begin_sample: set_reference and set_params first");
  if (c->in_sample) return fail(c, CMB_E_ARG, "cmb_begin_sample: previous sample not ended");
  CU_TRY(c, cudaSetDevice(c->device));
  c->timing = cmb_sample_timing{};
  c->k1_events_used = 0;
  c->block_minmax_used = 0;
  c->have_xrange = false;
  c->n_records = c->n_intervals = 0;
  CU_TRY(c, cudaEventRecord(c->ev[0], c->stream));
  if (c->n_local) {
    if (c->arena_dirty) CU_TRY(c, cudaMemsetAsync(c->d_arena, 0, c->arena_elems * 4, c->stream));
    CU_TRY(c, cudaMemsetAsync(c->d_tail_sum, 0, 4ull * c->n_chunks, c->stream));
  }
  CU_TRY(c, cudaMemsetAsync(c->d_rows, 0, sizeof(cmb_contig_stats) * (size_t)c->n_contigs, c->stream));
  CU_TRY(c, cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
  if (c->gene_mode) CU_TRY(c, cudaMemsetAsync(c->d_contig_seen, 0, std::max<size_t>(1, c->n_ref_contigs), c->stream));
  CU_TRY(c, cudaEventRecord(c->ev[1], c->stream));
  c->arena_dirty = true;  // until K2 has cleaned it
  if ((c->params.want & CMB_WANT_HIST_CSR) && c->n_local) {
    uint64_t want = std::max<uint64_t>(1u << 20, c->arena_elems / 16);
    if (getenv("CMB_TEST_SMALL_HIST")) want = 64;  // testing aid: start with buffers that overflow at once (cmb_grow_buffers path)
    if (c->pair_capacity < want) {
      cudaFree(c->d_pairs);
      c->d_pairs = nullptr;
      c->pair_capacity = 0;
      CU_TRY(c, cudaMalloc(&c->d_pairs, sizeof(cmb_hist_pair) * want));
      c->pair_capacity = want;
    }
  }
  c->in_sample = true;
  c->ended = false;
  c->n_acquired = 0;
  return CMB_OK;
}

int cmb_acquire_batch(cmb_ctx* c, cmb_read_batch* batch) {
  if (!c || !batch) return fail(c, CMB_E_ARG, "cmb_acquire_batch: null argument");
  if (!c->in_sample) return fail(c, CMB_E_ARG, "cmb_acquire_batch: no sample in progress");
  if (c->n_acquired >= c->cfg.n_staging) return fail(c, CMB_E_ARG, "cmb_acquire_batch: every staging batch is already acquired");
  const uint32_t i = c->next_batch;
  if (c->batch_busy[i]) {  // its previous H2D + K1 must have drained
    CU_TRY(c, cudaEventSynchronize(c->batch_done[i]));
    c->batch_busy[i] = false;
  }
  *batch = c->host_batch[i];
  c->next_batch = (i + 1) % c->cfg.n_staging;
  c->n_acquired += 1;
  return CMB_OK;
}

int cmb_submit_batch(cmb_ctx* c, uint32_t n_records, uint32_t n_intervals) {
  NvtxRange nvtx_fn("cmb_submit_batch: H2D + K1");
  if (!c) return CMB_E_ARG;
  if (!c->in_sample || c->n_acquired == 0) return fail(c, CMB_E_ARG, "cmb_submit_batch: no acquired batch");
  if (n_records > c->cfg.batch_records || n_intervals > c->cfg.batch_intervals) return fail(c, CMB_E_ARG, "cmb_submit_batch: batch exceeds capacity");
  const uint32_t i = (c->next_batch + c->cfg.n_staging - c->n_acquired) % c->cfg.n_staging;  // oldest acquired batch
  c->n_acquired -= 1;
  if (n_records == 0) return CMB_OK;
  if (c->n_local == 0) return CMB_OK;
  const cmb_read_batch& h = c->host_batch[i];
  const cmb_read_batch& d = c->dev_batch[i].ptr;
  CU_TRY(c, cudaSetDevice(c->device));
#define H2D(col, bytes) CU_TRY(c, cudaMemcpyAsync(d.col, h.col, (bytes), cudaMemcpyHostToDevice, c->stream))
  H2D(tid, 4ull * n_records);
  H2D(pos, 4ull * n_records);
  H2D(nm, 4ull * n_records);
  H2D(l_seq, 4ull * n_records);
  H2D(aligned, 4ull * n_records);
  H2D(del, 4ull * n_records);
  H2D(ins, 4ull * n_records);
  H2D(iv_begin, 4ull * (n_records + 1));
  if (n_intervals) {
    H2D(iv_start, 4ull * n_intervals);
    H2D(iv_len, 4ull * n_intervals);
  }
  H2D(flag, 2ull * n_records);
  H2D(mapq, 1ull * n_records);
  H2D(nm_state, 1ull * n_records);
#undef H2D
  int rc = launch_k1(c, d, n_records, n_intervals);
  if (rc) return rc;
  CU_TRY(c, cudaEventRecord(c->batch_done[i], c->stream));
  c->batch_busy[i] = true;
  return CMB_OK;
}

int cmb_submit_device_batch(cmb_ctx* c, const cmb_read_batch* dev, uint32_t n_records, uint32_t n_intervals) {
  NvtxRange nvtx_fn("cmb_submit_device_batch: K1");
  if (!c || !dev) return fail(c, CMB_E_ARG, "cmb_submit_device_batch: null argument");
  if (!c->in_sample) return fail(c, CMB_E_ARG, "cmb_submit_device_batch: no sample in progress");
  if (c->n_local == 0) return CMB_OK;
  CU_TRY(c, cudaSetDevice(c->device));
  // re-submitting the tuples of the last device decode (cmb_last_bgzf_batch) in pair mode: its mate table goes with it
  const bool is_last = c->dec.last_valid && (const void*)dev->tid == c->dec.d_tuple_slab;
  const int32_t* mate = (is_last && c->dec.last_mate && c->mode.filter_pairs) ? c->dec.last_mate : nullptr;
  return launch_k1(c, *dev, n_records, n_intervals, is_last ? c->dec.last_excl_n : 0xffffffffu, mate);
}

int cmb_end_sample_device(cmb_ctx* c, const cmb_contig_stats** dev_stats) {
  NvtxRange nvtx_fn("cmb_end_sample: K1c K1b K2 K3");
  if (!c) return CMB_E_ARG;
  if (!c->in_sample) return fail(c, CMB_E_ARG, "cmb_end_sample: no sample in progress");
  if (c->n_acquired) return fail(c, CMB_E_ARG, "cmb_end_sample: an acquired batch was not submitted");
  CU_TRY(c, cudaSetDevice(c->device));
  c->in_sample = false;
  if (c->n_local) {
    int rc = run_end_of_sample(c);
    if (rc) return rc;
  } else {
    for (int i = 2; i <= 5; ++i) CU_TRY(c, cudaEventRecord(c->ev[i], c->stream));
  }
  uint32_t counters[6];
  int rc = collect_errors_and_timing(c, counters);
  if (rc) return rc;
  c->ended = true;
  if (dev_stats) *dev_stats = c->d_rows;
  return CMB_OK;
}

int cmb_end_sample(cmb_ctx* c, cmb_contig_stats* stats, cmb_hist_pair* pairs, uint64_t pairs_capacity, uint64_t* n_pairs) {
  NvtxRange nvtx_fn("cmb_end_sample: kernels + D2H");
  if (!c) return fail(c, CMB_E_ARG, "cmb_end_sample: null argument");
  int rc = cmb_end_sample_device(c, nullptr);
  if (rc) return rc;
  if (stats) CU_TRY(c, cudaMemcpyAsync(stats, c->d_rows, sizeof(cmb_contig_stats) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost, c->stream));
  uint64_t np = 0;
  if ((c->params.want & CMB_WANT_HIST_CSR) && c->n_local) {
    unsigned long long cnt = 0;
    CU_TRY(c, cudaMemcpyAsync(&cnt, c->d_counters + 4, 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    np = cnt;
    if (np > c->pair_capacity) return fail(c, CMB_E_CAPACITY, "device histogram pair buffer overflowed");
    if (pairs) {
      if (np > pairs_capacity) return fail(c, CMB_E_CAPACITY, "cmb_end_sample: caller's pair buffer too small (%llu needed)", (unsigned long long)np);
      if (np) CU_TRY(c, cudaMemcpyAsync(pairs, c->d_pairs, sizeof(cmb_hist_pair) * np, cudaMemcpyDeviceToHost, c->stream));
    }
  }
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  if (n_pairs) *n_pairs = np;
  return CMB_OK;
}

int cmb_fetch_pairs(cmb_ctx* c, cmb_hist_pair* pairs, uint64_t n_pairs) {
  if (!c || (!pairs && n_pairs)) return fail(c, CMB_E_ARG, "cmb_fetch_pairs: null argument");
  if (!c->ended) return fail(c, CMB_E_ARG, "cmb_fetch_pairs: no ended sample");
  if (n_pairs > c->pair_capacity) return fail(c, CMB_E_ARG, "cmb_fetch_pairs: more pairs requested than produced");
  if (n_pairs) {
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaMemcpyAsync(pairs, c->d_pairs, sizeof(cmb_hist_pair) * n_pairs, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
  }
  return CMB_OK;
}

int cmb_grow_buffers(cmb_ctx* c) {
  if (!c || !c->d_rows) return fail(c, CMB_E_ARG, "cmb_grow_buffers: no reference set");
  if (c->in_sample) return fail(c, CMB_E_ARG, "cmb_grow_buffers: a sample is in progress");
  if (c->n_local == 0) return CMB_OK;
  CU_TRY(c, cudaSetDevice(c->device));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  const uint64_t rec = std::min<uint64_t>(0xfffffff0ull, (uint64_t)c->rec_capacity * 4);
  const uint64_t ovf = std::min<uint64_t>(1ull << 30, (uint64_t)c->ovf_capacity * 4);
  cudaFree(c->d_rec);
  cudaFree(c->d_ovf);
  c->d_rec = nullptr;
  c->d_ovf = nullptr;
  CU_TRY(c, cudaMalloc(&c->d_rec, 8ull * rec));
  CU_TRY(c, cudaMalloc(&c->d_ovf, 16ull * ovf));
  c->rec_capacity = (uint32_t)rec;
  c->ovf_capacity = (uint32_t)ovf;
  if (c->d_pairs) {
    const uint64_t want = c->pair_capacity * 4;
    cudaFree(c->d_pairs);
    c->d_pairs = nullptr;
    c->pair_capacity = 0;
    CU_TRY(c, cudaMalloc(&c->d_pairs, sizeof(cmb_hist_pair) * want));
    c->pair_capacity = want;
  }
  c->arena_dirty = true;
  return CMB_OK;
}

int cmb_get_timing(const cmb_ctx* c, cmb_sample_timing* out) {
  if (!c || !out) return CMB_E_ARG;
  *out = c->timing;
  return CMB_OK;
}

void* cmb_stream(cmb_ctx* c) { return c ? (void*)c->stream : nullptr; }

void cmb_nvtx_push(const char* name) { nvtxRangePushA(name ? name : "?"); }
void cmb_nvtx_pop(void) { nvtxRangePop(); }

// ------------------------------------------------------------------------------------------------ multi-GPU (NCCL)
#define NCCL_TRY(ctx, expr)                                                                                       \
  do {                                                                                                            \
    ncclResult_t r_ = (expr);                                                                                     \
    if (r_ != ncclSuccess) return fail(ctx, CMB_E_CUDA, "%s failed: %s (%s:%d)", #expr, ncclGetErrorString(r_), __FILE__, __LINE__); \
  } while (0)

namespace {
// NCCL writes its banner / debug lines to stdout by default; stdout carries the coverage table.
void nccl_output_to_stderr() {
  static const bool once = [] {
    // NCCL honours NCCL_DEBUG_FILE only above the VERSION level: at NCCL_DEBUG=VERSION the banner goes to stdout regardless
    const char* lvl = getenv("NCCL_DEBUG");
    if (lvl && !strcasecmp(lvl, "VERSION")) setenv("NCCL_DEBUG", "WARN", 1);  // WARN prints the same banner, to the debug file
    if (!getenv("NCCL_DEBUG_FILE")) setenv("NCCL_DEBUG_FILE", "/dev/stderr", 0);
    return true;
  }();
  (void)once;
}
// While a communicator is created, file descriptor 1 points at stderr: whatever NCCL (or a plugin it loads) prints during
// initialisation cannot end up in the coverage table.  Nothing else writes to stdout at that point (tables are printed at the end).
struct StdoutGuard {
  static std::mutex& mu() { static std::mutex m; return m; }
  std::lock_guard<std::mutex> lock{mu()};
  int saved = -1;
  StdoutGuard() {
    fflush(stdout);
    saved = dup(1);
    if (saved >= 0) dup2(2, 1);
  }
  ~StdoutGuard() {
    fflush(stdout);
    if (saved >= 0) {
      dup2(saved, 1);
      close(saved);
    }
  }
};
}  // namespace

int cmb_comm_unique_id(uint8_t id[CMB_COMM_ID_BYTES]) {
  nccl_output_to_stderr();
  static_assert(sizeof(ncclUniqueId) == CMB_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  if (!id) return fail(nullptr, CMB_E_ARG, "cmb_comm_unique_id: null argument");
  ncclUniqueId u;
  StdoutGuard guard;
  NCCL_TRY(nullptr, ncclGetUniqueId(&u));
  memcpy(id, &u, sizeof u);
  return CMB_OK;
}

int cmb_comm_init(cmb_ctx* c, const uint8_t id[CMB_COMM_ID_BYTES], int rank, int n_ranks) {
  if (!c || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(c, CMB_E_ARG, "cmb_comm_init: bad arguments");
  if (c->comm) return fail(c, CMB_E_ARG, "cmb_comm_init: the context already has a communicator");
  nccl_output_to_stderr();
  CU_TRY(c, cudaSetDevice(c->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof u);
  {
    StdoutGuard guard;
    NCCL_TRY(c, ncclCommInitRank(&c->comm, n_ranks, u, rank));
  }
  c->comm_rank = rank;
  c->comm_size = n_ranks;
  return CMB_OK;
}

int cmb_comm_init_local(cmb_ctx* const* ctxs, int n_ranks) {
  if (!ctxs || n_ranks < 1) return fail(nullptr, CMB_E_ARG, "cmb_comm_init_local: bad arguments");
  std::vector<int> devs(n_ranks);
  for (int r = 0; r < n_ranks; ++r) {
    if (!ctxs[r] || ctxs[r]->comm) return fail(ctxs[r], CMB_E_ARG, "cmb_comm_init_local: null context or communicator already set");
    devs[r] = ctxs[r]->device;
  }
  std::vector<ncclComm_t> comms(n_ranks);
  nccl_output_to_stderr();
  {
    StdoutGuard guard;
    NCCL_TRY(ctxs[0], ncclCommInitAll(comms.data(), n_ranks, devs.data()));
  }
  auto barrier = std::make_shared<LocalBarrier>();
  barrier->n = n_ranks;
  for (int r = 0; r < n_ranks; ++r) {
    ctxs[r]->local_barrier = barrier;
    ctxs[r]->comm = comms[r];
    ctxs[r]->comm_rank = r;
    ctxs[r]->comm_size = n_ranks;
  }
  return CMB_OK;
}

void cmb_comm_destroy(cmb_ctx* c) {
  if (!c || !c->comm) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  ncclCommDestroy(c->comm);
  c->comm = nullptr;
  c->local_barrier.reset();
  c->comm_rank = 0;
  c->comm_size = 1;
}

int cmb_comm_allgather(cmb_ctx* c, const void* send, void* recv, size_t bytes) {
  if (!c || !send || !recv || !bytes) return fail(c, CMB_E_ARG, "cmb_comm_allgather: bad arguments");
  if (!c->comm) return fail(c, CMB_E_ARG, "cmb_comm_allgather: no communicator (cmb_comm_init first)");
  CU_TRY(c, cudaSetDevice(c->device));
  const size_t need = bytes * (size_t)(c->comm_size + 1);
  if (c->xchg_cap < need) {
    cudaFree(c->d_xchg);
    c->d_xchg = nullptr;
    c->xchg_cap = 0;
    CU_TRY(c, cudaMalloc(&c->d_xchg, need + 4096));
    c->xchg_cap = need + 4096;
  }
  uint8_t* d_send = c->d_xchg;
  uint8_t* d_recv = c->d_xchg + bytes;
  if (c->local_barrier) c->local_barrier->arrive_and_wait();
  CU_TRY(c, cudaMemcpyAsync(d_send, send, bytes, cudaMemcpyHostToDevice, c->stream));
  NCCL_TRY(c, ncclAllGather(d_send, d_recv, bytes, ncclChar, c->comm, c->stream));
  CU_TRY(c, cudaMemcpyAsync(recv, d_recv, bytes * (size_t)c->comm_size, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  return CMB_OK;
}

int cmb_allgather_stats(cmb_ctx* c, const uint32_t* tid_cuts, const uint64_t* pair_base, cmb_contig_stats* stats, cmb_hist_pair* pairs) {
  NvtxRange nvtx_fn("cmb_allgather_stats: NCCL gather");
  if (!c || !tid_cuts) return fail(c, CMB_E_ARG, "cmb_allgather_stats: null argument");
  if (!c->comm) return fail(c, CMB_E_ARG, "cmb_allgather_stats: no communicator (cmb_comm_init first)");
  if (!c->ended || !c->d_rows) return fail(c, CMB_E_ARG, "cmb_allgather_stats: no ended sample");
  const int N = c->comm_size, me = c->comm_rank;
  if (tid_cuts[0] != 0 || tid_cuts[N] != c->n_contigs || tid_cuts[me] != c->tid_begin || tid_cuts[me + 1] != c->tid_end)
    return fail(c, CMB_E_ARG, "cmb_allgather_stats: tid_cuts do not match this context's shard");
  for (int r = 0; r < N; ++r)
    if (tid_cuts[r] > tid_cuts[r + 1]) return fail(c, CMB_E_ARG, "cmb_allgather_stats: tid_cuts must be non-decreasing");
  CU_TRY(c, cudaSetDevice(c->device));
  const bool csr = pair_base && (c->params.want & CMB_WANT_HIST_CSR);
  if (csr) {
    const uint64_t total = pair_base[N];
    if (pair_base[me + 1] - pair_base[me] > c->pair_capacity) return fail(c, CMB_E_ARG, "cmb_allgather_stats: pair_base exceeds this rank's pairs");
    if (c->pairs_all_capacity < total || !c->d_pairs_all) {
      cudaFree(c->d_pairs_all);
      c->d_pairs_all = nullptr;
      c->pairs_all_capacity = 0;
      const uint64_t want = total + total / 8 + 1024;
      CU_TRY(c, cudaMalloc(&c->d_pairs_all, sizeof(cmb_hist_pair) * want));
      c->pairs_all_capacity = want;
    }
    const uint32_t n_own = c->tid_end - c->tid_begin;
    if (n_own && pair_base[me]) {
      k_rebase_hist_offsets<<<(n_own + 255) / 256, 256, 0, c->stream>>>(c->d_rows + c->tid_begin, n_own, pair_base[me]);
      CU_TRY(c, cudaGetLastError());
    }
  }
  if (c->local_barrier) c->local_barrier->arrive_and_wait();
  // every rank broadcasts its own row range in place: afterwards each rank's table is complete (an all-gather with ragged counts)
  NCCL_TRY(c, ncclGroupStart());
  for (int r = 0; r < N; ++r) {
    const size_t n = (size_t)(tid_cuts[r + 1] - tid_cuts[r]) * sizeof(cmb_contig_stats);
    if (!n) continue;
    cmb_contig_stats* p = c->d_rows + tid_cuts[r];
    NCCL_TRY(c, ncclBroadcast(p, p, n, ncclChar, r, c->comm, c->stream));
  }
  if (csr) {
    for (int r = 0; r < N; ++r) {
      const size_t n = (size_t)(pair_base[r + 1] - pair_base[r]) * sizeof(cmb_hist_pair);
      if (!n) continue;
      NCCL_TRY(c, ncclBroadcast(c->d_pairs, c->d_pairs_all + pair_base[r], n, ncclChar, r, c->comm, c->stream));
    }
  }
  NCCL_TRY(c, ncclGroupEnd());
  if (stats) CU_TRY(c, cudaMemcpyAsync(stats, c->d_rows, sizeof(cmb_contig_stats) * (size_t)c->n_contigs, cudaMemcpyDeviceToHost, c->stream));
  if (csr && pairs && pair_base[N])
    CU_TRY(c, cudaMemcpyAsync(pairs, c->d_pairs_all, sizeof(cmb_hist_pair) * pair_base[N], cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  return CMB_OK;
}

int cmb_kept_tid_range(cmb_ctx* c, int32_t* min_tid, int32_t* max_tid) {
  if (!c || !min_tid || !max_tid) return fail(c, CMB_E_ARG, "cmb_kept_tid_range: null argument");
  if (!c->ended) return fail(c, CMB_E_ARG, "cmb_kept_tid_range: no ended sample");
  if (c->kept_range[0] == 0) {
    *min_tid = INT_MAX;
    *max_tid = INT_MIN;
  } else {
    *max_tid = (int32_t)(c->kept_range[0] - 1);
    *min_tid = INT_MAX - (int32_t)c->kept_range[1];
  }
  return CMB_OK;
}

void* cmb_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void cmb_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ device-side decode
namespace {
constexpr size_t DEC_COPY_CHUNK = 8u << 20;    // pinned staging slot
constexpr size_t DEC_WINDOW_BYTES = 32u << 20; // compressed bytes per copy+inflate window
size_t dec_window_bytes() {  // CMB_DECODE_WINDOW_KB: testing aid, lets a small file span many windows
  static const size_t v = [] {
    const char* e = getenv("CMB_DECODE_WINDOW_KB");
    const long kb = e ? atol(e) : 0;
    return kb > 0 ? (size_t)kb << 10 : DEC_WINDOW_BYTES;
  }();
  return v;
}
constexpr size_t DEC_SLACK = 1024;
constexpr size_t DEC_FRONT = 256;              // readable bytes in front of the first uploaded block (the bit readers align down)
constexpr uint64_t DEC_TAIL_BYTES = 4u << 20;  // ranged decode: inflated bytes kept beyond the range for its last straddling record

// First-pass inflate kernel: 0 = kd_inflate_t1 (a thread per block, then kd_crc32), 1 = kd_inflate_g8 (four blocks per warp),
// 2 = kd_inflate (a warp per block; it is also the second pass over the blocks the first pass declined).  t1 has the higher
// THROUGHPUT (its ~75 000 streams in flight need that many blocks) but every block takes ~50 ms however few there are; g8
// finishes a block in ~20 ms.  So the choice follows the number of blocks: a whole 10 M-read file (46 000 blocks) goes to t1,
// a rank's share of it on 4 or 8 GPUs to g8.  CMB_INFLATE=t1|g8|w1 forces one kernel, e.g. to run each of them on a small file.
constexpr uint32_t T1_MIN_BLOCKS = 28000;
int inflate_kind(uint32_t n_blocks) {
  static const int forced = [] {
    const char* e = getenv("CMB_INFLATE");
    if (e && !strcmp(e, "t1")) return 0;
    if (e && !strcmp(e, "g8")) return 1;
    if (e && !strcmp(e, "w1")) return 2;
    return -1;
  }();
  if (forced >= 0) return forced;
  return n_blocks >= T1_MIN_BLOCKS ? 0 : 1;
}
// Two launch disciplines for the inflate stage.  Persistent (the default): ONE launch before the copies, whose threads poll
// the windows' arrival flags (bounded wait), so that every SM has work as soon as the first window is in.
// Serial mode: copy everything, then ONE inflate launch ordered behind the copies on the context stream -- no flags, nothing on
// the device waits for anything.  Used for files of a single window (nothing to overlap), on request (CMB_INFLATE_SERIAL=1),
// and when a CUDA tool is injected into the process (ncu, compute-sanitizer: they serialise kernels against the other streams,
// so a kernel that polls for copies would only ever see its bounded wait expire).
bool inflate_serial_requested() {
  static const bool v = [] {
    if (const char* e = getenv("CMB_INFLATE_SERIAL")) return e[0] == '1';
    for (const char* name : {"CUDA_INJECTION64_PATH", "NV_NSIGHT_INJECTION_PORT_BASE", "NV_COMPUTE_PROFILER_PERFWORKS_DIR", "NV_SANITIZER_INJECTION_PORT_BASE"})
      if (const char* e = getenv(name))
        if (e[0]) return true;
    return false;
  }();
  return v;
}
// kd_crc32 over the blocks of `a` (the t1 path: its inflate kernel leaves the CRC to a second kernel)
int launch_crc32(cmb_ctx* c, const InflateArgs& a, cudaStream_t st) {
  const uint32_t nb = a.b1 - a.b0;
  kd_crc32<<<std::min<uint32_t>((nb + 7) / 8, (uint32_t)c->sm_count * 8), 256, 0, st>>>(a);
  CU_TRY(c, cudaGetLastError());
  return CMB_OK;
}
// Launch the first-pass (or, with first_pass false or a block list, the second-pass) inflate kernel over blocks [a.b0, a.b1).
// *crc_pending (when given) is set instead of launching kd_crc32: the caller launches it once nothing else has to get past it
// in the hardware queue (a kernel waiting for its predecessor blocks the queue for every stream that shares it).
int launch_inflate(cmb_ctx* c, const InflateArgs& a, cudaStream_t st, bool first_pass = true, bool* crc_pending = nullptr) {
  const int which = inflate_kind(a.b1 - a.b0);
  const int k = (first_pass && !a.block_list) ? which : 2;
  const uint32_t nb = a.b1 - a.b0;
  if (k == 0) {
    CU_TRY(c, cudaFuncSetAttribute(kd_inflate_t1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T1_SMEM_BYTES));
    // every resident warp takes part; with fewer blocks than lanes, each warp works with its first `lanes` lanes only
    const uint32_t max_grid = (uint32_t)c->sm_count * 5, warps = max_grid * (T1_THREADS / 32);
    const uint32_t lanes = std::min<uint32_t>(32, std::max<uint32_t>(1, (nb + warps - 1) / warps));
    const uint32_t per_cta = lanes * (T1_THREADS / 32);
    const uint32_t grid = std::min<uint32_t>((nb + per_cta - 1) / per_cta, max_grid);
    InflateArgs at = a;
    at.lane_limit = lanes;
    kd_inflate_t1<<<grid, T1_THREADS, T1_SMEM_BYTES, st>>>(at);
    CU_TRY(c, cudaGetLastError());
    if (crc_pending) *crc_pending = true;
    else if (int rc = launch_crc32(c, a, st)) return rc;
  } else if (k == 1) {
    CU_TRY(c, cudaFuncSetAttribute(kd_inflate_g8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G8_SMEM_BYTES));
    const uint32_t per_cta = G8_WARPS * G8_STREAMS;
    const uint32_t grid = std::min<uint32_t>((nb + per_cta - 1) / per_cta, (uint32_t)c->sm_count * 2);
    kd_inflate_g8<<<grid, G8_WARPS * 32, G8_SMEM_BYTES, st>>>(a);
  } else {
    CU_TRY(c, cudaFuncSetAttribute(kd_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INF_SMEM_BYTES));
    const uint32_t grid = std::min<uint32_t>((nb + INF_WARPS - 1) / INF_WARPS, (uint32_t)c->sm_count * 2);
    kd_inflate<<<grid, INF_WARPS * 32, INF_SMEM_BYTES, st>>>(a);
  }
  CU_TRY(c, cudaGetLastError());
  return CMB_OK;
}

template <class T>
int dec_grow(cmb_ctx* c, T*& p, size_t& cap, size_t need, size_t extra_bytes = 0) {
  if (cap >= need && p) return CMB_OK;
  cudaFree(p);
  p = nullptr;
  cap = 0;
  const size_t want = need + need / 8 + 16;
  CU_TRY(c, cudaMalloc(&p, want * sizeof(T) + extra_bytes));
  cap = want;
  return CMB_OK;
}

// zlib's raw inflate of BGZF block b into tmp (grown to fit); true when the stream ends with exactly the block's isize bytes
bool zlib_inflate_block(z_stream& zs, const cmb_bgzf_input* in, uint32_t b, std::vector<uint8_t>& tmp, int* zrc = nullptr) {
  const uint32_t isz = in->block_isize[b];
  if (tmp.size() < isz) tmp.resize(isz);
  inflateReset(&zs);
  zs.next_in = const_cast<Bytef*>(in->data + in->block_coffset[b]);
  zs.avail_in = in->block_clen[b];
  zs.next_out = tmp.data();
  zs.avail_out = isz;
  const int rc = inflate(&zs, Z_FINISH);
  if (zrc) *zrc = rc;
  return rc == Z_STREAM_END && zs.avail_out == 0;
}
}  // namespace

namespace {
int submit_bgzf_impl(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out, bool decode_only);
}
// Device memory for the decode buffers (compressed file + inflated stream + tuples) is requested before anything is
// accumulated, so running out of it simply declines the sample: the host decoder needs only the staging batches.
extern "C" int cmb_last_bgzf_batch(cmb_ctx* c, cmb_read_batch* dev_batch, uint32_t* n_records, uint32_t* n_intervals) {
  if (!c || !dev_batch || !n_records || !n_intervals) return fail(c, CMB_E_ARG, "cmb_last_bgzf_batch: null argument");
  if (!c->dec.last_valid || !c->dec.d_tuple_slab) return fail(c, CMB_E_ARG, "cmb_last_bgzf_batch: no device-decoded sample is resident");
  carve_batch(c->dec.d_tuple_slab, c->dec.last_n_rec, c->dec.last_n_cig, dev_batch);
  *n_records = c->dec.last_n_rec;
  *n_intervals = c->dec.last_n_cig;
  return CMB_OK;
}

namespace {
int bgzf_entry(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out, bool decode_only);
}
extern "C" int cmb_submit_bgzf(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out) { return bgzf_entry(c, in, out, false); }
extern "C" int cmb_decode_bgzf(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out) { return bgzf_entry(c, in, out, true); }

extern "C" int cmb_filter_plan(cmb_ctx* c, int inverse, uint64_t* n_records, uint64_t* n_bytes) {
  if (!c || !n_records || !n_bytes) return fail(c, CMB_E_ARG, "cmb_filter_plan: null argument");
  auto& d = c->dec;
  if (!d.last_valid || !d.d_tuple_slab || !c->have_params) return fail(c, CMB_E_ARG, "cmb_filter_plan: no device-decoded sample is resident (cmb_decode_bgzf first)");
  CU_TRY(c, cudaSetDevice(c->device));
  *n_records = 0;
  *n_bytes = 0;
  d.filter_planned = false;
  const uint32_t n = d.last_n_rec;
  if (n == 0) {
    d.filter_bytes = 0;
    d.filter_planned = true;
    return CMB_OK;
  }
  const bool pair_path = !(c->mode.filter_single_reads && !c->mode.filter_pairs);
  if (pair_path && !d.last_mate) return fail(c, CMB_E_ARG, "cmb_filter_plan: the sample was decoded without mate matching (set the parameters before cmb_decode_bgzf)");
  if (d.filter_rec_cap < (size_t)n + 1 || !d.d_filter_anchor) {
    cudaFree(d.d_filter_anchor); cudaFree(d.d_filter_role);
    d.d_filter_anchor = nullptr; d.d_filter_role = nullptr; d.filter_rec_cap = 0;
    const size_t want = (size_t)n + n / 8 + 16;
    CU_TRY(c, cudaMalloc(&d.d_filter_anchor, 8 * want));
    CU_TRY(c, cudaMalloc(&d.d_filter_role, want));
    d.filter_rec_cap = want;
  }
  cmb_read_batch tb;
  carve_batch(d.d_tuple_slab, d.last_n_rec, d.last_n_cig, &tb);
  FilterArgs a{};
  a.data = d.last_infl_base; a.rec_off = d.d_rec_off; a.n = n; a.flag = tb.flag; a.mapq = tb.mapq; a.nm_state = tb.nm_state; a.nm = tb.nm;
  a.l_seq = tb.l_seq; a.aligned = tb.aligned; a.del = tb.del; a.mate = pair_path ? d.last_mate : nullptr; a.p = c->params;
  a.filter_single = c->mode.filter_single_reads; a.pair_path = pair_path; a.filter_out = inverse ? 0 : 1;
  a.anchor_bytes = d.d_filter_anchor; a.role = d.d_filter_role; a.error_flags = d.d_cnt + 12; a.n_emit = (unsigned long long*)(d.d_cnt + 14);
  CU_TRY(c, cudaMemsetAsync(d.d_cnt + 12, 0, 16, c->stream));
  kf_decide<<<(n + 255) / 256, 256, 0, c->stream>>>(a);
  kf_scan<<<1, 1024, 0, c->stream>>>(d.d_filter_anchor, n);
  CU_TRY(c, cudaGetLastError());
  uint32_t h[4];
  unsigned long long total = 0;
  CU_TRY(c, cudaMemcpyAsync(h, d.d_cnt + 12, 16, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaMemcpyAsync(&total, d.d_filter_anchor + n, 8, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  if (h[0] & ERR_NM)
    return fail(c, CMB_E_NM, "Mapping record encountered that does not have an 'NM' auxiliary tag in the SAM/BAM format. This is required to work out some coverage statistics");
  unsigned long long n_emit;
  memcpy(&n_emit, h + 2, 8);
  if (d.filter_out_cap < total || !d.d_filter_out) {
    cudaFree(d.d_filter_out);
    d.d_filter_out = nullptr;
    d.filter_out_cap = 0;
    const size_t want = (size_t)total + (size_t)total / 8 + 4096;
    CU_TRY(c, cudaMalloc(&d.d_filter_out, want));
    d.filter_out_cap = want;
  }
  a.out = d.d_filter_out;
  kf_gather<<<(n + 7) / 8, 256, 0, c->stream>>>(a);
  CU_TRY(c, cudaGetLastError());
  d.filter_bytes = total;
  d.filter_planned = true;
  *n_records = n_emit;
  *n_bytes = total;
  return CMB_OK;
}

extern "C" int cmb_filter_fetch(cmb_ctx* c, uint8_t* records, uint64_t n_bytes) {
  if (!c || (!records && n_bytes)) return fail(c, CMB_E_ARG, "cmb_filter_fetch: null argument");
  auto& d = c->dec;
  if (!d.filter_planned || n_bytes != d.filter_bytes) return fail(c, CMB_E_ARG, "cmb_filter_fetch: call cmb_filter_plan first and pass the size it reported");
  CU_TRY(c, cudaSetDevice(c->device));
  if (n_bytes) CU_TRY(c, cudaMemcpyAsync(records, d.d_filter_out, n_bytes, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  return CMB_OK;
}

namespace {
int bgzf_entry(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out, bool decode_only) {
  if (c) {
    c->dec.last_valid = false;
    c->dec.filter_planned = false;
  }
  const auto t_call0 = std::chrono::steady_clock::now();
  const int rc = submit_bgzf_impl(c, in, out, decode_only);
  if (out) out->ms_host_wall = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call0).count();
  if (rc == CMB_E_NOMEM) {
    cudaGetLastError();
    auto& d = c->dec;  // give the big buffers back so that the rest of the sample has room
    cudaFree(d.d_comp); d.d_comp = nullptr; d.comp_cap = 0;
    cudaFree(d.d_inflated); d.d_inflated = nullptr; d.infl_cap = 0;
    cudaFree(d.d_tuple_slab); d.d_tuple_slab = nullptr; d.tuple_slab_bytes = 0;
    cudaFree(d.d_rec_off); d.d_rec_off = nullptr; d.rec_cap = 0;
    return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: not enough device memory for device-side decode");
  }
  return rc;
}
}  // namespace
namespace {
int submit_bgzf_impl(cmb_ctx* c, const cmb_bgzf_input* in, cmb_bgzf_result* out, bool decode_only) {
  NvtxRange nvtx_fn("cmb_submit_bgzf");
  if (!c || !in || !out || !in->data || !in->block_coffset || !in->block_clen || !in->block_isize)
    return fail(c, CMB_E_ARG, "cmb_submit_bgzf: null argument");
  if (!decode_only && !c->in_sample) return fail(c, CMB_E_ARG, "cmb_submit_bgzf: no sample in progress");
  if (decode_only && (c->in_sample || !c->have_params)) return fail(c, CMB_E_ARG, "cmb_decode_bgzf: set the parameters first; not inside a sample");
  if (c->n_acquired) return fail(c, CMB_E_ARG, "cmb_submit_bgzf: a staging batch is still acquired");
  *out = cmb_bgzf_result{};
  const uint32_t nb = in->n_blocks;
  if (nb == 0) return CMB_OK;
  CU_TRY(c, cudaSetDevice(c->device));
  auto& d = c->dec;
  // ---- host block table
  std::vector<uint64_t> ustart((size_t)nb + 1, 0);
  for (uint32_t b = 0; b < nb; ++b) {
    if (in->block_coffset[b] + in->block_clen[b] + 8 > in->size) return fail(c, CMB_E_ARG, "cmb_submit_bgzf: block %u lies outside the data", b);
    ustart[b + 1] = ustart[b] + in->block_isize[b];
  }
  const uint64_t stream_total = ustart[nb];
  if (in->records_at > stream_total) return fail(c, CMB_E_ARG, "cmb_submit_bgzf: records_at beyond the end of the stream");
  if (in->records_at == stream_total) return CMB_OK;  // header only
  // Blocks: records starting in [first_block, walk_end) are decoded; [first_block, data_end) are uploaded and inflated (the tail
  // beyond walk_end only supplies the bytes of a record that straddles out of the range).  Whole file: walk_end = data_end = nb.
  uint32_t first_block = (uint32_t)(std::upper_bound(ustart.begin(), ustart.end(), in->records_at) - ustart.begin()) - 1;
  uint32_t walk_end = nb, data_end = nb;
  if (in->ranged) {
    if (in->walk_begin_block != first_block || in->walk_end_block > nb || in->walk_end_block < in->walk_begin_block)
      return fail(c, CMB_E_ARG, "cmb_submit_bgzf: inconsistent block range");
    walk_end = in->walk_end_block;
    if (walk_end == first_block) return CMB_OK;  // an empty share
    data_end = walk_end;
    uint64_t tail = 0;
    while (data_end < nb && tail < DEC_TAIL_BYTES) tail += in->block_isize[data_end++];
  }
  // Device buffers hold only [byte_lo, byte_hi) of the file and [u_lo, total) of the inflated stream; the kernels index both
  // with absolute offsets through biased base pointers.
  const uint64_t byte_lo = in->block_coffset[first_block];
  const uint64_t byte_hi = data_end == nb ? in->size : in->block_coffset[data_end - 1] + in->block_clen[data_end - 1] + 8;
  const uint64_t u_lo = ustart[first_block];
  const uint64_t total = ustart[data_end];  // end of the inflated bytes available to this call
  // ---- buffers
  if (const char* lim = getenv("CMB_DECODE_MEM_LIMIT_MB")) {  // testing aid: behave as if the device had this much room
    if (((byte_hi - byte_lo) + (total - u_lo)) >> 20 > strtoull(lim, nullptr, 10)) return CMB_E_NOMEM;
  }
  int rc;
  if ((rc = dec_grow(c, d.d_comp, d.comp_cap, (size_t)(byte_hi - byte_lo) + DEC_FRONT + DEC_SLACK))) return rc;
  if ((rc = dec_grow(c, d.d_inflated, d.infl_cap, (size_t)(total - u_lo) + DEC_SLACK))) return rc;
  uint8_t* const comp_base = reinterpret_cast<uint8_t*>(reinterpret_cast<uintptr_t>(d.d_comp) + DEC_FRONT - byte_lo);
  uint8_t* const infl_base = reinterpret_cast<uint8_t*>(reinterpret_cast<uintptr_t>(d.d_inflated) - u_lo);
  if (d.blocks_cap < (size_t)nb + 1 || !d.d_coff) {
    const size_t want = (size_t)nb + nb / 8 + 64;
    cudaFree(d.d_coff); cudaFree(d.d_ustart); cudaFree(d.d_guess); cudaFree(d.d_exit); cudaFree(d.d_rec_base); cudaFree(d.d_cig_base);
    cudaFree(d.d_clen); cudaFree(d.d_isize); cudaFree(d.d_status); cudaFree(d.d_nrec); cudaFree(d.d_ncig); cudaFree(d.d_dirty);
    d.d_coff = d.d_ustart = d.d_guess = d.d_exit = d.d_rec_base = d.d_cig_base = nullptr;
    d.d_clen = d.d_isize = d.d_status = d.d_nrec = d.d_ncig = d.d_dirty = nullptr;
    d.blocks_cap = 0;
    CU_TRY(c, cudaMalloc(&d.d_coff, 8 * want)); CU_TRY(c, cudaMalloc(&d.d_ustart, 8 * want)); CU_TRY(c, cudaMalloc(&d.d_guess, 8 * want));
    CU_TRY(c, cudaMalloc(&d.d_exit, 8 * want)); CU_TRY(c, cudaMalloc(&d.d_rec_base, 8 * want)); CU_TRY(c, cudaMalloc(&d.d_cig_base, 8 * want));
    CU_TRY(c, cudaMalloc(&d.d_clen, 4 * want)); CU_TRY(c, cudaMalloc(&d.d_isize, 4 * want)); CU_TRY(c, cudaMalloc(&d.d_status, 4 * want));
    CU_TRY(c, cudaMalloc(&d.d_nrec, 4 * want)); CU_TRY(c, cudaMalloc(&d.d_ncig, 4 * want)); CU_TRY(c, cudaMalloc(&d.d_dirty, 4 * want));
    cudaFree(d.d_t1_scratch);
    d.d_t1_scratch = nullptr;
    CU_TRY(c, cudaMalloc(&d.d_t1_scratch, (size_t)T1_LENS_BYTES * want));
    d.blocks_cap = want;
  }
  if (!d.d_cnt) CU_TRY(c, cudaMalloc(&d.d_cnt, 64));
  if (!d.have_events) {
    for (auto& e : d.ev) CU_TRY(c, cudaEventCreate(&e));
    d.have_events = true;
  }
  NvtxRange nvtx_copy("bgzf: H2D copy + inflate");
  // ---- windows of whole blocks, ~DEC_WINDOW_BYTES of file each
  struct Window { uint32_t b0, b1; uint64_t byte0, byte1; };
  std::vector<Window> windows;
  {
    uint32_t b = first_block;
    uint64_t byte0 = byte_lo;
    while (b < data_end) {
      uint32_t e = b;
      uint64_t byte1 = byte0;
      while (e < data_end && (e == b || in->block_coffset[e] + in->block_clen[e] + 8 - byte0 <= dec_window_bytes())) {
        byte1 = in->block_coffset[e] + in->block_clen[e] + 8;
        ++e;
      }
      if (e == data_end) byte1 = byte_hi;
      windows.push_back({b, e, byte0, byte1});
      b = e;
      byte0 = byte1;
    }
  }
  if (d.tickets_cap < windows.size() + 8 || !d.d_tickets) {  // [0] block ticket, [1, 1 + W) arrival flags
    cudaFree(d.d_tickets);
    d.d_tickets = nullptr;
    d.tickets_cap = 0;
    const size_t want = windows.size() * 3 + 64;
    CU_TRY(c, cudaMalloc(&d.d_tickets, 4 * want));
    d.tickets_cap = want;
  }
  if ((rc = dec_grow(c, d.d_block_window, d.block_window_cap, (size_t)nb))) return rc;
  if (!d.h_ones) {
    CU_TRY(c, cudaHostAlloc((void**)&d.h_ones, 64, cudaHostAllocDefault));
    for (int k = 0; k < 16; ++k) d.h_ones[k] = 1;
  }
  std::vector<uint32_t> block_window(nb, 0);
  for (size_t w = 0; w < windows.size(); ++w)
    for (uint32_t b = windows[w].b0; b < windows[w].b1; ++b) block_window[b] = (uint32_t)w;
  // ---- copy threads, their streams and pinned slots
  cudaPointerAttributes attr{};
  const bool src_pinned = cudaPointerGetAttributes(&attr, in->data) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();  // cudaPointerGetAttributes on pageable memory may leave a sticky-free error code
  uint32_t T = in->copy_threads ? in->copy_threads : 4;
  T = std::min<uint32_t>(std::min<uint32_t>(T, 16), (uint32_t)windows.size());
  while (d.streams.size() < T) {
    cudaStream_t st;
    CU_TRY(c, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    d.streams.push_back(st);
    cudaEvent_t e;
    CU_TRY(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    d.done_events.push_back(e);
    for (int k = 0; k < 2; ++k) {
      CU_TRY(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      d.slot_events.push_back(e);
      void* p = nullptr;
      CU_TRY(c, cudaHostAlloc(&p, DEC_COPY_CHUNK, cudaHostAllocDefault));
      d.pinned.push_back(p);
    }
  }
  // ---- upload the block table, reset counters (ctx stream), then let the copy streams start after it
  CU_TRY(c, cudaEventRecord(d.ev[0], c->stream));
  CU_TRY(c, cudaMemcpyAsync(d.d_coff, in->block_coffset, 8ull * nb, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(d.d_clen, in->block_clen, 4ull * nb, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(d.d_isize, in->block_isize, 4ull * nb, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemcpyAsync(d.d_ustart, ustart.data(), 8ull * (nb + 1), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemsetAsync(d.d_cnt, 0, 64, c->stream));
  CU_TRY(c, cudaMemsetAsync(d.d_status, 0, 4ull * nb, c->stream));
  CU_TRY(c, cudaMemcpyAsync(d.d_block_window, block_window.data(), 4ull * nb, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(c, cudaMemsetAsync(d.d_tickets, 0, 4 * (windows.size() + 1), c->stream));
  CU_TRY(c, cudaMemsetAsync(infl_base + total, 0, DEC_SLACK, c->stream));
  CU_TRY(c, cudaMemsetAsync(comp_base + byte_hi, 0, DEC_SLACK, c->stream));
  CU_TRY(c, cudaMemsetAsync(d.d_comp, 0, DEC_FRONT, c->stream));
  CU_TRY(c, cudaEventRecord(d.ev[1], c->stream));
  for (uint32_t t = 0; t < T; ++t) CU_TRY(c, cudaStreamWaitEvent(d.streams[t], d.ev[1], 0));
  // the InflateArgs of every inflate launch over blocks [b0, b1); the caller adds the block list or the arrival flags
  auto inflate_args = [&](uint32_t b0, uint32_t b1, uint32_t* fail_count) {
    InflateArgs a{};
    a.comp = comp_base; a.coff = d.d_coff; a.clen = d.d_clen; a.isize = d.d_isize; a.uoff = d.d_ustart; a.scratch = d.d_t1_scratch;
    a.b0 = b0; a.b1 = b1; a.out = infl_base; a.status = d.d_status; a.ticket = d.d_tickets; a.fail_count = fail_count;
    return a;
  };
  const bool serial = windows.size() <= 1 || inflate_serial_requested();
  bool crc_pending = false;
  InflateArgs persistent_args{};
  if (!serial) {  // one persistent launch over every block; its threads wait for their block's window to arrive
    // blocks before the one holding the first record are header text the host has already read: not inflated here
    persistent_args = inflate_args(first_block, data_end, d.d_cnt + 0);
    persistent_args.block_window = d.d_block_window; persistent_args.ready = d.d_tickets + 1;
    if ((rc = launch_inflate(c, persistent_args, c->stream, true, &crc_pending))) return rc;
  }
  std::atomic<size_t> next_window{0};
  std::atomic<int> first_err{0};
  auto worker = [&](uint32_t t) {
    cudaSetDevice(c->device);
    cudaStream_t st = d.streams[t];
    int slot = 0;
    bool used[2] = {false, false};
    auto check = [&](cudaError_t e) {
      if (e != cudaSuccess) {
        int z = 0;
        first_err.compare_exchange_strong(z, (int)e);
      }
      return e == cudaSuccess;
    };
    for (;;) {
      const size_t w = next_window.fetch_add(1);
      if (w >= windows.size() || first_err.load()) break;
      const Window& win = windows[w];
      if (src_pinned) {
        if (!check(cudaMemcpyAsync(comp_base + win.byte0, in->data + win.byte0, win.byte1 - win.byte0, cudaMemcpyHostToDevice, st))) break;
      } else {
        for (uint64_t o = win.byte0; o < win.byte1; o += DEC_COPY_CHUNK) {
          const size_t n = (size_t)std::min<uint64_t>(DEC_COPY_CHUNK, win.byte1 - o);
          const size_t si = (size_t)t * 2 + slot;
          if (used[slot] && !check(cudaEventSynchronize(d.slot_events[si]))) return;
          memcpy(d.pinned[si], in->data + o, n);
          if (!check(cudaMemcpyAsync(comp_base + o, d.pinned[si], n, cudaMemcpyHostToDevice, st))) return;
          if (!check(cudaEventRecord(d.slot_events[si], st))) return;
          used[slot] = true;
          slot ^= 1;
        }
      }
      if (!check(cudaMemcpyAsync(d.d_tickets + 1 + w, d.h_ones, 4, cudaMemcpyHostToDevice, st))) break;  // window w has arrived
    }
    check(cudaEventRecord(d.done_events[t], st));
  };
  const auto copy_t0 = std::chrono::steady_clock::now();
  {
    std::vector<std::thread> threads;
    for (uint32_t t = 1; t < T; ++t) threads.emplace_back(worker, t);
    worker(0);
    for (auto& th : threads) th.join();
  }
  const double copy_wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - copy_t0).count();
  out->ms_copy_enqueue_wall = (float)copy_wall_ms;
  if (crc_pending && (rc = launch_crc32(c, persistent_args, c->stream))) return rc;  // every copy is enqueued: nothing left to hold up
  if (serial && !first_err.load()) {
    for (uint32_t t = 0; t < T; ++t) CU_TRY(c, cudaStreamWaitEvent(c->stream, d.done_events[t], 0));
    if ((rc = launch_inflate(c, inflate_args(first_block, data_end, d.d_cnt + 0), c->stream))) return rc;
  }
  if (first_err.load()) {  // release the warps still waiting for windows that will never arrive
    cudaMemsetAsync(d.d_tickets + 1, 1, 4 * windows.size(), d.streams[0]);
    cudaStreamSynchronize(d.streams[0]);
    cudaStreamSynchronize(c->stream);
  }
  out->n_launches = 1;
  out->h2d_bytes = (byte_hi - byte_lo) + 24ull * nb + 8;
  if (first_err.load()) return fail(c, CMB_E_CUDA, "cmb_submit_bgzf: copy/inflate stage failed: %s", cudaGetErrorString((cudaError_t)first_err.load()));
  for (uint32_t t = 0; t < T; ++t) CU_TRY(c, cudaStreamWaitEvent(c->stream, d.done_events[t], 0));
  if (getenv("CMB_PIPELINE_STATS")) {  // how long the window copies alone took (the done events carry no timing: time them on the host)
    const auto h0 = std::chrono::steady_clock::now();
    for (uint32_t t = 0; t < T; ++t) cudaEventSynchronize(d.done_events[t]);
    const double wait_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
    fprintf(stderr, "#decode_h2d\twindows=%zu\tbytes=%llu\tcopy_streams_done_after_ms=%.1f (host clock from the end of the enqueue; enqueue took %.1f ms)\n",
            windows.size(), (unsigned long long)(byte_hi - byte_lo), wait_ms, copy_wall_ms);
  }
  CU_TRY(c, cudaEventRecord(d.ev[2], c->stream));
  if (getenv("CMB_DECODE_PROFILE")) {  // debugging aid: the inflate kernel alone, all blocks resident, one launch
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    cudaEvent_t p0, p1;
    cudaEventCreate(&p0);
    cudaEventCreate(&p1);
    CU_TRY(c, cudaMemsetAsync(d.d_tickets, 0, 4, c->stream));
    cudaEventRecord(p0, c->stream);
    if ((rc = launch_inflate(c, inflate_args(first_block, data_end, d.d_cnt + 8), c->stream))) return rc;
    cudaEventRecord(p1, c->stream);
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, p0, p1);
    fprintf(stderr, "#decode_profile\tinflate_only_ms=%.3f\tblocks=%u\tcompressed=%llu\tinflated=%llu\tinflated_GBps=%.2f\tcopy_threads=%u\tsrc_pinned=%d\tcopy_enqueue_wall_ms=%.2f\n", ms, data_end - first_block,
            (unsigned long long)(byte_hi - byte_lo), (unsigned long long)(total - u_lo), (total - u_lo) / ms * 1e-6, T, (int)src_pinned, copy_wall_ms);
    cudaEventDestroy(p0);
    cudaEventDestroy(p1);
  }
  nvtx_copy.end();
  NvtxRange nvtx_declined("bgzf: declined blocks (second pass, host zlib)");
  // ---- blocks the device declined: zlib on the host, patched into the inflated stream
  uint32_t h_cnt[16];
  CU_TRY(c, cudaMemcpyAsync(h_cnt, d.d_cnt, 64, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  if (h_cnt[0] || getenv("CMB_DECODE_RETRY_TEST")) {
    std::vector<uint32_t> status(nb);
    CU_TRY(c, cudaMemcpy(status.data(), d.d_status, 4ull * nb, cudaMemcpyDeviceToHost));
    if (getenv("CMB_DECODE_RETRY_TEST"))  // testing aid: pretend every 7th block was declined by the first pass (code 29)
      for (uint32_t b = first_block; b < data_end; b += 7) status[b] = 29;
    if (getenv("CMB_DECODE_VERIFY") || getenv("CMB_PIPELINE_STATS")) {
      uint32_t hist[32] = {0};
      for (uint32_t b = 0; b < nb; ++b) hist[std::min<uint32_t>(status[b], 31)]++;
      fprintf(stderr, "#decode_status");
      for (int k = 0; k < 32; ++k)
        if (hist[k]) fprintf(stderr, "\t%d:%u", k, hist[k]);
      fprintf(stderr, "\n");
    }
    // Second chance on the device: the one-stream-per-warp kernel has larger Huffman tables (10-bit roots, 128 long-code
    // prefixes) than the four-streams-per-warp one, so most blocks the first pass declined for table space fit there.
    {
      std::vector<uint32_t> again;
      for (uint32_t b = first_block; b < data_end; ++b)
        if (status[b] != INF_OK) again.push_back(b);
      out->n_blocks_second_pass = (uint32_t)again.size();
      if (!again.empty()) {
        uint32_t* d_list = d.d_dirty;  // free until the record chain starts (nb entries)
        CU_TRY(c, cudaMemcpyAsync(d_list, again.data(), 4ull * again.size(), cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaMemsetAsync(d.d_tickets, 0, 4, c->stream));
        CU_TRY(c, cudaMemsetAsync(d.d_cnt, 0, 4, c->stream));
        InflateArgs a2 = inflate_args(0, (uint32_t)again.size(), d.d_cnt + 0);
        a2.block_list = d_list;
        if ((rc = launch_inflate(c, a2, c->stream, false))) return rc;
        out->n_launches += 1;
        for (uint32_t b : again) status[b] = INF_OK;  // refreshed from the device below
        std::vector<uint32_t> st2(nb);
        CU_TRY(c, cudaMemcpyAsync(st2.data(), d.d_status, 4ull * nb, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        for (uint32_t b : again) status[b] = st2[b];
      }
    }
    std::vector<uint8_t> tmp(65536 + 64);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return fail(c, CMB_E_NOMEM, "zlib init failed");
    for (uint32_t b = first_block; b < data_end; ++b) {
      if (status[b] == INF_OK) continue;
      const uint32_t isz = in->block_isize[b];
      uint32_t want_crc;
      memcpy(&want_crc, in->data + in->block_coffset[b] + in->block_clen[b], 4);
      if (!zlib_inflate_block(zs, in, b, tmp) || (uint32_t)crc32(0, tmp.data(), isz) != want_crc) {
        inflateEnd(&zs);
        return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: BGZF block %u does not inflate", b);
      }
      CU_TRY(c, cudaMemcpy(infl_base + ustart[b], tmp.data(), isz, cudaMemcpyHostToDevice));
      out->n_blocks_host += 1;
    }
    inflateEnd(&zs);
  }
  if (getenv("CMB_DECODE_VERIFY")) {  // debugging aid: compare every device-inflated block with zlib's output
    std::vector<uint8_t> dev(total - u_lo), tmp(65536 + 64);
    CU_TRY(c, cudaMemcpy(dev.data(), d.d_inflated, total - u_lo, cudaMemcpyDeviceToHost));
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    inflateInit2(&zs, -15);
    uint32_t bad = 0;
    for (uint32_t b = first_block; b < data_end; ++b) {
      const uint32_t isz = in->block_isize[b];
      if (!isz) continue;
      int zr = 0;
      if (!zlib_inflate_block(zs, in, b, tmp, &zr) || memcmp(tmp.data(), dev.data() + (ustart[b] - u_lo), isz) != 0) {
        uint32_t k = 0;
        while (k < isz && tmp[k] == dev[ustart[b] - u_lo + k]) ++k;
        if (bad < 8) fprintf(stderr, "#decode_verify\tblock %u (clen %u isize %u): zlib rc %d, first difference at byte %u\n", b, in->block_clen[b], isz, zr, k);
        ++bad;
      }
    }
    inflateEnd(&zs);
    fprintf(stderr, "#decode_verify\t%u of %u blocks differ from zlib; %u inflated on the host\n", bad, data_end - first_block, out->n_blocks_host);
  }
  nvtx_declined.end();
  NvtxRange nvtx_chain("bgzf: record chain (guess, walk, verify, offsets)");
  // ---- record chain
  WalkArgs wa{};
  // The chain is walked over [first_block, walk_hi): one block past the range when there is one, so that the range's last
  // record boundary is also checked against an independent guess.
  const uint32_t walk_hi = std::min<uint32_t>(walk_end + 1, data_end);
  wa.data = infl_base; wa.total = total; wa.ustart = d.d_ustart; wa.first_block = first_block; wa.n_blocks = walk_hi;
  wa.records_at = in->records_at; wa.n_ref = (int32_t)in->n_ref; wa.guess = d.d_guess; wa.exit_off = d.d_exit; wa.n_rec = d.d_nrec;
  wa.n_cig = d.d_ncig; wa.dirty = d.d_dirty; wa.flags = d.d_cnt + 1; wa.only_dirty = 0;
  const uint32_t nwb = walk_hi - first_block;
  CU_TRY(c, cudaMemsetAsync(d.d_dirty, 0, 4ull * nb, c->stream));
  kd_guess<<<(nwb * 32 + 255) / 256, 256, 0, c->stream>>>(wa);
  kd_walk<<<(nwb + 127) / 128, 128, 0, c->stream>>>(wa);
  CU_TRY(c, cudaGetLastError());
  out->n_launches += 2;
  uint64_t h_exit = 0;
  for (uint32_t round = 0;; ++round) {
    if (nwb > 1) {
      CU_TRY(c, cudaMemsetAsync(d.d_cnt + 2, 0, 4, c->stream));
      kd_verify<<<(nwb - 1 + 255) / 256, 256, 0, c->stream>>>(wa);
      CU_TRY(c, cudaGetLastError());
      out->n_launches += 1;
    }
    CU_TRY(c, cudaMemcpyAsync(h_cnt, d.d_cnt, 64, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaMemcpyAsync(&h_exit, d.d_exit + (walk_end - 1), 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (nwb <= 1 || !h_cnt[2]) break;
    if (round >= 256) return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: record chain did not settle");
    out->chain_repairs += 1;
    out->n_launches += 1;
    wa.only_dirty = 1;
    kd_walk<<<(nwb + 127) / 128, 128, 0, c->stream>>>(wa);
    CU_TRY(c, cudaGetLastError());
  }
  if (walk_end == nb ? h_exit != stream_total : (h_exit == WALK_UNKNOWN || h_exit > total))
    return fail(c, CMB_E_DECLINED, walk_end == nb ? "cmb_submit_bgzf: record chain does not end at the end of the stream"
                                                  : "cmb_submit_bgzf: a record runs past the inflated tail of the block range");
  kd_scan_items<<<1, 1024, 0, c->stream>>>(d.d_nrec, d.d_ncig, first_block, walk_end, d.d_rec_base, d.d_cig_base, (uint64_t*)(d.d_cnt + 6));
  CU_TRY(c, cudaGetLastError());
  out->n_launches += 1;
  uint64_t totals[2] = {0, 0};
  CU_TRY(c, cudaMemcpyAsync(totals, d.d_cnt + 6, 16, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(c, cudaStreamSynchronize(c->stream));
  CU_TRY(c, cudaEventRecord(d.ev[3], c->stream));
  nvtx_chain.end();
  NvtxRange nvtx_extract("bgzf: extract, mate matching, K1");
  const uint64_t n_rec = totals[0], n_cig = totals[1];
  if (n_rec >= 0xffffff00ull || n_cig >= 0xffffff00ull) return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: more than 2^32 records or cigar operations");
  out->n_records = n_rec;
  out->n_intervals = n_cig;
  if (n_rec) {
    if ((rc = dec_grow(c, d.d_rec_off, d.rec_cap, (size_t)n_rec))) return rc;
    size_t offs[13];
    const size_t need = batch_slab_bytes((uint32_t)n_rec, (uint32_t)n_cig, offs);
    if (d.tuple_slab_bytes < need || !d.d_tuple_slab) {
      cudaFree(d.d_tuple_slab);
      d.d_tuple_slab = nullptr;
      d.tuple_slab_bytes = 0;
      const size_t want = need + need / 8;
      CU_TRY(c, cudaMalloc(&d.d_tuple_slab, want));
      d.tuple_slab_bytes = want;
    }
    cmb_read_batch tb;
    carve_batch(d.d_tuple_slab, (uint32_t)n_rec, (uint32_t)n_cig, &tb);
    d.last_n_rec = (uint32_t)n_rec;
    d.last_n_cig = (uint32_t)n_cig;
    OffsetArgs oa{};
    oa.data = infl_base; oa.ustart = d.d_ustart; oa.guess = d.d_guess; oa.rec_base = d.d_rec_base; oa.cig_base = d.d_cig_base;
    oa.first_block = first_block; oa.n_blocks = walk_end; oa.rec_off = d.d_rec_off; oa.iv_begin = tb.iv_begin; oa.n_records = n_rec; oa.n_cig_total = n_cig;
    kd_offsets<<<(walk_end - first_block + 127) / 128, 128, 0, c->stream>>>(oa);
    CU_TRY(c, cudaGetLastError());
    ExtractArgs ea{};
    ea.data = infl_base; ea.rec_off = d.d_rec_off; ea.n_records = n_rec;
    ea.own_lo = in->ranged ? in->own_tid_begin : INT_MIN; ea.own_hi = in->ranged ? in->own_tid_end : INT_MAX;
    ea.own_unplaced = in->ranged ? in->own_unplaced : 1u; ea.n_owned = (unsigned long long*)(d.d_cnt + 10);
    ea.tid = tb.tid; ea.pos = tb.pos; ea.flag = tb.flag; ea.mapq = tb.mapq; ea.nm_state = tb.nm_state; ea.nm = tb.nm; ea.l_seq = tb.l_seq;
    ea.aligned = tb.aligned; ea.del = tb.del; ea.ins = tb.ins; ea.iv_begin = tb.iv_begin; ea.iv_start = tb.iv_start; ea.iv_len = tb.iv_len;
    ea.n_primary = (unsigned long long*)(d.d_cnt + 4); ea.flags = d.d_cnt + 1;
    kd_extract<<<(uint32_t)((n_rec + 255) / 256), 256, 0, c->stream>>>(ea);
    CU_TRY(c, cudaGetLastError());
    out->n_launches += 2;
    CU_TRY(c, cudaMemcpyAsync(h_cnt, d.d_cnt, 64, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (h_cnt[1]) return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: malformed alignment record (flags %u)", h_cnt[1]);
    memcpy(&out->n_primary, h_cnt + 4, 8);
    memcpy(&out->n_records, h_cnt + 10, 8);  // records this call owns (all of them unless ranged)
    d.last_valid = true;
    d.last_mate = nullptr;
    d.last_infl_base = infl_base;
    // mate matching on the device (filter.rs:117-233; cmb_pairs.cuh): for coverage when the pair thresholds apply; for
    // `coverm filter` whenever the filter's pair path runs (everything but "single-read thresholds only", filter.rs:88)
    const bool need_mates = decode_only ? !(c->mode.filter_single_reads && !c->mode.filter_pairs) : (bool)c->mode.filter_pairs;
    if (need_mates) {
      if (d.pair_rec_cap < (size_t)n_rec || !d.d_pair_key) {
        cudaFree(d.d_filter_anchor); cudaFree(d.d_filter_role); cudaFree(d.d_filter_out);
    cudaFree(d.d_pair_key); cudaFree(d.d_pair_mate); cudaFree(d.d_pair_next);
        d.d_pair_key = nullptr; d.d_pair_mate = nullptr; d.d_pair_next = nullptr; d.pair_rec_cap = 0;
        const size_t want = (size_t)n_rec + (size_t)n_rec / 8 + 16;
        CU_TRY(c, cudaMalloc(&d.d_pair_key, 8 * want));
        CU_TRY(c, cudaMalloc(&d.d_pair_mate, 4 * want));
        CU_TRY(c, cudaMalloc(&d.d_pair_next, 4 * want));
        d.pair_rec_cap = want;
      }
      size_t table = 1u << 16;
      while (table < 2 * (size_t)n_rec) table <<= 1;
      if (d.pair_table_cap < table) {
        cudaFree(d.d_pair_tag); cudaFree(d.d_pair_head);
        d.d_pair_tag = nullptr; d.d_pair_head = nullptr; d.pair_table_cap = 0;
        CU_TRY(c, cudaMalloc(&d.d_pair_tag, 8 * table));
        CU_TRY(c, cudaMalloc(&d.d_pair_head, 4 * table));
        d.pair_table_cap = table;
      }
      CU_TRY(c, cudaMemsetAsync(d.d_pair_tag, 0, 8 * table, c->stream));
      CU_TRY(c, cudaMemsetAsync(d.d_pair_head, 0xff, 4 * table, c->stream));
      PairArgs pa{};
      pa.data = infl_base; pa.rec_off = d.d_rec_off; pa.n_records = (uint32_t)n_rec; pa.key = d.d_pair_key; pa.mate = d.d_pair_mate;
      pa.next = d.d_pair_next; pa.slot_tag = d.d_pair_tag; pa.slot_head = d.d_pair_head; pa.table_mask = (uint32_t)(table - 1);
      pa.flags = d.d_cnt + 1;
      const uint32_t gr = (uint32_t)((n_rec + 255) / 256);
      kd_pair_keys<<<gr, 256, 0, c->stream>>>(pa);
      kd_pair_insert<<<gr, 256, 0, c->stream>>>(pa);
      kd_pair_resolve<<<(uint32_t)((table + 255) / 256), 256, 0, c->stream>>>(pa);
      CU_TRY(c, cudaGetLastError());
      out->n_launches += 3;
      CU_TRY(c, cudaMemcpyAsync(h_cnt, d.d_cnt, 64, cudaMemcpyDeviceToHost, c->stream));
      CU_TRY(c, cudaStreamSynchronize(c->stream));
      if (h_cnt[1]) return fail(c, CMB_E_DECLINED, "cmb_submit_bgzf: mate matching gave up (flags %u)", h_cnt[1]);
      d.last_mate = d.d_pair_mate;
    }
    CU_TRY(c, cudaEventRecord(d.ev[4], c->stream));
    if (c->n_local && !decode_only) {
      // records that start before excl_end_block are this rank's exclusive share of the stream (cmb_kept_tid_range)
      uint32_t excl_n = 0xffffffffu;
      if (in->ranged && in->excl_end_block < walk_end) {
        if (in->excl_end_block <= first_block) excl_n = 0;
        else {
          uint64_t base = 0;
          CU_TRY(c, cudaMemcpyAsync(&base, d.d_rec_base + in->excl_end_block, 8, cudaMemcpyDeviceToHost, c->stream));
          CU_TRY(c, cudaStreamSynchronize(c->stream));
          excl_n = (uint32_t)base;
        }
      }
      d.last_excl_n = excl_n;
      rc = launch_k1(c, tb, (uint32_t)n_rec, (uint32_t)n_cig, excl_n, d.last_mate);
      if (rc) return rc;
    }
  } else {
    CU_TRY(c, cudaEventRecord(d.ev[4], c->stream));
  }
  CU_TRY(c, cudaEventRecord(d.ev[5], c->stream));
  CU_TRY(c, cudaEventSynchronize(d.ev[4]));
  cudaEventElapsedTime(&out->ms_copy_inflate, d.ev[0], d.ev[2]);
  cudaEventElapsedTime(&out->ms_chain, d.ev[2], d.ev[3]);
  cudaEventElapsedTime(&out->ms_extract, d.ev[3], d.ev[4]);
  cudaEventElapsedTime(&out->ms_total, d.ev[0], d.ev[4]);
  return CMB_OK;
}
}  // namespace
