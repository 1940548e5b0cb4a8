// K2: segmented prefix sum of the delta arena + every O(L) reduction of EST::add_contig, one pass, HBM-bound.
//
// Persistent CTAs (CMB_K2_MINBLOCKS = 3 per SM, 256 threads).  CTA b works on the 8192-element chunks b, b + gridDim.x, ...
// (a static schedule) and keeps a K2_STAGES-deep ring (2 by default) of 32 KB tiles in flight with TMA
// (cp.async.bulk.tensor.2d, 128B swizzle, mbarrier complete_tx).  Since every thread knows its next chunk, the chunk's
// metadata is loaded an iteration ahead and the contig lookup of a span runs while its tile is still arriving.  A thread
// owns one 32-element span (one tile row: 8 x LDS.128, conflict-free through the swizzle) and re-zeroes the 16-byte units
// of the arena that hold an event, so the arena is clean again for the next sample; contigs start on span boundaries,
// so a span never straddles two contigs.  Running depth at a span = chunk carry (K1b) + segmented warp/CTA scan of the
// span totals.  Depth is piecewise constant and deltas are sparse (~1-2 % of positions), so a thread only keeps the
// span total and a 32-bit mask of its non-zero positions; covered bases, sum of depth and the depth histogram of the
// end-trimmed window are then accumulated per RUN in a short loop over the set bits (the deltas are re-read from the
// shared-memory tile, which stays resident until the next iteration's barrier).  The histogram lives in shared memory
// per (contig slot, depth % 128) with the high depth bits as a tag, and is flushed as (depth,count) records while the
// next chunk is being scanned (double-buffered: one __syncthreads per chunk).
#pragma once

struct K2Args {
  const uint32_t* off_span;
  const uint32_t* len;
  const uint32_t* chunk_first;
  const int32_t* carry_in;
  cmb_contig_stats* rows;
  uint32_t tid_begin, n_local, n_chunks, excl;
  int32_t* arena;
  uint2* rec;
  uint32_t rec_capacity;
  uint32_t* rec_count;
  uint2* warp_table;  // [n_chunks * HIST_SLOTS] {offset, count}: records of contig slot w of the chunk
  uint4* ovf;         // {contig_local, depth, count, next} — per-chunk linked lists
  uint32_t* ovf_head; // [n_chunks] list heads (OVF_NIL = empty)
  uint32_t ovf_capacity;
  uint32_t* ovf_count;
  uint32_t* error_flags;
};

constexpr uint32_t K2_SMEM_STAGE_BYTES = K2_STAGES * CHUNK_BYTES;
constexpr uint32_t K2_SMEM_MISC = 64 /*barriers*/ + 2 * K2_WARPS * 8 /*warp aggregates, double-buffered*/;
constexpr uint32_t K2_SMEM_BYTES_HIST = K2_SMEM_STAGE_BYTES + K2_SMEM_MISC + 2 * HIST_TOTAL * 4;
constexpr uint32_t K2_SMEM_BYTES_NOHIST = K2_SMEM_STAGE_BYTES + K2_SMEM_MISC;

template <bool HIST>
__global__ void __launch_bounds__(K2_THREADS, CMB_K2_MINBLOCKS) k2_scan_reduce(const __grid_constant__ CUtensorMap tmap, const K2Args a) {
  extern __shared__ __align__(1024) uint8_t smem[];  // stage tiles need the 1024 B swizzle-atom alignment
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + K2_SMEM_STAGE_BYTES);
  int2* wagg2 = reinterpret_cast<int2*>(smem + K2_SMEM_STAGE_BYTES + 64);
  uint32_t* hist2 = reinterpret_cast<uint32_t*>(wagg2 + 2 * K2_WARPS);

  const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;

  // Static schedule: iteration i of CTA b works on chunk b + i * gridDim.x.  Every thread knows its next chunk, so the chunk's
  // metadata (first / last contig, carry-in) is requested one iteration ahead and the dependent lookups (contig of the span,
  // its start and length) can start before the tile has even arrived.
  auto chunk_of = [&](uint32_t i) -> uint32_t { return blockIdx.x + i * gridDim.x; };
  auto issue = [&](uint32_t s, uint32_t ck) {  // thread 0: start the TMA load of chunk ck into stage s
    if (ck < a.n_chunks) {
      const uint32_t bar = smem_u32(full + s);
      mbar_arrive_expect_tx(bar, CHUNK_BYTES);
      tma_load_2d(smem_u32(smem + s * CHUNK_BYTES), &tmap, 0, (int32_t)(ck * CHUNK_ROWS), bar);
    }
  };

  // flush one histogram buffer: a warp takes contig slots warp, warp + K2_WARPS, ... (128 bins, 4 per lane) -> (depth,count) records
  auto flush_hist = [&](uint32_t* hist, uint32_t chunk, uint32_t n_slots) {
    for (uint32_t sl = warp; sl < HIST_SLOTS && sl < n_slots; sl += K2_WARPS) {
      uint32_t word[4], msk[4], total = 0;
#pragma unroll
      for (uint32_t k = 0; k < 4; ++k) {
        word[k] = hist[sl * HIST_BINS + lane + 32 * k];
        msk[k] = __ballot_sync(FULL, word[k] != 0);
        total += __popc(msk[k]);
      }
      uint32_t base = 0;
      if (total) {
        if (lane == 0) base = atomicAdd(a.rec_count, total);
        base = __shfl_sync(FULL, base, 0);
        const bool fits = (uint64_t)base + total <= a.rec_capacity;
        if (!fits && lane == 0) atomicOr(a.error_flags, ERR_CAPACITY);
        uint32_t before = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          if (word[k]) {
            const uint32_t depth = ((word[k] >> HIST_CNT_BITS) - 1) * HIST_BINS + lane + 32 * k;
            if (fits) a.rec[base + before + __popc(msk[k] & ((1u << lane) - 1))] = make_uint2(depth, word[k] & ((1u << HIST_CNT_BITS) - 1));
            hist[sl * HIST_BINS + lane + 32 * k] = 0;
          }
          before += __popc(msk[k]);
        }
        if (!fits) total = 0;
      }
      if (lane == 0) a.warp_table[(uint64_t)chunk * HIST_SLOTS + sl] = make_uint2(base, total);
    }
  };

  if (t == 0) {
    for (uint32_t s = 0; s < K2_STAGES; ++s) mbar_init(smem_u32(full + s), 1);
    fence_barrier_init();
  }
  if (HIST)
    for (uint32_t b = t; b < 2 * HIST_TOTAL; b += K2_THREADS) hist2[b] = 0;
  __syncthreads();
  if (t == 0)
    for (uint32_t s = 0; s < K2_STAGES; ++s) issue(s, chunk_of(s));
  __syncthreads();

  static_assert(SPAN == ROW_ELEMS, "a span is one 128-byte tile row");
  constexpr uint32_t UNITS = SPAN / 4;  // 16-byte units per span
  const uint32_t row = t;               // the tile row of this thread's span
  // byte offset inside a stage tile of element e of this thread's span
  auto elem_off = [&](uint32_t e) -> uint32_t {
    const uint32_t idx = e >> 2;
    const uint32_t r = row + (idx >> 3);
    return r * 128 + (((idx & 7) ^ (r & 7)) << 4) + ((e & 3) << 2);
  };
  const uint32_t E = a.excl;
  uint32_t prev_chunk = 0, prev_slots = 0;
  uint32_t n_cf = 0, n_cl = 0;  // metadata of the NEXT iteration's chunk, requested an iteration ahead
  int n_cin = 0;
  if (chunk_of(0) < a.n_chunks) {
    n_cf = __ldg(a.chunk_first + chunk_of(0));
    n_cl = __ldg(a.chunk_first + chunk_of(0) + 1);
    n_cin = __ldg(a.carry_in + chunk_of(0));
  }
  uint32_t it = 0;

  for (;; ++it) {
    const uint32_t s = it % K2_STAGES;
    const uint32_t chunk = chunk_of(it);
    if (chunk >= a.n_chunks) break;
    const uint32_t cf = n_cf, cl = n_cl;
    const int cin = n_cin;
    {
      const uint32_t nx = chunk_of(it + 1);
      if (nx < a.n_chunks) {
        n_cf = __ldg(a.chunk_first + nx);
        n_cl = __ldg(a.chunk_first + nx + 1);
        n_cin = __ldg(a.carry_in + nx);
      }
    }
    // ---- which contig owns this thread's span (needs no tile data: these loads fly while the tile arrives and is scanned)
    const uint32_t span = chunk * CHUNK_SPANS + t;
    uint32_t c;
    {
      uint32_t lo = cf, hi = cl;
      while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (__ldg(a.off_span + mid) <= span) lo = mid;
        else hi = mid - 1;
      }
      c = lo;
    }
    const uint32_t cstart = __ldg(a.off_span + c);
    const uint32_t L = __ldg(a.len + c);
    mbar_wait(smem_u32(full + s), (it / K2_STAGES) & 1);
    int2* wagg = wagg2 + (it & 1) * K2_WARPS;
    uint32_t* hist = hist2 + (it & 1) * HIST_TOTAL;

    // ---- SPAN consecutive deltas per thread: LDS.128s through the 128B swizzle (conflict-free).
    //      Only their sum and the mask of non-zero positions stay in registers.
    const uint8_t* tilep = smem + s * CHUNK_BYTES;
    int total = 0;
    uint32_t ev = 0;
    {
      int4* g = reinterpret_cast<int4*>(a.arena + (uint64_t)span * SPAN);
#pragma unroll
      for (uint32_t j = 0; j < UNITS; ++j) {
        const int4 q = *reinterpret_cast<const int4*>(tilep + row * 128 + ((j ^ (row & 7)) << 4));
        const uint32_t e4 = (q.x != 0 ? 1u : 0u) | (q.y != 0 ? 2u : 0u) | (q.z != 0 ? 4u : 0u) | (q.w != 0 ? 8u : 0u);
        total += (q.x + q.y) + (q.z + q.w);
        ev |= e4 << (4 * j);
        if (e4) g[j] = make_int4(0, 0, 0, 0);  // re-zero only the 16 B units that hold an event
      }
    }

    const bool is_head = span == cstart;
    const uint32_t rel = (span - cstart) * SPAN;  // position in the contig of the span's first element
    const uint32_t n_in = rel >= L ? 0u : min(SPAN, L - rel);
    uint32_t w0 = 0, w1 = 0;
    if (2ull * E < L) {
      const uint32_t ws = E, we = L - E;
      w0 = rel >= ws ? 0u : min(SPAN, ws - rel);
      w1 = rel >= we ? 0u : min(SPAN, we - rel);
      if (w1 < w0) w1 = w0;
    }

    // ---- segmented (by contig head) inclusive scan of span totals across the warp
    int val = total;
    int flg = is_head;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int ov = __shfl_up_sync(FULL, val, d);
      const int of = __shfl_up_sync(FULL, flg, d);
      if ((int)lane >= d) {
        if (!flg) val += ov;
        flg |= of;
      }
    }
    int pval = __shfl_up_sync(FULL, val, 1), pflg = __shfl_up_sync(FULL, flg, 1);
    if (lane == 0) {
      pval = 0;
      pflg = 0;
    }
    if (lane == 31) wagg[warp] = make_int2(val, flg);
    __syncthreads();  // warp aggregates visible; the previous iteration's tile and histogram adds are complete
    if (it > 0) {
      if (t == 0) issue((it - 1) % K2_STAGES, chunk_of(it - 1 + K2_STAGES));  // refill the tile of the previous iteration
      if (HIST) flush_hist(hist2 + ((it & 1) ^ 1) * HIST_TOTAL, prev_chunk, prev_slots);
    }

    int wv, wf;
    {
      const int2 wa = lane < K2_WARPS ? wagg[lane] : make_int2(0, 0);
      wv = wa.x;
      wf = wa.y;
#pragma unroll
      for (int d = 1; d < (int)K2_WARPS; d <<= 1) {
        const int ov = __shfl_up_sync(FULL, wv, d);
        const int of = __shfl_up_sync(FULL, wf, d);
        if ((int)lane >= d) {
          if (!wf) wv += ov;
          wf |= of;
        }
      }
      const int src = warp ? (int)warp - 1 : 0;
      wv = __shfl_sync(FULL, wv, src);
      wf = __shfl_sync(FULL, wf, src);
      if (warp == 0) {
        wv = 0;
        wf = 0;
      }
    }
    int carry;
    if (is_head) carry = 0;
    else if (pflg) carry = pval;
    else if (wf) carry = wv + pval;
    else carry = cin + wv + pval;

    // ---- reductions over this span (EST:393-404, 447-465, 494-501), run by run
    uint32_t cov_full = 0, cov_win = 0;
    uint64_t sum_win = 0;
    const uint32_t slot = c - cf;
    auto hist_add = [&](int depth, uint32_t cnt) {
      // direct-mapped bin (depth % 128) holding (depth / 128 + 1) << 14 | count: conflict-free while the depths of one
      // contig inside one chunk span < 128 values, wherever that range sits
      if (depth < 0) {  // impossible for a consistent arena (every -1 follows its +1 within the contig)
        atomicOr(a.error_flags, ERR_INTERNAL);
        return;
      }
      bool done = false;
      if (slot < HIST_SLOTS && (uint32_t)depth < HIST_MAX_DEPTH) {
        uint32_t* w = hist + slot * HIST_BINS + ((uint32_t)depth & (HIST_BINS - 1));
        const uint32_t tag = ((uint32_t)depth / HIST_BINS) + 1;
        uint32_t cur = *(volatile uint32_t*)w;
        if (cur == 0) cur = atomicCAS(w, 0u, (tag << HIST_CNT_BITS) | cnt);
        if (cur == 0) done = true;  // we installed tag and count
        else if ((cur >> HIST_CNT_BITS) == tag) {
          atomicAdd(w, cnt);
          done = true;
        }
      }
      if (!done) {  // > 16 contigs in the chunk, or two depths 128 apart in one chunk: per-chunk overflow list
        const uint32_t o = atomicAdd(a.ovf_count, 1u);
        if (o < a.ovf_capacity) {
          const uint32_t next = atomicExch(a.ovf_head + chunk, o);
          a.ovf[o] = make_uint4(c, (uint32_t)depth, cnt, next);
        } else {
          atomicOr(a.error_flags, ERR_CAPACITY);
        }
      }
    };
    // a run [from, to) of the span at one depth, clipped to the contig and to its end-trimmed window
    auto close_run = [&](int depth, uint32_t from, uint32_t to) {
      const uint32_t nc = min(to, n_in) - min(from, n_in);
      const uint32_t nw = min(max(to, w0), w1) - min(max(from, w0), w1);
      if (depth > 0) {
        cov_full += nc;
        cov_win += nw;
      }
      if (nw) {
        sum_win += (uint64_t)(int64_t)depth * nw;
        if (HIST) hist_add(depth, nw);
      }
    };
    if (ev) {
      int depth = carry;
      uint32_t from = 0;
      uint32_t m = ev;
      while (m) {
        const uint32_t j = (uint32_t)__ffs((int)m) - 1;
        m &= m - 1;
        close_run(depth, from, j);
        depth += *reinterpret_cast<const int*>(tilep + elem_off(j));  // the delta at position j
        from = j;
      }
      close_run(depth, from, SPAN);
    } else {  // no event in the span: constant depth
      const uint32_t nc = n_in, nw = w1 - w0;
      if (carry > 0) {
        cov_full += nc;
        cov_win += nw;
      }
      sum_win += (uint64_t)(int64_t)carry * nw;
    }
    if (HIST) {
      // event-free spans: aggregate the lanes that agree with the first such lane into one shared-memory atomic
      const uint32_t nw = w1 - w0;
      const bool cand = ev == 0 && nw > 0;
      const uint32_t cm = __ballot_sync(FULL, cand);
      if (cm) {
        const int leader = __ffs(cm) - 1;
        const int d0 = __shfl_sync(FULL, carry, leader);
        const uint32_t c0 = __shfl_sync(FULL, c, leader);
        const bool same = cand && carry == d0 && c == c0;
        const uint32_t m = __ballot_sync(FULL, same);
        if (same) {
          const uint32_t tot = __reduce_add_sync(m, nw);
          if ((int)lane == leader) hist_add(carry, tot);
        } else if (cand) {
          hist_add(carry, nw);
        }
      }
    }

    // ---- per-contig accumulation: one RED triple per (warp, contig)
    {
      const uint32_t c0 = __shfl_sync(FULL, c, 0);
      if (__all_sync(FULL, c == c0)) {
        const uint32_t sf = __reduce_add_sync(FULL, cov_full), sw = __reduce_add_sync(FULL, cov_win);
        const uint64_t sd = warp_sum_u64(sum_win);
        if (lane == 0) {
          cmb_contig_stats* rowp2 = a.rows + a.tid_begin + c0;
          if (sf) atomicAdd((unsigned long long*)&rowp2->covered_full, (unsigned long long)sf);
          if (sw) atomicAdd((unsigned long long*)&rowp2->covered_window, (unsigned long long)sw);
          if (sd) atomicAdd((unsigned long long*)&rowp2->sum_depth_window, (unsigned long long)sd);
        }
      } else {
        cmb_contig_stats* rowp2 = a.rows + a.tid_begin + c;
        if (cov_full) atomicAdd((unsigned long long*)&rowp2->covered_full, (unsigned long long)cov_full);
        if (cov_win) atomicAdd((unsigned long long*)&rowp2->covered_window, (unsigned long long)cov_win);
        if (sum_win) atomicAdd((unsigned long long*)&rowp2->sum_depth_window, (unsigned long long)sum_win);
      }
    }
    prev_chunk = chunk;
    prev_slots = cl - cf + 1;
  }
  if (HIST && it > 0) {
    __syncthreads();  // the last chunk's histogram adds
    flush_hist(hist2 + ((it & 1) ^ 1) * HIST_TOTAL, prev_chunk, prev_slots);
  }
}
