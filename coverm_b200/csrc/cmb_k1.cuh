// K1: filter + delta accumulation, K1c: cross-block sortedness check (see cmb_device.cu header).
#pragma once
// ------------------------------------------------------------------------------------------------ K1
struct K1Args {
  // batch (device pointers)
  const int32_t* tid;
  const int32_t* pos;
  const uint16_t* flag;
  const uint8_t* mapq;
  const uint8_t* nm_state;
  const uint32_t* nm;
  const uint32_t* l_seq;
  const uint32_t* aligned;
  const uint32_t* del;
  const uint32_t* ins;
  const uint32_t* iv_begin;
  const int32_t* iv_start;
  const int32_t* iv_len;
  uint32_t n;
  // reference
  const uint32_t* off_span;  // [n_local+1]
  const uint32_t* len;       // [n_local]
  uint32_t n_contigs, tid_begin, tid_end;
  // outputs
  int32_t* arena;
  int32_t* tail_sum;
  cmb_contig_stats* rows;
  int2* block_minmax;  // per block {min kept tid, max kept tid} for the cross-block sortedness check
  uint32_t* error_flags;
  // cross-RANK half of the sortedness check (multi-GPU contig sharding only, else NULL): per block {min, max} kept tid of
  // the records with index < excl_n (INT_MAX / INT_MIN = none); k1c_check_sorted folds them into the rank's kept range
  int2* block_xrange;
  uint32_t excl_n;
  // per-gene coverage (genes.rs): the arena's segments are genes, records carry contig tids.  NULL = contig mode.
  const uint32_t* gene_first;   // [n_contigs + 1] first gene of each contig (genes sorted by (tid, start))
  const uint32_t* gene_start;   // [n_genes] gene range on its contig, clamped to the contig
  const uint32_t* gene_end;
  const uint32_t* gene_maxlen;  // [n_contigs] longest gene of the contig (bounds the backward search for overlaps)
  const uint32_t* contig_len;   // [n_contigs]
  uint8_t* contig_seen;         // [n_contigs] a kept record mapped here (genes.rs:220-246)
  unsigned long long* kept_primary;  // primaries among the kept records (ReadsMapped.num_mapped_reads, genes.rs:249-252)
  // pair path: partner of each record (cmb_pairs.cuh, records in file order) or NULL = the host layout (completed pairs
  // only, stored first mate at the even index, its partner right after)
  const int32_t* mate;
  // params
  cmb_params p;
  uint8_t filter_single, filter_pairs;
};

struct RecView {
  uint32_t flag, mapq, nm_state, nm, l_seq, aligned, del;
};

// filter.rs:243-279.  Sets *nm_err when the reference would reach nm() on a record without a usable NM tag.
__device__ __forceinline__ bool single_read_passes(const RecView& r, const cmb_params& p, bool* nm_err) {
  if (p.min_mapq != 255 && (r.mapq < p.min_mapq || r.mapq == 255)) return false;
  if (r.nm_state != 1) *nm_err = true;
  const float aligned_f = __uint2float_rn(r.aligned);
  return r.aligned >= p.min_aligned_length_single &&
         __fdiv_rn(aligned_f, __uint2float_rn(r.l_seq)) >= p.min_aligned_percent_single &&
         __fsub_rn(1.0f, __fdiv_rn(__uint2float_rn(r.nm), aligned_f)) >= p.min_percent_identity_single;
}
// filter.rs:281-336 (D is not part of the pair aligned length).
__device__ __forceinline__ bool read_pair_passes(const RecView& a, const RecView& b, const cmb_params& p, bool* nm_err) {
  if (p.min_mapq != 255 && (a.mapq < p.min_mapq || b.mapq < p.min_mapq || a.mapq == 255 || b.mapq == 255)) return false;
  if (a.nm_state != 1 || b.nm_state != 1) *nm_err = true;
  const uint32_t aligned = (a.aligned - a.del) + (b.aligned - b.del);
  const float aligned_f = __uint2float_rn(aligned);
  const float seq_f = __ull2float_rn((unsigned long long)a.l_seq + (unsigned long long)b.l_seq);
  const float edit_f = __ull2float_rn((unsigned long long)a.nm + (unsigned long long)b.nm);
  return aligned >= p.min_aligned_length_pair && __fdiv_rn(aligned_f, seq_f) >= p.min_aligned_percent_pair &&
         __fsub_rn(1.0f, __fdiv_rn(edit_f, aligned_f)) >= p.min_percent_identity_pair;
}

#ifndef CMB_K1_MINBLOCKS
#define CMB_K1_MINBLOCKS 6
#endif
__global__ void __launch_bounds__(K1_THREADS, CMB_K1_MINBLOCKS) k1_filter_accumulate(const K1Args a) {
  const uint32_t i = blockIdx.x * K1_THREADS + threadIdx.x;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool valid = i < a.n;
  const cmb_params& p = a.p;

  RecView r = {};
  int32_t tid = -1, pos = 0;
  uint32_t ins = 0, ivb = 0, ive = 0;
  if (valid) {
    tid = a.tid[i];
    pos = a.pos[i];
    r.flag = a.flag[i];
    r.mapq = a.mapq[i];
    r.nm_state = a.nm_state[i];
    r.nm = a.nm[i];
    r.l_seq = a.l_seq[i];
    r.aligned = a.aligned[i];
    r.del = a.del[i];
    ins = a.ins[i];
    ivb = a.iv_begin[i];
    ive = a.iv_begin[i + 1];
  }
  // K1 is latency-bound (a thread's loads form the chain columns -> intervals -> segment table -> REDs).  The segment of a
  // record depends on its tid only and its first aligned block on iv_begin only, so both are requested here, before the
  // filter arithmetic and the block-wide sortedness scan, and are in registers by the time the events are added.
  uint32_t pre_L = 0, pre_off0 = 0, pre_off1 = 0;
  int32_t pre_s = INT_MIN, pre_n = 0;
  const bool pre_seg = valid && !a.gene_first && tid >= 0 && (uint32_t)tid >= a.tid_begin && (uint32_t)tid < a.tid_end &&
                       (uint32_t)tid < a.n_contigs;
  if (pre_seg) {
    const uint32_t lc = (uint32_t)tid - a.tid_begin;
    pre_L = __ldg(a.len + lc);
    pre_off0 = __ldg(a.off_span + lc);
    pre_off1 = __ldg(a.off_span + lc + 1);
  }
  if (valid && ivb < ive) {
    pre_s = __ldg(a.iv_start + ivb);
    pre_n = __ldg(a.iv_len + ivb);
  }
  const bool unmapped = r.flag & 0x4, secondary = r.flag & 0x100, supplementary = r.flag & 0x800, proper = r.flag & 0x2;
  // FlagFilter::passes, lib.rs:67-78
  const bool flag_pass = !(secondary && !p.include_secondary) && !(supplementary && !p.include_supplementary) &&
                         !(!proper && !p.include_improper_pairs);
  bool keep = valid && flag_pass && !unmapped;  // contig.rs:119-125
  bool nm_err = false;
  if (valid && p.filtering) {
    bool passes;
    if (a.filter_single && !a.filter_pairs) {  // filter.rs:88-116
      const bool passes_filter1 = !unmapped && (p.include_supplementary || !supplementary) && (p.include_secondary || !secondary);
      passes = passes_filter1 && single_read_passes(r, p, &nm_err);
    } else {  // filter.rs:117-233: the host submits completed pairs only; stored first mate at the even index
      const int32_t mi = a.mate ? a.mate[i] : (int32_t)(i ^ 1u);
      const uint32_t m = (uint32_t)mi;
      RecView o = {};
      const bool have_mate = mi >= 0 && m < a.n;
      const bool i_is_second = a.mate ? m < i : (i & 1u);  // the stored first mate is the earlier record
      if (have_mate) {
        o.flag = a.flag[m];
        o.mapq = a.mapq[m];
        o.nm_state = a.nm_state[m];
        o.nm = a.nm[m];
        o.l_seq = a.l_seq[m];
        o.aligned = a.aligned[m];
        o.del = a.del[m];
      }
      const RecView& first = i_is_second ? o : r;   // record1 (stored)
      const RecView& second = i_is_second ? r : o;  // record (just read)
      bool ok = have_mate;
      if (ok && a.filter_single) ok = single_read_passes(first, p, &nm_err) && single_read_passes(second, p, &nm_err);
      if (ok) ok = read_pair_passes(second, first, p, &nm_err);
      passes = ok;
    }
    keep = keep && passes;
  }
  uint32_t err = 0;
  if (keep && r.nm_state != 1) nm_err = true;  // nm(&record), contig.rs:206
  if (nm_err) err |= ERR_NM;
  if (keep && (tid < 0 || (uint32_t)tid >= a.n_contigs)) {
    err |= ERR_TID;
    keep = false;
  }

  // ---- sortedness of the kept stream (contig.rs:128-132): prefix max over the block
  __shared__ int s_wmax[K1_THREADS / 32];
  __shared__ int s_wmin[K1_THREADS / 32];
  {
    const int key = keep ? tid : INT_MIN;
    int pm = key;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(FULL, pm, d);
      if ((int)lane >= d) pm = max(pm, o);
    }
    int excl = __shfl_up_sync(FULL, pm, 1);
    if (lane == 0) excl = INT_MIN;
    int kmin = keep ? tid : INT_MAX;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) kmin = min(kmin, __shfl_xor_sync(FULL, kmin, d));
    if (lane == 31) s_wmax[warp] = pm;
    if (lane == 0) s_wmin[warp] = kmin;
    __shared__ int s_xmax[K1_THREADS / 32];
    __shared__ int s_xmin[K1_THREADS / 32];
    if (a.block_xrange) {
      const bool xk = keep && i < a.excl_n;
      const int xmax = __reduce_max_sync(FULL, xk ? tid : INT_MIN);
      const int xmin = __reduce_min_sync(FULL, xk ? tid : INT_MAX);
      if (lane == 0) {
        s_xmax[warp] = xmax;
        s_xmin[warp] = xmin;
      }
    }
    __syncthreads();
    if (a.block_xrange && threadIdx.x == 0) {
      int xmax = INT_MIN, xmin = INT_MAX;
      for (uint32_t w = 0; w < K1_THREADS / 32; ++w) {
        xmax = max(xmax, s_xmax[w]);
        xmin = min(xmin, s_xmin[w]);
      }
      a.block_xrange[blockIdx.x] = make_int2(xmin, xmax);
    }
    int before = INT_MIN;
    for (uint32_t w = 0; w < warp; ++w) before = max(before, s_wmax[w]);
    if (keep && tid < max(before, excl)) err |= ERR_UNSORTED;
    if (threadIdx.x == 0) {
      int bmax = INT_MIN, bmin = INT_MAX;
      for (uint32_t w = 0; w < K1_THREADS / 32; ++w) {
        bmax = max(bmax, s_wmax[w]);
        bmin = min(bmin, s_wmin[w]);
      }
      a.block_minmax[blockIdx.x] = make_int2(bmin, bmax);
    }
  }

  // +1 at `s` and -1 at `e` (when e lies inside the segment) of segment `lc`, plus the chunk tail sums K1b scans
  auto add_events_in = [&](uint32_t L, uint32_t off0, uint32_t off1, uint32_t s, uint64_t e) {
    const uint64_t base = (uint64_t)off0 * SPAN;
    const uint64_t end_padded = (uint64_t)off1 * SPAN;  // first element of the next segment
    const uint64_t gs = base + s;
    const bool has_end = e < L;  // "True unless the read hits the contig end"
    atomicAdd(a.arena + gs, 1);
    const uint64_t ks = gs / CHUNK;
    const bool cont_s = end_padded > (ks + 1) * (uint64_t)CHUNK;  // this segment continues past chunk ks
    if (has_end) {
      const uint64_t ge = base + e;
      atomicAdd(a.arena + ge, -1);
      const uint64_t ke = ge / CHUNK;
      if (ke != ks) {
        if (cont_s) atomicAdd(a.tail_sum + ks, 1);
        if (end_padded > (ke + 1) * (uint64_t)CHUNK) atomicAdd(a.tail_sum + ke, -1);
      }
    } else if (cont_s) {
      atomicAdd(a.tail_sum + ks, 1);
    }
  };
  auto add_events = [&](uint32_t lc, uint32_t s, uint64_t e) { add_events_in(a.len[lc], a.off_span[lc], a.off_span[lc + 1], s, e); };

  if (a.gene_first) {
    // ---- per-gene coverage (genes.rs:182-344, 467-552).  A gene's delta array is the contig's, cut to [start, end) with the
    //      running depth at `start` as its first element: exactly what clipping every aligned block to the gene gives.  Reads
    //      are assigned to the genes that contain their leftmost position.
    if (keep) {
      const bool primary = !secondary && !supplementary;
      a.contig_seen[tid] = 1;
      if (primary) atomicAdd(a.kept_primary, 1ull);
      const uint32_t CL = a.contig_len[tid];
      uint64_t ref_end = (uint32_t)pos;  // end of the last aligned block
      for (uint32_t k = ivb; k < ive; ++k) {
        const int32_t s = a.iv_start[k];
        if (s == INT_MIN) continue;
        if (s < 0 || (uint32_t)s >= CL) {  // `ups_and_downs[cursor] += 1` would panic
          err |= ERR_BOUNDS;
          continue;
        }
        ref_end = max(ref_end, (uint64_t)(uint32_t)s + (uint32_t)a.iv_len[k]);
      }
      const uint32_t g0 = a.gene_first[tid], g1 = a.gene_first[tid + 1];
      if (g0 < g1 && !(err & ERR_BOUNDS)) {
        const uint32_t maxlen = a.gene_maxlen[tid];
        const uint32_t from = (uint32_t)pos >= maxlen ? (uint32_t)pos - maxlen + 1 : 0;  // a gene starting earlier ends at or before pos
        uint32_t lo = g0, hi = g1;  // first gene with start >= from
        while (lo < hi) {
          const uint32_t mid = (lo + hi) >> 1;
          if (a.gene_start[mid] < from) lo = mid + 1;
          else hi = mid;
        }
        const uint64_t indels = (uint64_t)ins + r.del;
        for (uint32_t g = lo; g < g1; ++g) {
          const uint32_t gsx = a.gene_start[g], gex = a.gene_end[g];
          if ((uint64_t)gsx >= max(ref_end, (uint64_t)(uint32_t)pos + 1)) break;  // genes are sorted by start
          if ((uint32_t)pos >= gsx && (uint32_t)pos < gex) {  // read_starts.partition_point range (genes.rs:518-523)
            cmb_contig_stats* row = a.rows + g;
            atomicAdd((unsigned long long*)&row->n_records, 1ull);
            if (primary) atomicAdd((unsigned long long*)&row->n_primary, 1ull);
            const uint64_t mis = r.nm >= indels ? r.nm - indels : 0;  // edit.saturating_sub(indels), genes.rs:297
            if (mis) atomicAdd((unsigned long long*)&row->sum_edit, (unsigned long long)mis);
            if (primary && r.aligned > 0) atomicAdd(&row->sum_identity_primary, ((double)r.aligned - (double)r.nm) / (double)r.aligned);
          }
          for (uint32_t k = ivb; k < ive; ++k) {
            const int32_t s = a.iv_start[k];
            if (s == INT_MIN) continue;
            const uint64_t e = (uint64_t)(uint32_t)s + (uint32_t)a.iv_len[k];
            if (e <= gsx || (uint32_t)s >= gex) continue;  // no overlap
            const uint32_t cs = max((uint32_t)s, gsx) - gsx;
            add_events(g, cs, e - gsx);  // e - gsx >= gene length: the block runs past the gene, no -1
          }
        }
      }
    }
    err = __reduce_or_sync(FULL, err);
    if (err && lane == 0) atomicOr(a.error_flags, err);
    return;
  }

  const bool mine = keep && (uint32_t)tid >= a.tid_begin && (uint32_t)tid < a.tid_end;
  // ---- per-contig read counters (contig.rs:157-159, 204-211; genome.rs:173-174, 220-223, 677-682, 724-727)
  {
    const bool primary = !secondary && !supplementary;
    const uint64_t c_rec = mine ? 1 : 0, c_pri = (mine && primary) ? 1 : 0, c_ns = (mine && !supplementary) ? 1 : 0;
    const uint64_t c_edit = mine ? r.nm : 0, c_indel = mine ? (uint64_t)ins + r.del : 0;
    double idn = 0.0;
    if (mine && r.aligned > 0) idn = ((double)r.aligned - (double)r.nm) / (double)r.aligned;
    const double id_pri = primary ? idn : 0.0, id_ns = !supplementary ? idn : 0.0;
    const uint32_t mine_mask = __ballot_sync(FULL, mine);
    if (mine_mask) {
      const int leader = __ffs(mine_mask) - 1;
      const int ltid = __shfl_sync(FULL, tid, leader);
      const bool uniform = __all_sync(FULL, !mine || tid == ltid);
      if (uniform) {
        const uint64_t s_rec = warp_sum_u64(c_rec), s_pri = warp_sum_u64(c_pri), s_ns = warp_sum_u64(c_ns),
                       s_edit = warp_sum_u64(c_edit), s_indel = warp_sum_u64(c_indel);
        double s_idp = id_pri, s_idn = id_ns;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          s_idp += __shfl_xor_sync(FULL, s_idp, d);
          s_idn += __shfl_xor_sync(FULL, s_idn, d);
        }
        if ((int)lane == leader) {
          cmb_contig_stats* row = a.rows + ltid;
          atomicAdd((unsigned long long*)&row->n_records, (unsigned long long)s_rec);
          if (s_pri) atomicAdd((unsigned long long*)&row->n_primary, (unsigned long long)s_pri);
          if (s_ns) atomicAdd((unsigned long long*)&row->n_nonsupp, (unsigned long long)s_ns);
          if (s_edit) atomicAdd((unsigned long long*)&row->sum_edit, (unsigned long long)s_edit);
          if (s_indel) atomicAdd((unsigned long long*)&row->sum_indel, (unsigned long long)s_indel);
          if (s_idp != 0.0) atomicAdd(&row->sum_identity_primary, s_idp);
          if (s_idn != 0.0) atomicAdd(&row->sum_identity_nonsupp, s_idn);
        }
      } else if (mine) {
        cmb_contig_stats* row = a.rows + tid;
        atomicAdd((unsigned long long*)&row->n_records, 1ull);
        if (c_pri) atomicAdd((unsigned long long*)&row->n_primary, 1ull);
        if (c_ns) atomicAdd((unsigned long long*)&row->n_nonsupp, 1ull);
        if (c_edit) atomicAdd((unsigned long long*)&row->sum_edit, (unsigned long long)c_edit);
        if (c_indel) atomicAdd((unsigned long long*)&row->sum_indel, (unsigned long long)c_indel);
        if (id_pri != 0.0) atomicAdd(&row->sum_identity_primary, id_pri);
        if (id_ns != 0.0) atomicAdd(&row->sum_identity_nonsupp, id_ns);
      }
    }
  }

  // ---- delta events (contig.rs:171-186)
  if (mine) {
    const uint32_t L = pre_L, off0 = pre_off0, off1 = pre_off1;
    for (uint32_t k = ivb; k < ive; ++k) {
      const int32_t s = k == ivb ? pre_s : a.iv_start[k];
      const uint32_t n = (uint32_t)(k == ivb ? pre_n : a.iv_len[k]);
      if (s == INT_MIN) continue;  // CMB_IV_PAD: unused slot of the interval pool
      if (s < 0 || (uint32_t)s >= L) {  // `ups_and_downs[cursor] += 1` would panic
        err |= ERR_BOUNDS;
        continue;
      }
      add_events_in(L, off0, off1, (uint32_t)s, (uint64_t)(uint32_t)s + n);
    }
  }
  err = __reduce_or_sync(FULL, err);
  if (err && lane == 0) atomicOr(a.error_flags, err);
}

// Cross-block sortedness: block b's smallest kept tid must be >= every earlier block's largest.
// With block_xrange (multi-GPU): also folds the blocks' exclusive kept tid ranges into kept_range[0] = max tid + 1 (0 = none),
// kept_range[1] = INT_MAX - min tid.
__global__ void __launch_bounds__(1024) k1c_check_sorted(const int2* block_minmax, uint32_t n_blocks, uint32_t* error_flags,
                                                         const int2* block_xrange, uint32_t* kept_range) {
  __shared__ int s_max[1024];
  const uint32_t t = threadIdx.x;
  const uint32_t per = (n_blocks + 1023) / 1024;
  const uint32_t b0 = t * per, b1 = min(n_blocks, b0 + per);
  if (block_xrange) {
    int xmin = INT_MAX, xmax = INT_MIN;
    for (uint32_t b = b0; b < b1; ++b) {
      const int2 x = block_xrange[b];
      xmin = min(xmin, x.x);
      xmax = max(xmax, x.y);
    }
    xmin = __reduce_min_sync(FULL, xmin);
    xmax = __reduce_max_sync(FULL, xmax);
    if ((t & 31) == 0 && xmax != INT_MIN) {
      atomicMax(kept_range + 0, (uint32_t)xmax + 1u);
      atomicMax(kept_range + 1, (uint32_t)(INT_MAX - xmin));
    }
  }
  int lmax = INT_MIN;
  bool bad = false;
  for (uint32_t b = b0; b < b1; ++b) {
    const int2 mm = block_minmax[b];
    if (mm.x != INT_MAX && mm.x < lmax) bad = true;
    lmax = max(lmax, mm.y);
  }
  s_max[t] = lmax;
  __syncthreads();
  int before = INT_MIN;
  for (uint32_t k = 0; k < t; ++k) before = max(before, s_max[k]);
  for (uint32_t b = b0; b < b1 && !bad; ++b) {
    const int2 mm = block_minmax[b];
    if (mm.x != INT_MAX && mm.x < before) bad = true;
  }
  if (bad) atomicOr(error_flags, ERR_UNSORTED);
}

