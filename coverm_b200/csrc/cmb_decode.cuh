// Device-side BAM decode (SURVEY §8f-1): the compressed BGZF blocks cross PCIe, the GPU inflates them, finds the record
// boundaries and reduces every record to the cmb_read_batch tuple K1 consumes.  Replaces, for the stream (non-pair) path,
// htslib's bgzf_read + bam_read1 behind BamFileNamedReader::read (bam_generator.rs:103-134).
//
//   KD1 kd_inflate   one warp per BGZF block (RFC 1951); kd_inflate_g8 (cmb_decode_g8.cuh) takes four blocks per warp and
//                    kd_inflate_t1 (cmb_decode_t1.cuh) one block per lane; this form is CMB_INFLATE=w1 (see inflate_kind).
//                    All 32 lanes run the decoder redundantly (uniform control flow), which turns the lanes into
//                    resources: the compressed bytes are held as a 2 x 128-byte register window fetched with
//                    coalesced loads and read with shuffles; length/distance base tables live one entry per lane;
//                    LZ77 matches are copied by all lanes; Huffman tables (10-bit root + 5-bit subtables, u16
//                    entries) are built cooperatively in shared memory.  The block's CRC-32 is then
//                    checked against the BGZF footer (per-lane slices combined in GF(2)).
//   KD2 kd_guess     one warp per block: the first offset >= the block start from which a chain of plausible record
//                    headers runs (records straddle blocks freely).
//   KD3 kd_walk      one thread per block: follow block_size from the guess to the block end -> exit offset, counts.
//   KD4 kd_verify    guess[i] must equal exit[i-1]; a mismatch is repaired and the block re-walked (host loop).
//   KD5 kd_scan_items / kd_offsets   record and interval bases per block, then per-record offsets.
//   KD6 kd_extract   one thread per record: fixed fields, CIGAR walk (contig.rs:166-202 operands), NM aux (lib.rs:138-158).
// Anything this path cannot vouch for (table overflow, malformed stream, implausible chain) is *declined* before K1
// touches the arena; the caller then runs the host decoder, which raises the reference's error if there is one.
#pragma once

// ------------------------------------------------------------------------------------------------ KD1 inflate
constexpr uint32_t INF_WARPS = 16;  // warps per CTA
constexpr uint32_t INF_ROOT = 10, INF_SUBBITS = 5;
constexpr uint32_t INF_SUBQ = 128;  // distinct root-bit prefixes of codes longer than the root
constexpr uint32_t INF_LIT_ENTRIES = (1u << INF_ROOT) + 512;  // zlib's ENOUGH bound for (286, root 10, max 15) is 1024 + 308
constexpr uint32_t INF_DST_ENTRIES = (1u << INF_ROOT) + 128;
constexpr uint32_t INF_OK = 0, INF_DECLINED = 1;

struct InfWarpSmem {
  uint16_t lit[INF_LIT_ENTRIES];  // entry: symbol << 4 | bits ; or 0x8000 | subtable_offset << 4 | subtable index bits
  uint16_t dst[INF_DST_ENTRIES];
  uint8_t lens[320];
  uint16_t codes[320];
  uint32_t nc[16];
  uint32_t subq[INF_SUBQ];  // per long-code prefix: longest remainder, then subtable offset << 4 | bits
  uint32_t overflow;
  uint32_t pad[3];
};
constexpr uint32_t INF_SMEM_BYTES = INF_WARPS * sizeof(InfWarpSmem) + 4 * 256 * 4 /* CRC-32 slicing tables */;

__constant__ uint16_t c_len_base[32] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258, 0, 0, 0};
__constant__ uint8_t c_len_extra[32] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0, 0, 0, 0};
__constant__ uint16_t c_dist_base[32] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577, 0, 0};
__constant__ uint8_t c_dist_extra[32] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13, 0, 0};
__constant__ uint8_t c_clen_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct InflateArgs {
  const uint8_t* comp;   // the whole file in device memory (>= 512 readable bytes after the end)
  const uint64_t* coff;  // per block: offset of the deflate payload
  const uint32_t* clen;  // its length
  const uint32_t* isize; // uncompressed size (BGZF footer)
  const uint64_t* uoff;  // offset in the inflated stream
  uint32_t b0, b1;
  uint8_t* out;
  uint32_t* status;
  uint32_t* ticket;
  uint32_t* fail_count;
  // the kernel runs while the file is still arriving: block b may be read once ready[block_window[b]] != 0
  // (written by the copy stream after the window's bytes; NULL = everything is resident)
  const uint32_t* block_window;
  const uint32_t* ready;
  uint32_t lane_limit;  // kd_inflate_t1: lanes per warp that take blocks (0 = all 32)
  // optional indirection: ticket t in [b0, b1) names block block_list[t] (second pass over the blocks the first declined)
  const uint32_t* block_list;
  uint8_t* scratch;  // kd_inflate_t1: 160 bytes per BGZF block (indexed by block number)
};

// The compressed stream seen through a 64-bit bit buffer; words come from a per-lane register window.
struct BitReader {
  const uint32_t* base;  // 128-byte aligned
  uint32_t wcur, wnext;  // this lane's word of the current / next 128-byte line
  uint32_t widx;         // next word to take (uniform across the warp)
  uint64_t buf;
  uint32_t cnt;

  __device__ __forceinline__ uint32_t next_word(uint32_t lane) {
    const uint32_t w = __shfl_sync(FULL, wcur, widx & 31);
    ++widx;
    if ((widx & 31) == 0) {
      wcur = wnext;
      wnext = __ldcg(base + widx + 32 + lane);
    }
    return w;
  }
  __device__ __forceinline__ void init(const uint8_t* p, uint32_t lane) {
    const uintptr_t a = (uintptr_t)p;
    base = (const uint32_t*)(a & ~(uintptr_t)127);
    const uint32_t skip = (uint32_t)(a & 127);
    // L2-only loads: the bytes are written by the copy engine while this kernel runs, and the look-ahead of an earlier
    // block may have touched this line before its window arrived (a stale L1 copy would be read back)
    wcur = __ldcg(base + lane);
    wnext = __ldcg(base + 32 + lane);
    widx = skip >> 2;
    const uint32_t drop = (skip & 3) * 8;
    const uint32_t w = next_word(lane);
    buf = (uint64_t)(w >> drop);
    cnt = 32 - drop;
    refill(lane);
  }
  __device__ __forceinline__ void refill(uint32_t lane) {
    if (cnt <= 32) {
      buf |= (uint64_t)next_word(lane) << cnt;
      cnt += 32;
    }
  }
  __device__ __forceinline__ void consume(uint32_t n) {
    buf >>= n;
    cnt -= n;
  }
  __device__ __forceinline__ uint32_t bits(uint32_t n) const { return (uint32_t)buf & ((1u << n) - 1); }
  // address of the first byte not yet (even partially) consumed; exact when cnt is a multiple of 8
  __device__ __forceinline__ const uint8_t* byte_pos() const { return (const uint8_t*)base + (((uint64_t)widx * 32 - cnt) >> 3); }
  __device__ __forceinline__ const uint8_t* byte_pos_ceil() const { return (const uint8_t*)base + (((uint64_t)widx * 32 - cnt + 7) >> 3); }
};

// Canonical Huffman table from code lengths (lens[0..n), values 0..15) into tab: 2^root direct entries, then one
// subtable per root-bit prefix shared by longer codes, sized by the longest code under that prefix.  Canonical codes of
// increasing length are numerically increasing, so the prefixes of the long codes are the contiguous range [P0, 2^root)
// (MSB-first); q = prefix - P0 indexes the small per-prefix scratch array.
// Returns false on an over-subscribed code or when the subtables do not fit.
__device__ bool inf_build_table(InfWarpSmem& S, const uint8_t* lens, uint32_t n, uint16_t* tab, uint32_t root, uint32_t n_entries, uint32_t lane) {
  for (uint32_t i = lane; i < n_entries / 2; i += 32) reinterpret_cast<uint32_t*>(tab)[i] = 0;
  // lane L counts the codes of length L
  uint32_t cnt = 0;
  for (uint32_t s = 0; s < n; ++s) cnt += (lens[s] == lane) ? 1u : 0u;
  if (lane == 0 || lane > 15) cnt = 0;
  uint32_t code = 0, my_first = 0;
  int left = 1;
  bool over = false;
  for (uint32_t L = 1; L <= 15; ++L) {
    code = (code + __shfl_sync(FULL, cnt, L - 1)) << 1;
    if (lane == L) my_first = code;
    left = (left << 1) - (int)__shfl_sync(FULL, cnt, L);
    if (left < 0) over = true;
  }
  if (over) return false;
  const uint32_t P0 = __shfl_sync(FULL, my_first, root + 1) >> 1;
  if (lane < 16) S.nc[lane] = my_first;
  for (uint32_t q = lane; q < INF_SUBQ; q += 32) S.subq[q] = 0;
  if (lane == 0) S.overflow = 0;
  __syncwarp();
  const uint32_t root_size = 1u << root;
  bool any_long = false;
  for (uint32_t base = 0; base < n; base += 32) {
    const uint32_t s = base + lane;
    const uint32_t L = s < n ? lens[s] : 0;
    const uint32_t mask = __match_any_sync(FULL, L);
    const uint32_t rank = __popc(mask & ((1u << lane) - 1));
    const uint32_t leader = __ffs(mask) - 1;
    const uint32_t c0 = S.nc[L & 15];
    __syncwarp();
    if (lane == leader && L) S.nc[L] = c0 + __popc(mask);
    __syncwarp();
    const uint32_t cd = c0 + rank;
    if (s < n) S.codes[s] = (uint16_t)cd;
    if (L && L <= root) {
      const uint32_t rev = __brev(cd) >> (32 - L);
      const uint16_t e = (uint16_t)((s << 4) | L);
      for (uint32_t i = rev; i < root_size; i += 1u << L) tab[i] = e;
    } else if (L > root) {
      const uint32_t q = (cd >> (L - root)) - P0;
      if (q < INF_SUBQ) atomicMax(&S.subq[q], L - root);
      else S.overflow = 1;
    }
    any_long = any_long || __any_sync(FULL, L > root);
  }
  __syncwarp();
  if (any_long) {
    uint32_t running = 0;
    for (uint32_t qb = 0; qb < INF_SUBQ; qb += 32) {
      const uint32_t r = S.subq[qb + lane];
      const uint32_t sz = r ? (1u << r) : 0;
      uint32_t incl = sz;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(FULL, incl, d);
        if ((int)lane >= d) incl += o;
      }
      const uint32_t off = running + incl - sz;
      if (r) {
        if (root_size + off + sz <= n_entries) {
          const uint32_t slot = __brev(P0 + qb + lane) >> (32 - root);
          tab[slot] = (uint16_t)(0x8000u | ((root_size + off) << 4) | r);
        } else {
          S.overflow = 1;
        }
      }
      S.subq[qb + lane] = (off << 4) | r;
      running += __shfl_sync(FULL, incl, 31);
    }
    __syncwarp();
    if (S.overflow == 0) {
      for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t s = base + lane;
        const uint32_t L = s < n ? lens[s] : 0;
        if (L > root) {
          const uint32_t cd = S.codes[s];
          const uint32_t v = S.subq[(cd >> (L - root)) - P0];
          const uint32_t r = v & 15, off = v >> 4, rem = L - root;
          const uint32_t rev = __brev(cd) >> (32 - L);
          const uint16_t e = (uint16_t)((s << 4) | rem);
          for (uint32_t i = rev >> root; i < (1u << r); i += 1u << rem) tab[root_size + off + i] = e;
        }
      }
    }
  }
  __syncwarp();
  return S.overflow == 0;
}

// Inflate one BGZF block with the whole warp.  Returns INF_OK, or a non-zero code naming the check that declined the block.
__device__ uint32_t inf_block(InfWarpSmem& S, const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t n_out, uint32_t lane,
                              uint32_t lbase_r, uint32_t lext_r, uint32_t dbase_r, uint32_t dext_r) {
  BitReader br;
  br.init(in, lane);
  const uint8_t* const in_end = in + in_len;
  uint32_t op = 0;
  for (;;) {
    if (br.byte_pos_ceil() > in_end) return 1u /* declined */;  // ran past the block: not a well-formed stream
    br.refill(lane);
    const uint32_t bfinal = br.bits(1);
    const uint32_t btype = ((uint32_t)br.buf >> 1) & 3;
    br.consume(3);
    if (btype == 0) {
      br.consume(br.cnt & 7);
      br.refill(lane);
      const uint32_t len = (uint32_t)br.buf & 0xffff, nlen = ((uint32_t)br.buf >> 16) & 0xffff;
      br.consume(32);
      if ((len ^ nlen) != 0xffff) return 2u /* declined */;
      const uint8_t* src = br.byte_pos();
      if (src + len > in_end || op + len > n_out) return 3u /* declined */;
      for (uint32_t i = lane; i < len; i += 32) out[op + i] = __ldcg(src + i);
      op += len;
      br.init(src + len, lane);
    } else if (btype == 3) {
      return 4u /* declined */;
    } else {
      uint32_t hlit, hdist;
      if (btype == 1) {
        hlit = 288;
        hdist = 32;
        for (uint32_t i = lane; i < 320; i += 32) S.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
        __syncwarp();
      } else {
        br.refill(lane);
        hlit = br.bits(5) + 257;
        hdist = (((uint32_t)br.buf >> 5) & 31) + 1;
        const uint32_t hclen = (((uint32_t)br.buf >> 10) & 15) + 4;
        br.consume(14);
        if (hlit > 286 || hdist > 30) return 5u /* declined */;
        if (lane < 19) S.lens[lane] = 0;
        __syncwarp();
        for (uint32_t i = 0; i < hclen; ++i) {
          br.refill(lane);
          if (lane == 0) S.lens[c_clen_order[i]] = (uint8_t)br.bits(3);
          br.consume(3);
        }
        __syncwarp();
        if (!inf_build_table(S, S.lens, 19, S.dst, 7, 128, lane)) return 6u /* declined */;
        const uint32_t total = hlit + hdist;
        uint32_t n = 0, prev = 0;
        while (n < total) {
          br.refill(lane);
          const uint32_t e = S.dst[(uint32_t)br.buf & 127];
          const uint32_t l = e & 15;
          if (!l) return 7u /* declined */;
          br.consume(l);
          const uint32_t sym = e >> 4;
          if (sym < 16) {
            if (lane == 0) S.lens[n] = (uint8_t)sym;
            prev = sym;
            ++n;
          } else {
            uint32_t rep, val = 0;
            if (sym == 16) {
              if (n == 0) return 8u /* declined */;
              val = prev;
              rep = 3 + br.bits(2);
              br.consume(2);
            } else if (sym == 17) {
              rep = 3 + br.bits(3);
              br.consume(3);
            } else {
              rep = 11 + br.bits(7);
              br.consume(7);
            }
            if (n + rep > total) return 9u /* declined */;
            for (uint32_t i = lane; i < rep; i += 32) S.lens[n + i] = (uint8_t)val;
            prev = val;
            n += rep;
          }
        }
        __syncwarp();
        if (S.lens[256] == 0) return 10u /* declined */;
      }
      // the distance lengths follow the literal/length ones in S.lens; build dist first from a copy-free view
      if (!inf_build_table(S, S.lens + hlit, hdist, S.dst, INF_ROOT, INF_DST_ENTRIES, lane)) return 11u /* declined */;
      if (!inf_build_table(S, S.lens, hlit, S.lit, INF_ROOT, INF_LIT_ENTRIES, lane)) return 12u /* declined */;
      // ---- symbols
      for (;;) {
        br.refill(lane);
        uint32_t e = S.lit[(uint32_t)br.buf & ((1u << INF_ROOT) - 1)];
        if (e & 0x8000) {
          br.consume(INF_ROOT);
          e = S.lit[((e >> 4) & 0x7ff) + br.bits(e & 15)];
        }
        uint32_t l = e & 15;
        if (!l) return 13u /* declined */;
        br.consume(l);
        uint32_t sym = (e >> 4) & 0x1ff;
        if (sym < 256) {
          if (op >= n_out) return 14u /* declined */;
          if (lane == 0) out[op] = (uint8_t)sym;
          ++op;
          continue;
        }
        if (sym == 256) break;
        sym -= 257;
        if (sym > 28) return 15u /* declined */;
        const uint32_t xl = __shfl_sync(FULL, lext_r, sym);
        const uint32_t len = __shfl_sync(FULL, lbase_r, sym) + br.bits(xl);
        br.consume(xl);
        br.refill(lane);
        e = S.dst[(uint32_t)br.buf & ((1u << INF_ROOT) - 1)];
        if (e & 0x8000) {
          br.consume(INF_ROOT);
          e = S.dst[((e >> 4) & 0x7ff) + br.bits(e & 15)];
        }
        l = e & 15;
        if (!l) return 16u /* declined */;
        br.consume(l);
        const uint32_t dsym = (e >> 4) & 0x1ff;
        if (dsym > 29) return 17u /* declined */;
        const uint32_t xd = __shfl_sync(FULL, dext_r, dsym);
        const uint32_t dist = __shfl_sync(FULL, dbase_r, dsym) + br.bits(xd);
        br.consume(xd);
        if (dist > op || op + len > n_out) return 18u /* declined */;
        __syncwarp();  // earlier stores of other lanes are visible to the loads below
        uint8_t* dstp = out + op;
        const uint8_t* srcp = dstp - dist;
        if (dist >= len) {
          for (uint32_t i = lane; i < len; i += 32) dstp[i] = srcp[i];
        } else {
          for (uint32_t i = lane; i < len; i += 32) dstp[i] = srcp[i % dist];
        }
        op += len;
      }
    }
    if (bfinal) break;
  }
  if (op != n_out) return 19u /* declined */;
  if (br.byte_pos_ceil() > in_end) return 20u /* declined */;  // consumed bits that are not part of the block
  return INF_OK;
}

// ---- CRC-32 (ISO-HDLC, the gzip/BGZF checksum; reflected polynomial 0xEDB88320) of a block's output, by the whole warp:
// every lane checksums a 2 KB slice with slicing-by-4 tables, then the slices are combined through the linearity of the
// CRC: crc(A||B) = crc(A) * x^(8|B|) mod P  xor  crc(B)  (polynomial arithmetic over GF(2), bit 31 = x^0).
constexpr uint32_t CRC_POLY = 0xedb88320u;
constexpr uint32_t CRC_SLICE = 2048;
constexpr uint32_t INF_CRC_TABLE_BYTES = 4 * 256 * 4;

__device__ __forceinline__ uint32_t gf2_mulmod(uint32_t a, uint32_t b) {  // a(x) * b(x) mod P(x)
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1) ? (b >> 1) ^ CRC_POLY : b >> 1;
  }
  return p;
}
__device__ uint32_t gf2_x_pow_8n(uint32_t n_bytes) {  // x^(8 n) mod P by square and multiply
  uint32_t sq = 0x00800000u;  // x^8: x^0 is bit 31, x^k is bit 31-k
  uint32_t r = 1u << 31;
  while (n_bytes) {
    if (n_bytes & 1) r = gf2_mulmod(sq, r);
    sq = gf2_mulmod(sq, sq);
    n_bytes >>= 1;
  }
  return r;
}
__device__ uint32_t warp_crc32(const uint8_t* data, uint32_t n, const uint32_t* T, uint32_t lane) {
  const uint32_t b0 = min(n, lane * CRC_SLICE), b1 = min(n, (lane + 1) * CRC_SLICE);
  uint32_t c = 0;
  if (b1 > b0) {
    const uint8_t* p = data + b0;
    const uint8_t* e = data + b1;
    c = 0xffffffffu;
    while (p < e && ((uintptr_t)p & 3)) c = T[(c ^ __ldcg(p++)) & 0xff] ^ (c >> 8);
    for (; p + 4 <= e; p += 4) {
      c ^= __ldcg(reinterpret_cast<const uint32_t*>(p));
      c = T[768 + (c & 0xff)] ^ T[512 + ((c >> 8) & 0xff)] ^ T[256 + ((c >> 16) & 0xff)] ^ T[c >> 24];
    }
    while (p < e) c = T[(c ^ __ldcg(p++)) & 0xff] ^ (c >> 8);
    c = ~c;
    c = gf2_mulmod(gf2_x_pow_8n(n - b1), c);
  }
  return __reduce_xor_sync(FULL, c);
}

__global__ void __launch_bounds__(INF_WARPS * 32, 2) kd_inflate(const InflateArgs a) {
  extern __shared__ __align__(16) uint8_t inf_smem[];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  InfWarpSmem& S = reinterpret_cast<InfWarpSmem*>(inf_smem)[warp];
  uint32_t* crcT = reinterpret_cast<uint32_t*>(inf_smem + INF_WARPS * sizeof(InfWarpSmem));
  if (threadIdx.x < 256) {
    uint32_t c = threadIdx.x;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
    crcT[threadIdx.x] = c;
  }
  __syncthreads();
  if (threadIdx.x < 256) {
    uint32_t c = crcT[threadIdx.x];
    for (int k = 1; k < 4; ++k) {
      c = crcT[c & 0xff] ^ (c >> 8);
      crcT[k * 256 + threadIdx.x] = c;
    }
  }
  __syncthreads();
  const uint32_t lbase_r = c_len_base[lane], lext_r = c_len_extra[lane], dbase_r = c_dist_base[lane], dext_r = c_dist_extra[lane];
  for (;;) {
    uint32_t b = 0;
    if (lane == 0) b = a.b0 + atomicAdd(a.ticket, 1u);
    b = __shfl_sync(FULL, b, 0);
    if (b >= a.b1) break;
    if (a.block_list) b = a.block_list[b];
    bool arrived = true;
    if (a.ready) {
      const volatile uint32_t* flag = a.ready + a.block_window[b];
      uint32_t spins = 0;
      unsigned long long waited_ns = 0;
      while (*flag == 0 && waited_ns < 4000000000ull) {  // bounded (4 s): a copy that never lands must not hang the GPU
        const uint32_t ns = 256u << min(spins, 4u);      // 0.25 .. 4 us back-off; the warp has nothing else to do
        __nanosleep(ns);
        waited_ns += ns;
        ++spins;
      }
      arrived = __all_sync(FULL, *flag != 0);
      __threadfence_system();  // order the payload reads behind the flag (written by the copy engine after the window's bytes)
    }
    const uint32_t n_out = a.isize[b];
    uint32_t st = arrived ? INF_OK : 31u;
    if (n_out && arrived) {
      const uint8_t* in = a.comp + a.coff[b];
      const uint32_t in_len = a.clen[b];
      st = inf_block(S, in, in_len, a.out + a.uoff[b], n_out, lane, lbase_r, lext_r, dbase_r, dext_r);
      __syncwarp();
      if (st == INF_OK) {  // htslib verifies the block's CRC32 (bgzf.c); so do we, from the footer that follows the payload
        const uint8_t* f = in + in_len;
        const uint32_t want = (uint32_t)__ldcg(f) | ((uint32_t)__ldcg(f + 1) << 8) | ((uint32_t)__ldcg(f + 2) << 16) | ((uint32_t)__ldcg(f + 3) << 24);
        if (warp_crc32(a.out + a.uoff[b], n_out, crcT, lane) != want) st = 30u;
      }
    }
    __syncwarp();
    if (lane == 0) {
      a.status[b] = st;
      if (st != INF_OK) atomicAdd(a.fail_count, 1u);
    }
  }
}

// ------------------------------------------------------------------------------------------------ record chain
constexpr uint64_t WALK_UNKNOWN = ~0ull;      // no guess / no valid exit
constexpr uint32_t GUESS_SCAN_LIMIT = 1u << 20;  // bytes scanned for a first record boundary
constexpr uint32_t DEC_ERR_CHAIN = 1u, DEC_ERR_RECORD = 2u, DEC_ERR_AUX = 4u;

__device__ __forceinline__ uint32_t ldu32(const uint8_t* p) {
  const uintptr_t a = (uintptr_t)p;
  const uint32_t* q = (const uint32_t*)(a & ~(uintptr_t)3);
  const uint32_t sh = (uint32_t)(a & 3) * 8;
  const uint32_t lo = q[0];
  if (sh == 0) return lo;
  return __funnelshift_r(lo, q[1], sh);
}
__device__ __forceinline__ uint32_t ldu16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

struct WalkArgs {
  const uint8_t* data;   // inflated stream (>= 8 readable bytes after `total`)
  uint64_t total;
  const uint64_t* ustart;  // per block, n_blocks + 1 entries
  uint32_t first_block;    // block holding the first record
  uint32_t n_blocks;
  uint64_t records_at;
  int32_t n_ref;
  uint64_t* guess;
  uint64_t* exit_off;
  uint32_t* n_rec;
  uint32_t* n_cig;
  uint32_t* dirty;
  uint32_t* flags;  // [0] error bits, [1] changed
  uint32_t only_dirty;
};

// A BAM record header that could be real (same tests as the host decoder, decode_runner.hpp `plausible`).
__device__ __forceinline__ bool rec_plausible(const uint8_t* d, uint64_t s, uint64_t total, int32_t n_ref) {
  if (s + 36 > total) return false;
  const uint8_t* r = d + s;
  const uint32_t bs = ldu32(r);
  if (bs < 32 || bs > (64u << 20)) return false;
  const int32_t tid = (int32_t)ldu32(r + 4), pos = (int32_t)ldu32(r + 8), mtid = (int32_t)ldu32(r + 24);
  if (tid < -1 || tid >= n_ref || mtid < -1 || mtid >= n_ref || pos < -1) return false;
  const uint32_t l_name = r[12], n_cig = ldu16(r + 16), l_seq = ldu32(r + 20);
  if (l_name == 0 || l_seq > (1u << 28)) return false;
  const uint64_t fixed = 32ull + l_name + 4ull * n_cig + (l_seq + 1) / 2 + l_seq;
  if (fixed > bs) return false;
  if (s + 36 + l_name <= total && r[36 + l_name - 1] != 0) return false;
  return true;
}

__global__ void __launch_bounds__(256) kd_guess(const WalkArgs a) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t b = a.first_block + (blockIdx.x * 256 + threadIdx.x) / 32;
  if (b >= a.n_blocks) return;
  if (b == a.first_block) {
    if (lane == 0) a.guess[b] = a.records_at;
    return;
  }
  const uint64_t u0 = a.ustart[b];
  if (u0 >= a.total) {  // trailing empty blocks (the BGZF EOF marker)
    if (lane == 0) a.guess[b] = a.total;
    return;
  }
  const uint64_t limit = min(a.total, u0 + GUESS_SCAN_LIMIT);
  uint64_t found = WALK_UNKNOWN;
  for (uint64_t s0 = u0; s0 < limit; s0 += 32) {
    const uint64_t s = s0 + lane;
    bool ok = s < limit && rec_plausible(a.data, s, a.total, a.n_ref);
    if (ok) {  // a run of six consistent headers (or reaching the end of the stream) confirms the guess
      uint64_t q = s;
      for (int hop = 0; hop < 6; ++hop) {
        if (q == a.total) break;
        if (!rec_plausible(a.data, q, a.total, a.n_ref)) {
          ok = false;
          break;
        }
        q += 4ull + ldu32(a.data + q);
      }
    }
    const uint32_t m = __ballot_sync(FULL, ok);
    if (m) {
      found = s0 + (uint32_t)(__ffs(m) - 1);
      break;
    }
  }
  if (lane == 0) a.guess[b] = found;
}

__global__ void __launch_bounds__(128) kd_walk(const WalkArgs a) {
  const uint32_t b = a.first_block + blockIdx.x * 128 + threadIdx.x;
  if (b >= a.n_blocks) return;
  if (a.only_dirty && !a.dirty[b]) return;
  a.dirty[b] = 0;
  uint64_t pos = a.guess[b];
  const uint64_t end = a.ustart[b + 1];
  uint32_t n = 0, cig = 0;
  if (pos != WALK_UNKNOWN) {
    while (pos < end) {
      if (pos + 36 > a.total) {
        pos = WALK_UNKNOWN;
        break;
      }
      const uint32_t bs = ldu32(a.data + pos);
      if (bs < 32 || pos + 4ull + bs > a.total) {
        pos = WALK_UNKNOWN;
        break;
      }
      cig += ldu16(a.data + pos + 16);
      ++n;
      pos += 4ull + bs;
    }
  }
  a.exit_off[b] = pos;
  a.n_rec[b] = n;
  a.n_cig[b] = cig;
}

__global__ void __launch_bounds__(256) kd_verify(const WalkArgs a) {
  const uint32_t b = a.first_block + 1 + blockIdx.x * 256 + threadIdx.x;
  if (b >= a.n_blocks) return;
  const uint64_t want = a.exit_off[b - 1];
  if (a.guess[b] != want) {
    a.guess[b] = want;
    a.dirty[b] = 1;
    atomicOr(a.flags + 1, 1u);
  }
}

// Exclusive scan of the per-block record / cigar-op counts (single CTA).  totals[0] = records, totals[1] = cigar ops.
__global__ void __launch_bounds__(1024) kd_scan_items(const uint32_t* n_rec, const uint32_t* n_cig, uint32_t first_block, uint32_t n_blocks,
                                                      uint64_t* rec_base, uint64_t* cig_base, uint64_t* totals) {
  __shared__ uint64_t s_rec[1024], s_cig[1024];
  const uint32_t t = threadIdx.x;
  const uint32_t n = n_blocks - first_block;
  const uint32_t per = (n + 1023) / 1024;
  const uint32_t i0 = min(n, t * per), i1 = min(n, i0 + per);
  uint64_t r = 0, c = 0;
  for (uint32_t i = i0; i < i1; ++i) {
    r += n_rec[first_block + i];
    c += n_cig[first_block + i];
  }
  s_rec[t] = r;
  s_cig[t] = c;
  __syncthreads();
  for (uint32_t d = 1; d < 1024; d <<= 1) {
    const uint64_t ar = t >= d ? s_rec[t - d] : 0, ac = t >= d ? s_cig[t - d] : 0;
    __syncthreads();
    s_rec[t] += ar;
    s_cig[t] += ac;
    __syncthreads();
  }
  uint64_t rb = s_rec[t] - r, cb = s_cig[t] - c;
  for (uint32_t i = i0; i < i1; ++i) {
    rec_base[first_block + i] = rb;
    cig_base[first_block + i] = cb;
    rb += n_rec[first_block + i];
    cb += n_cig[first_block + i];
  }
  if (t == 1023) {
    totals[0] = s_rec[1023];
    totals[1] = s_cig[1023];
  }
}

struct OffsetArgs {
  const uint8_t* data;
  const uint64_t* ustart;
  const uint64_t* guess;
  const uint64_t* rec_base;
  const uint64_t* cig_base;
  uint32_t first_block, n_blocks;
  uint64_t* rec_off;   // [n_records]
  uint32_t* iv_begin;  // [n_records + 1]
  uint64_t n_records, n_cig_total;
};

__global__ void __launch_bounds__(128) kd_offsets(const OffsetArgs a) {
  const uint32_t b = a.first_block + blockIdx.x * 128 + threadIdx.x;
  if (b >= a.n_blocks) return;
  uint64_t pos = a.guess[b];
  const uint64_t end = a.ustart[b + 1];
  uint64_t r = a.rec_base[b];
  uint64_t c = a.cig_base[b];
  while (pos < end) {
    a.rec_off[r] = pos;
    a.iv_begin[r] = (uint32_t)c;
    c += ldu16(a.data + pos + 16);
    ++r;
    pos += 4ull + ldu32(a.data + pos);
  }
  if (b == a.n_blocks - 1) a.iv_begin[a.n_records] = (uint32_t)a.n_cig_total;
}

// ------------------------------------------------------------------------------------------------ KD6 extract
struct ExtractArgs {
  const uint8_t* data;
  const uint64_t* rec_off;
  uint64_t n_records;
  // SoA output (device cmb_read_batch)
  int32_t* tid;
  int32_t* pos;
  uint16_t* flag;
  uint8_t* mapq;
  uint8_t* nm_state;
  uint32_t* nm;
  uint32_t* l_seq;
  uint32_t* aligned;
  uint32_t* del;
  uint32_t* ins;
  const uint32_t* iv_begin;
  int32_t* iv_start;
  int32_t* iv_len;
  unsigned long long* n_primary;
  uint32_t* flags;
  // counters cover the records this call OWNS: own_lo <= tid < own_hi, plus tid < 0 when own_unplaced (multi-GPU: the walks
  // of neighbouring ranks overlap by a block; each record is counted by exactly one rank)
  int32_t own_lo, own_hi;
  uint32_t own_unplaced;
  unsigned long long* n_owned;
};

__global__ void __launch_bounds__(256) kd_extract(const ExtractArgs a) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  const bool valid = i < a.n_records;
  uint32_t err = 0;
  bool primary = false, owned = false;
  if (valid) {
    const uint8_t* rec = a.data + a.rec_off[i];
    const uint32_t block_size = ldu32(rec);
    const uint8_t* o = rec + 4;
    const uint8_t* end = o + block_size;
    const int32_t tid = (int32_t)ldu32(o), pos = (int32_t)ldu32(o + 4);
    const uint32_t w2 = ldu32(o + 8), w3 = ldu32(o + 12), l_seq = ldu32(o + 16);
    const uint32_t l_read_name = w2 & 0xff, mapq = (w2 >> 8) & 0xff, n_cigar = w3 & 0xffff, flag = w3 >> 16;
    a.tid[i] = tid;
    a.pos[i] = pos;
    a.flag[i] = (uint16_t)flag;
    a.mapq[i] = (uint8_t)mapq;
    a.l_seq[i] = l_seq;
    owned = tid < 0 ? a.own_unplaced != 0 : (tid >= a.own_lo && tid < a.own_hi);
    primary = owned && !(flag & 0x900);
    const uint8_t* cig = o + 32 + l_read_name;
    const uint8_t* aux = cig + 4ull * n_cigar + (l_seq + 1) / 2 + l_seq;
    uint32_t iv = a.iv_begin[i];
    const uint32_t iv_end = a.iv_begin[i + 1];
    uint32_t aligned = 0, del = 0, ins = 0;
    bool placeholder = false;
    if (aux > end) {
      err |= DEC_ERR_RECORD;
    } else {
      if (n_cigar) {
        const uint32_t v0 = ldu32(cig);
        placeholder = (v0 & 0xf) == 4 && (v0 >> 4) == l_seq && tid >= 0 && pos >= 0;
      }
      long long cursor = pos;
      for (uint32_t k = 0; k < n_cigar; ++k) {
        const uint32_t v = ldu32(cig + 4 * k);
        const uint32_t op = v & 0xf, len = v >> 4;
        if (op == 0 || op == 7 || op == 8) {  // M, =, X: contig.rs:171-186
          a.iv_start[iv] = cursor < 0 ? -1 : (int32_t)min(cursor, (long long)INT_MAX);
          a.iv_len[iv] = (int32_t)len;
          ++iv;
          cursor += len;
          aligned += len;
        } else if (op == 2) {  // D
          cursor += len;
          del += len;
          aligned += len;
        } else if (op == 3) {  // N
          cursor += len;
        } else if (op == 1) {  // I
          ins += len;
          aligned += len;
        }
      }
    }
    for (; iv < iv_end; ++iv) {  // unused part of the interval reservation
      a.iv_start[iv] = INT_MIN;
      a.iv_len[iv] = 0;
    }
    a.aligned[i] = aligned;
    a.del[i] = del;
    a.ins[i] = ins;
    // NM aux: first NM tag wins; types C/S/I are integers the reference accepts (lib.rs:139-156)
    uint32_t nm_state = 0, nm = 0;
    const uint8_t* p = aux;
    while (!err && p + 3 <= end) {
      const uint32_t t0 = p[0], t1 = p[1], ty = p[2];
      p += 3;
      uint64_t sz;
      if (ty == 'A' || ty == 'c' || ty == 'C') sz = 1;
      else if (ty == 's' || ty == 'S') sz = 2;
      else if (ty == 'i' || ty == 'I' || ty == 'f') sz = 4;
      else if (ty == 'Z' || ty == 'H') {
        const uint8_t* e = p;
        while (e < end && *e) ++e;
        sz = e < end ? (uint64_t)(e - p) + 1 : (uint64_t)(end - p);
      } else if (ty == 'B') {
        if (p + 5 > end) sz = (uint64_t)(end - p);
        else {
          const uint32_t sub = p[0], cnt = ldu32(p + 1);
          const uint64_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
          sz = 5 + es * (uint64_t)cnt;
        }
      } else {
        err |= DEC_ERR_AUX;
        break;
      }
      if (t0 == 'N' && t1 == 'M' && nm_state == 0) {
        if (ty == 'C') { nm_state = 1; nm = p[0]; }
        else if (ty == 'S') { nm_state = 1; nm = ldu16(p); }
        else if (ty == 'I') { nm_state = 1; nm = ldu32(p); }
        else nm_state = 2;
      }
      // A CG:B,I tag behind a `<l_seq>S...` placeholder is the real CIGAR of a read with > 65535 operations (htslib
      // bam_tag2cigar): its intervals do not fit the n_cigar_op reservation, so the stream goes to the host decoder.
      if (t0 == 'C' && t1 == 'G' && ty == 'B' && placeholder) err |= DEC_ERR_RECORD;
      p += sz;
    }
    a.nm_state[i] = (uint8_t)nm_state;
    a.nm[i] = nm;
  }
  const uint32_t np = __popc(__ballot_sync(FULL, primary)), no = __popc(__ballot_sync(FULL, owned));
  if ((threadIdx.x & 31) == 0 && np) atomicAdd(a.n_primary, (unsigned long long)np);
  if ((threadIdx.x & 31) == 0 && no) atomicAdd(a.n_owned, (unsigned long long)no);
  err = __reduce_or_sync(FULL, err);
  if (err && (threadIdx.x & 31) == 0) atomicOr(a.flags, err);
}
