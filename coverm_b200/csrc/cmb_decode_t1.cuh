// kd_inflate_t1: DEFLATE with ONE THREAD PER BGZF BLOCK.
//
// A DEFLATE stream is a serial chain (the position of every symbol depends on the one before), so the parallelism of a
// BAM file lies ACROSS its 64 KB BGZF blocks -- there are tens of thousands of them.  kd_inflate_g8 spends a warp on
// four blocks (18.8 warp instructions per output byte, issue-bound); here every lane of a warp runs its own block, so one
// issued instruction advances up to 32 streams.  What makes that fit: no lookup tables.  Huffman codes are canonical
// (RFC 1951 3.2.2), so a code of length L is found by comparing the next 15 bits, taken MSB-first, with fifteen
// left-justified limits held in REGISTERS (branch-free: L = 1 + number of limits <= peek), and the symbol is then
// perm[base[L] + (peek >> (15 - L))] with perm = the symbols sorted by (length, value) -- 868 bytes of shared memory per
// stream instead of 3.4 KB, 256 streams per SM.  Length / distance extra-bit bases are arithmetic.  Output bytes go
// straight to global memory; LZ77 copies read back what the same thread wrote (same-thread program order).  The block's
// CRC-32 is checked afterwards by kd_crc32 (a warp per block, slices combined in GF(2)), which also reads the data coalesced.
// Same contract as the other two inflate kernels: a block is either inflated and verified or declined (status != 0), and a
// declined block gets the one-stream-per-warp kernel and finally the library's zlib.
#pragma once

constexpr uint32_t T1_THREADS = 96;   // per CTA; five CTAs per SM (452 B of tables per thread + 1 KB reserved per CTA): 15 warps

struct T1Stream {           // per-thread tables; 113 words: an odd stride keeps the 32 lanes of a warp on 32 different banks
  uint8_t perm_lit_lo[288];  // literal/length symbols sorted by (code length, symbol): low 8 bits ...
  uint32_t perm_lit_hi[9];   // ... and bit 8 (symbol >= 256: end-of-block / length codes), one bit per entry
  int16_t base_lit[16];      // index of the first symbol of length L in perm minus the first code of length L
  int16_t base_dst[16];
  uint16_t tmp[16];          // counts / fill cursors while a table is built
  uint8_t perm_dst[32];      // distance symbols (and, while a dynamic header is read, the code-length code's symbols)
};
static_assert(sizeof(T1Stream) == 452, "T1Stream layout");
constexpr uint32_t T1_SMEM_BYTES = T1_THREADS * sizeof(T1Stream);
constexpr uint32_t T1_LENS_BYTES = 160;  // code lengths of the deflate block being set up, 4 bits each: global scratch per BGZF
                                         // block (InflateArgs::scratch), so they cost no shared memory

struct T1Reader {  // LSB-first bit reader over global memory; two aligned words are always in flight ahead of the buffer
  const uint32_t* wp;  // the word after w1
  uint32_t w0, w1;     // the next two words of the stream
  uint64_t buf;
  uint32_t cnt;
  __device__ __forceinline__ void init(const uint8_t* p) {
    const uintptr_t a = (uintptr_t)p;
    wp = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
    const uint32_t skip = (uint32_t)(a & 3) * 8;
    buf = (uint64_t)(__ldcg(wp++) >> skip);  // L2 only: the copy engine may still be writing neighbouring blocks
    cnt = 32 - skip;
    w0 = __ldcg(wp++);
    w1 = __ldcg(wp++);
    refill();
  }
  __device__ __forceinline__ void refill() {  // afterwards cnt >= 33
    const bool take = cnt <= 32;
    if (take) {
      buf |= (uint64_t)w0 << cnt;
      cnt += 32;
      w0 = w1;
    }
#ifdef __CUDA_ARCH__
    // the new word is loaded IN PLACE into w1 under a predicate: written as `if (take) w1 = load` the compiler loads into a
    // temporary and moves it at once, which waits for the load and defeats the prefetch (ncu: 10 % of the stall samples)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.u32 p, %2, 0;\n"
        "@p ld.global.cg.u32 %0, [%1];\n"
        "}\n"
        : "+r"(w1)
        : "l"(wp), "r"((uint32_t)take)
        : "memory");
#else
    if (take) w1 = __ldcg(wp);
#endif
    if (take) ++wp;
  }
  __device__ __forceinline__ void consume(uint32_t n) {
    buf >>= n;
    cnt -= n;
  }
  __device__ __forceinline__ uint32_t bits(uint32_t n) const { return (uint32_t)buf & ((1u << n) - 1); }
  __device__ __forceinline__ uint32_t peek15() const { return __brev((uint32_t)buf) >> 17; }  // next 15 bits, first bit on top
  // first byte boundary at or after the read position (w0's word starts at wp - 2; cnt unread bits precede it)
  __device__ __forceinline__ const uint8_t* byte_pos_ceil() const { return reinterpret_cast<const uint8_t*>(wp - 2) - (cnt >> 3); }
};

// Length of the code at the top of `p` (15 bits, MSB first): 1 + the number of limits <= p.  16 = not a code of this table.
__device__ __forceinline__ uint32_t t1_code_len(uint32_t p, const uint32_t (&lim)[15]) {
  uint32_t L = 1;
#pragma unroll
  for (int k = 0; k < 15; ++k) L += p >= lim[k] ? 1u : 0u;
  return L;
}

// Canonical Huffman table from n code lengths (`len_of(s)`, 0 = unused): perm (through `put(index, symbol)`), base[1..15]
// and the fifteen limits.
// Returns false for an over-subscribed set.
template <class LenOf, class Put>
__device__ __forceinline__ bool t1_build(LenOf len_of, uint32_t n, Put put, int16_t* base, uint16_t* tmp, uint32_t (&lim)[15]) {
#pragma unroll
  for (int L = 0; L < 16; ++L) tmp[L] = 0;
  for (uint32_t s = 0; s < n; ++s) tmp[len_of(s)] += 1;
  uint32_t code = 0, off = 0, prev = 0;  // prev = number of codes one bit shorter (length 0 does not count)
  int left = 1;
  bool ok = true;
#pragma unroll
  for (int L = 1; L <= 15; ++L) {
    const uint32_t c = tmp[L];
    code = (code + prev) << 1;  // first code of length L
    left = left * 2 - (int)c;
    if (left < 0) {
      ok = false;
      left = 0;
    }
    lim[L - 1] = (code + c) << (15 - L);  // == first code of length L + 1, left-justified: non-decreasing in L
    base[L] = (int16_t)((int)off - (int)code);
    tmp[L] = (uint16_t)off;  // fill cursor: index of the first symbol of length L
    off += c;
    prev = c;
  }
  for (uint32_t s = 0; s < n; ++s) {
    const uint32_t l = len_of(s);
    if (l) put((uint32_t)tmp[l]++, s);
  }
  return ok;
}

constexpr unsigned long long T1_WAIT_NS = 2000000000ull;  // bounded wait for a window, wall clock
#ifndef T1_HOST_TEST
__device__ __forceinline__ unsigned long long t1_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void t1_lane_busy(volatile uint32_t* w, int d) { atomicAdd(const_cast<uint32_t*>(w), (uint32_t)d); }
#else
static inline unsigned long long t1_now_ns() { return 0; }
static inline void t1_lane_busy(volatile uint32_t* w, int d) { *w += (uint32_t)d; }
static inline void __syncwarp() {}
#endif
__global__ void __launch_bounds__(T1_THREADS, 5) kd_inflate_t1(const InflateArgs a) {
  extern __shared__ __align__(16) uint8_t t1_smem[];
  T1Stream& S = reinterpret_cast<T1Stream*>(t1_smem)[threadIdx.x];
  uint32_t lit_lim[15], dst_lim[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) lit_lim[k] = dst_lim[k] = 0;
  T1Reader br;
  br.wp = nullptr;
  br.w0 = br.w1 = 0;
  br.buf = 0;
  br.cnt = 0;

  // The last short match of a thread stays PENDING: its source bytes are requested into registers and stored only when the
  // next match (or the end of the pass) needs them done, so the DRAM / L2 latency of the LZ77 history read -- the dominant
  // stall of this kernel, the live history of all streams is far larger than L2 -- overlaps the decoding of the next symbols.
  uint32_t pm_len = 0;
  uint8_t* pm_dp = nullptr;
  uint8_t pm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto flush_pending = [&]() {
    if (pm_len) {
#pragma unroll
      for (uint32_t k = 0; k < 8; ++k)
        if (k < pm_len) pm_dp[k] = pm[k];
      pm_len = 0;
    }
  };
  enum : uint32_t { IDLE, WAIT, HDR, SYM, FIN };
  uint32_t state = IDLE;
  uint32_t b = 0, n_out = 0, op = 0, bfinal = 0, spins = 0, skip = 0;
  unsigned long long wait_t0 = 0;
  // Lanes of one warp are in different states.  A lane whose window has not arrived must not hold up the lanes that are
  // decoding (every trip round this loop is one symbol for them), so it sleeps only while NO lane of its warp decodes
  // (t1_busy counts those) and otherwise just looks at the flag again some iterations later.
  __shared__ uint32_t t1_busy[T1_THREADS / 32];
  volatile uint32_t* const my_busy = t1_busy + (threadIdx.x >> 5);
  if ((threadIdx.x & 31) == 0) *my_busy = 0;
  __syncwarp();
  bool counted = false;
  const uint8_t* in_end = nullptr;
  uint8_t* out = nullptr;

  // A warp's lanes are in different states most of the time, so a block takes the longer the more lanes of its warp hold one.
  // With fewer blocks than the grid has lanes, only the first lane_limit lanes of every warp work: the blocks spread over all
  // the warps instead of filling the first ones.
  if (a.lane_limit && (threadIdx.x & 31) >= a.lane_limit) return;
  for (;;) {
    // ------------------------------------------------------------------ a new block
    if (state == IDLE) {
      const uint32_t tk = atomicAdd(a.ticket, 1u);
      if (tk >= a.b1 - a.b0) return;
      b = a.block_list ? a.block_list[tk] : a.b0 + tk;
      spins = 0;
      skip = 0;
      wait_t0 = 0;
      state = WAIT;
    }
    if (state == WAIT && skip) {
      --skip;
    } else if (state == WAIT) {
      bool arrived = true;
      if (a.ready) arrived = *(const volatile uint32_t*)(a.ready + a.block_window[b]) != 0;
      if (arrived) {
        if (a.ready) __threadfence_system();  // the flag was written by the copy engine after the window's bytes
        n_out = a.isize[b];
        const uint8_t* in = a.comp + a.coff[b];
        in_end = in + a.clen[b];
        out = a.out + a.uoff[b];
        op = 0;
        if (n_out == 0) {
          a.status[b] = 0;
          state = IDLE;
        } else {
          br.init(in);
          state = HDR;
          t1_lane_busy(my_busy, 1);
          counted = true;
        }
      } else {
        const unsigned long long now = t1_now_ns();
        if (wait_t0 == 0) wait_t0 = now;
        if (now - wait_t0 > T1_WAIT_NS) {  // the window never came (copy failure, a tool serialising the streams)
          a.status[b] = 31u;
          atomicAdd(a.fail_count, 1u);
          state = IDLE;
        } else if (*my_busy == 0) {  // the whole warp waits: back off, 0.25 .. 4 us, to keep the polls off the L2
          __nanosleep(256u << (spins < 4u ? spins : 4u));
          ++spins;
        } else {
          skip = 512;  // other lanes are decoding: no sleeping, look again 512 symbols later
        }
      }
    }
    uint32_t st = 0;  // the check that declined the block, 0 = fine
    // ------------------------------------------------------------------ a deflate block header
    if (state == HDR) {
      if (br.byte_pos_ceil() > in_end) st = 1;
      br.refill();
      bfinal = br.bits(1);
      const uint32_t btype = ((uint32_t)br.buf >> 1) & 3;
      br.consume(3);
      if (st == 0 && btype == 3) st = 4;
      if (st == 0 && btype == 0) {  // stored
        br.consume(br.cnt & 7);
        br.refill();
        const uint32_t len = (uint32_t)br.buf & 0xffff, nlen = ((uint32_t)br.buf >> 16) & 0xffff;
        br.consume(32);
        const uint8_t* src = br.byte_pos_ceil();
        if ((len ^ nlen) != 0xffff) st = 2;
        else if (src + len > in_end || op + len > n_out) st = 3;
        else {
          for (uint32_t i = 0; i < len; ++i) out[op + i] = __ldcg(src + i);
          op += len;
          br.init(src + len);
          // stays in HDR for the next block, or finishes below
        }
        if (st == 0 && bfinal) state = FIN;  // finished: verdict below
      } else if (st == 0) {
        uint8_t* const l4 = a.scratch + (size_t)b * T1_LENS_BYTES;  // this BGZF block's code-length scratch
        uint32_t hlit = 288, hdist = 32;
        if (btype == 1) {  // fixed code lengths (RFC 1951 3.2.6)
          for (uint32_t i = 0; i < 160; ++i) {
            const uint32_t s0 = 2 * i, s1 = 2 * i + 1;
            auto fl = [](uint32_t s) -> uint32_t { return s < 144 ? 8u : s < 256 ? 9u : s < 280 ? 7u : s < 288 ? 8u : 5u; };
            l4[i] = (uint8_t)(fl(s0) | (fl(s1) << 4));
          }
        } else {  // dynamic: HLIT, HDIST, HCLEN, the code-length code, then the run-length coded lengths
          br.refill();
          hlit = br.bits(5) + 257;
          hdist = (((uint32_t)br.buf >> 5) & 31) + 1;
          const uint32_t hclen = (((uint32_t)br.buf >> 10) & 15) + 4;
          br.consume(14);
          if (hlit > 286 || hdist > 30) st = 5;
          if (st == 0) {
            // code-length code: 19 lengths of 3 bits, kept in the last 10 bytes of the scratch while its table is built
            for (uint32_t i = 0; i < 10; ++i) l4[150 + i] = 0;
            for (uint32_t i = 0; i < hclen; ++i) {
              br.refill();
              const uint32_t sym = c_clen_order[i], v = br.bits(3);
              br.consume(3);
              l4[150 + (sym >> 1)] |= (uint8_t)(v << ((sym & 1) * 4));
            }
            uint8_t* pd = S.perm_dst;
            const bool okc = t1_build([l4](uint32_t s) -> uint32_t { return (l4[150 + (s >> 1)] >> ((s & 1) * 4)) & 15u; }, 19u,
                                      [pd](uint32_t i, uint32_t s) { pd[i] = (uint8_t)s; }, S.base_dst, S.tmp, dst_lim);
            if (!okc) st = 6;
          }
          if (st == 0) {
            const uint32_t total = hlit + hdist;
            uint32_t n = 0, prev = 0;
            auto put = [&](uint32_t i, uint32_t v) {
              const uint32_t sh = (i & 1) * 4;
              l4[i >> 1] = (uint8_t)((l4[i >> 1] & ~(15u << sh)) | (v << sh));
            };
            while (n < total && st == 0) {
              br.refill();
              const uint32_t p = br.peek15();
              const uint32_t L = t1_code_len(p, dst_lim);
              if (L > 7) {
                st = 7;
                break;
              }
              const uint32_t sym = S.perm_dst[(int)S.base_dst[L] + (int)(p >> (15 - L))];
              br.consume(L);
              if (sym < 16) {
                put(n, sym);
                prev = sym;
                ++n;
              } else {
                uint32_t rep, val = 0;
                if (sym == 16) {
                  if (n == 0) {
                    st = 8;
                    break;
                  }
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
                if (n + rep > total) {
                  st = 9;
                  break;
                }
                for (uint32_t i = 0; i < rep; ++i) put(n + i, val);
                prev = val;
                n += rep;
              }
            }
            if (st == 0 && ((l4[128] & 15u) == 0)) st = 10;  // no end-of-block code (symbol 256)
          }
        }
        if (st == 0) {
          const uint32_t hl = hlit;
          uint8_t* pd = S.perm_dst;
          uint8_t* plo = S.perm_lit_lo;
          uint32_t* phi = S.perm_lit_hi;
#pragma unroll
          for (int k = 0; k < 9; ++k) phi[k] = 0;
          const bool okd = t1_build([l4, hl](uint32_t s) -> uint32_t { const uint32_t i = hl + s; return (l4[i >> 1] >> ((i & 1) * 4)) & 15u; }, hdist,
                                    [pd](uint32_t i, uint32_t s) { pd[i] = (uint8_t)s; }, S.base_dst, S.tmp, dst_lim);
          const bool okl = t1_build([l4](uint32_t s) -> uint32_t { return (l4[s >> 1] >> ((s & 1) * 4)) & 15u; }, hlit,
                                    [plo, phi](uint32_t i, uint32_t s) {
                                      plo[i] = (uint8_t)s;
                                      if (s & 256u) phi[i >> 5] |= 1u << (i & 31);
                                    },
                                    S.base_lit, S.tmp, lit_lim);
          if (!okd) st = 11;
          else if (!okl) st = 12;
          else state = SYM;
        }
      }
    }
    // ------------------------------------------------------------------ symbols (a few per pass, so that lanes stay together)
    if (state == SYM && st == 0) {
      // a corrupt stream must not run away: at most 16 symbols (< 100 bytes) are read between two looks at the input bound
      if (br.byte_pos_ceil() > in_end + 8) st = 21;
#pragma unroll 1
      for (int pass = 0; pass < 16 && st == 0; ++pass) {
        br.refill();
        uint32_t p = br.peek15();
        uint32_t L = t1_code_len(p, lit_lim);
        if (L > 15) {
          st = 13;
          break;
        }
        const uint32_t li = (uint32_t)((int)S.base_lit[L] + (int)(p >> (15 - L)));
        const uint32_t sym = (uint32_t)S.perm_lit_lo[li] | (((S.perm_lit_hi[li >> 5] >> (li & 31)) & 1u) << 8);
        br.consume(L);
        if (sym < 256) {
          if (op >= n_out) {
            st = 14;
            break;
          }
          out[op++] = (uint8_t)sym;
          continue;
        }
        if (sym == 256) {  // end of block
          state = bfinal ? FIN : HDR;
          break;
        }
        const uint32_t c = sym - 257;
        if (c > 28) {
          st = 15;
          break;
        }
        uint32_t len, xl = 0;
        if (c < 8) len = 3 + c;
        else if (c == 28) len = 258;
        else {
          xl = (c >> 2) - 1;
          len = 3 + ((4 + (c & 3)) << xl);
        }
        len += br.bits(xl);
        br.consume(xl);
        br.refill();
        p = br.peek15();
        L = t1_code_len(p, dst_lim);
        if (L > 15) {
          st = 16;
          break;
        }
        const uint32_t d = S.perm_dst[(int)S.base_dst[L] + (int)(p >> (15 - L))];
        br.consume(L);
        if (d > 29) {
          st = 17;
          break;
        }
        uint32_t dist, xd = 0;
        if (d < 4) dist = 1 + d;
        else {
          xd = (d >> 1) - 1;
          dist = 1 + ((2 + (d & 1)) << xd);
        }
        dist += br.bits(xd);
        br.consume(xd);
        if (dist > op || op + len > n_out) {
          st = 18;
          break;
        }
        uint8_t* dp = out + op;
        const uint8_t* sp = dp - dist;
        flush_pending();  // this match may read what the pending one writes
        if (len <= 8 && dist >= len) {  // the common case: request the bytes, store them later
#pragma unroll
          for (uint32_t k = 0; k < 8; ++k)
            if (k < len) pm[k] = sp[k];
          pm_len = len;
          pm_dp = dp;
        } else if (dist >= len) {  // source and destination do not overlap: eight loads in flight, then eight stores
          for (uint32_t i = 0; i < len; i += 8) {
            uint8_t t8[8];
#pragma unroll
            for (uint32_t k = 0; k < 8; ++k)
              if (i + k < len) t8[k] = sp[i + k];
#pragma unroll
            for (uint32_t k = 0; k < 8; ++k)
              if (i + k < len) dp[i + k] = t8[k];
          }
        } else {
          for (uint32_t i = 0; i < len; ++i) dp[i] = sp[i];  // byte by byte: an overlapping copy replicates its own output
        }
        op += len;
      }
      flush_pending();
    }
    // ------------------------------------------------------------------ verdicts
    if (state == FIN && st == 0) {  // last deflate block done
      if (op != n_out) st = 19;
      else if (br.byte_pos_ceil() > in_end) st = 20;
      if (st == 0) {
        a.status[b] = 0;  // kd_crc32 has the last word
        state = IDLE;
      }
    }
    if (st != 0) {
      a.status[b] = st;
      atomicAdd(a.fail_count, 1u);
      state = IDLE;
    }
    if (state == IDLE && counted) {
      t1_lane_busy(my_busy, -1);
      counted = false;
    }
  }
}

#ifndef T1_HOST_TEST
// CRC-32 of every block a first pass inflated (status 0), one warp per block, against the BGZF footer as htslib does
// (bgzf.c); a mismatch declines the block (status 30).
__global__ void __launch_bounds__(256) kd_crc32(const InflateArgs a) {
  __shared__ uint32_t crcT[1024];
  {
    uint32_t c = threadIdx.x;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
    crcT[threadIdx.x] = c;
  }
  __syncthreads();
  {
    uint32_t c = crcT[threadIdx.x];
    for (int k = 1; k < 4; ++k) {
      c = crcT[c & 0xff] ^ (c >> 8);
      crcT[k * 256 + threadIdx.x] = c;
    }
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warps = gridDim.x * 8;
  for (uint32_t i = blockIdx.x * 8 + (threadIdx.x >> 5); i < a.b1 - a.b0; i += warps) {
    const uint32_t b = a.block_list ? a.block_list[i] : a.b0 + i;
    const uint32_t n = a.isize[b];
    if (n == 0 || a.status[b] != 0) continue;
    const uint8_t* f = a.comp + a.coff[b] + a.clen[b];
    const uint32_t want = (uint32_t)__ldcg(f) | ((uint32_t)__ldcg(f + 1) << 8) | ((uint32_t)__ldcg(f + 2) << 16) | ((uint32_t)__ldcg(f + 3) << 24);
    const uint32_t got = warp_crc32(a.out + a.uoff[b], n, crcT, lane);
    if (got != want && lane == 0) {
      a.status[b] = 30u;
      atomicAdd(a.fail_count, 1u);
    }
  }
}
#endif
