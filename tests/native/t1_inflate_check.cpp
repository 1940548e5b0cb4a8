// Host-side check of kd_inflate_t1's decoder logic (coverm_b200/csrc/cmb_decode_t1.cuh): the kernel body is compiled as
// plain C++ for ONE emulated thread (CUDA keywords and intrinsics shimmed below) and run over raw DEFLATE streams made by
// zlib at every level / strategy and several data shapes, plus corrupted streams (must be declined or caught by the
// length checks, never run away).  The GPU tests then only have to establish that the kernel behaves the same on the device.
#include <zlib.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <string>
#include <vector>
#include <algorithm>

#define __device__
#define __global__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __shared__
#define __align__(x)
#define T1_HOST_TEST 1
struct Dim3 { unsigned x = 0, y = 0, z = 0; };
static Dim3 threadIdx, blockIdx, gridDim;
static inline uint32_t __brev(uint32_t v) {
  v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
  v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
  v = ((v >> 4) & 0x0f0f0f0fu) | ((v & 0x0f0f0f0fu) << 4);
  v = ((v >> 8) & 0x00ff00ffu) | ((v & 0x00ff00ffu) << 8);
  return (v >> 16) | (v << 16);
}
template <class T> static inline T __ldcg(const T* p) { return *p; }
static inline uint32_t atomicAdd(uint32_t* p, uint32_t v) { uint32_t o = *p; *p += v; return o; }
static inline void __threadfence_system() {}
static inline void __nanosleep(unsigned) {}
using std::min;
static const uint8_t c_clen_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
struct InflateArgs {
  const uint8_t* comp; const uint64_t* coff; const uint32_t* clen; const uint32_t* isize; const uint64_t* uoff;
  uint32_t b0, b1; uint8_t* out; uint32_t* status; uint32_t* ticket; uint32_t* fail_count;
  const uint32_t* block_window; const uint32_t* ready; uint32_t lane_limit;
  const uint32_t* block_list; uint8_t* scratch;
};
uint8_t t1_smem[4096];
#include "cmb_decode_t1.cuh"

using namespace std;
static vector<uint8_t> deflate_raw(const vector<uint8_t>& in, int level, int strategy) {
  z_stream zs{};
  deflateInit2(&zs, level, Z_DEFLATED, -15, 8, strategy);
  vector<uint8_t> out(deflateBound(&zs, in.size()) + 64);
  zs.next_in = (Bytef*)in.data(); zs.avail_in = in.size(); zs.next_out = out.data(); zs.avail_out = out.size();
  deflate(&zs, Z_FINISH);
  out.resize(zs.total_out);
  deflateEnd(&zs);
  return out;
}

// Runs the kernel over `streams` (several blocks back to back in one buffer, like a BGZF file in device memory).
static void run(const vector<vector<uint8_t>>& comp, const vector<uint32_t>& isize, vector<vector<uint8_t>>& out, vector<uint32_t>& status) {
  vector<uint8_t> file(64, 0xEE);
  vector<uint64_t> coff, uoff;
  vector<uint32_t> clen;
  uint64_t u = 7;  // odd offsets on purpose
  for (size_t i = 0; i < comp.size(); ++i) {
    file.push_back(0xCD);  // misalign
    coff.push_back(file.size());
    clen.push_back((uint32_t)comp[i].size());
    file.insert(file.end(), comp[i].begin(), comp[i].end());
    file.insert(file.end(), 8, 0xAB);  // footer place holder
    uoff.push_back(u);
    u += isize[i] + 3;
  }
  file.resize(file.size() + 1024, 0);
  vector<uint8_t> inflated(u + 1024, 0x5A);
  status.assign(comp.size(), 99);
  uint32_t ticket = 0, fails = 0;
  InflateArgs a{};
  a.comp = file.data(); a.coff = coff.data(); a.clen = clen.data(); a.isize = isize.data(); a.uoff = uoff.data();
  a.b0 = 0; a.b1 = (uint32_t)comp.size(); a.out = inflated.data(); a.status = status.data(); a.ticket = &ticket; a.fail_count = &fails;
  vector<uint8_t> scratch(comp.size() * 160 + 16, 0x77);
  a.scratch = scratch.data();
  kd_inflate_t1(a);
  out.clear();
  for (size_t i = 0; i < comp.size(); ++i) {
    out.emplace_back(inflated.begin() + uoff[i], inflated.begin() + uoff[i] + isize[i]);
    // the bytes around each block's output must be untouched
    if (inflated[uoff[i] - 1] != 0x5A || inflated[uoff[i] + isize[i]] != 0x5A) status[i] |= 0x100;
  }
}

int main() {
  mt19937_64 rng(1);
  int fails = 0, n = 0, declined_bad = 0, n_bad = 0;
  vector<vector<uint8_t>> comp, want, got;
  vector<uint32_t> isz, status;
  for (int iter = 0; iter < 1500; ++iter) {
    size_t len = iter < 20 ? iter : rng() % 65281;
    vector<uint8_t> data(len);
    int kind = iter % 6;
    for (size_t i = 0; i < len; ++i) {
      switch (kind) {
        case 0: data[i] = rng(); break;
        case 1: data[i] = "ACGT"[rng() & 3]; break;
        case 2: data[i] = (i % 37) ^ (rng() % 100 == 0); break;
        case 3: data[i] = rng() % 8 ? 'A' : rng(); break;
        case 4: data[i] = i > 3 && rng() % 4 ? data[i - 1 - rng() % min<size_t>(i - 1, 5)] : rng(); break;
        case 5: { static const char* w = "the quick brown fox jumps over the lazy dog "; data[i] = w[(i + (rng() % 50 == 0)) % 44]; } break;
      }
    }
    int level = iter % 10;
    int strat = (iter / 10) % 4 == 3 ? Z_FIXED : (iter / 10) % 4 == 2 ? Z_HUFFMAN_ONLY : Z_DEFAULT_STRATEGY;
    comp.push_back(deflate_raw(data, level, strat));
    isz.push_back((uint32_t)len);
    want.push_back(data);
    if (comp.size() == 50 || iter == 1499) {
      run(comp, isz, got, status);
      for (size_t i = 0; i < comp.size(); ++i) {
        ++n;
        if (status[i] != 0 || got[i] != want[i]) {
          ++fails;
          if (fails < 10) printf("FAIL block %zu: status %u len %u\n", i, status[i], isz[i]);
        }
      }
      // corrupted copies: flip a bit / truncate / wrong isize; the decoder must stay inside its output and either decline or
      // produce SOMETHING of the right length (the CRC pass catches wrong bytes)
      vector<vector<uint8_t>> bad = comp;
      vector<uint32_t> bisz = isz;
      for (size_t i = 0; i < bad.size(); ++i) {
        if (bad[i].size() < 4) continue;
        switch (i % 3) {
          case 0: bad[i][rng() % bad[i].size()] ^= (uint8_t)(1u << (rng() % 8)); break;
          case 1: bad[i].resize(bad[i].size() / 2); break;
          case 2: bisz[i] = bisz[i] > 10 ? bisz[i] - 1 - (uint32_t)(rng() % 9) : bisz[i] + 1; break;
        }
      }
      run(bad, bisz, got, status);
      for (size_t i = 0; i < bad.size(); ++i) {
        if (bad[i].size() < 4) continue;
        ++n_bad;
        if (status[i] & 0x100) { ++fails; printf("FAIL corrupted block %zu wrote outside its output\n", i); }
        if (status[i] != 0 || got[i] != want[i]) ++declined_bad;
      }
      comp.clear(); isz.clear(); want.clear();
    }
  }
  printf("%d tests, %d fails; %d of %d corrupted streams declined or different\n", n, fails, declined_bad, n_bad);
  return fails ? 1 : 0;
}
