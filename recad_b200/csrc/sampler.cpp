// Host-side bit-exact replay of the reference samplers' consumption of numpy's legacy global
// MT19937 stream (reference: recad/dataset/implicit.py:18-35 shuffle, 50-74 pairwise_sample,
// 77-91 pointwise_sample; seeded by recad/__init__.py:11-14).
//
// numpy rule restated (numpy 2.3 RandomState.randint / choice / shuffle -> masked rejection on
// 32-bit words): for a closed range [0, r]: r == 0 consumes nothing; otherwise mask = smallest
// 2^k - 1 >= r and words are drawn until (word & mask) <= r.
#include <stdint.h>
#include <string.h>

#include <stdio.h>
#include <stdlib.h>
#include <sys/mman.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/recad_b200.h"

namespace recad { void set_error(const char* fmt, ...); }

namespace {

static inline void cpu_relax() {        // spin-wait hint
#if defined(__x86_64__) || defined(__i386__)
  __builtin_ia32_pause();
#elif defined(__aarch64__)
  asm volatile("yield" ::: "memory");
#endif
}

// numpy's legacy generator, state-compatible (key[624] + pos).  The 624 outputs of a twist are tempered in one
// vectorisable pass into `buf`, so that next() -- called 2-3 times per sample by the sequential stream parsers --
// is a load and an increment.
#if defined(__x86_64__) && defined(__GNUC__)
#define RECAD_CLONES __attribute__((target_clones("avx512f", "avx2", "default")))
#else
#define RECAD_CLONES
#endif

RECAD_CLONES
static void mt_refill(uint32_t* __restrict__ key, uint32_t* __restrict__ buf) {
  constexpr int N = 624, M = 397;
  constexpr uint32_t UP = 0x80000000u, LOW = 0x7fffffffu, MAG = 0x9908b0dfu;
  // key[k + 1] is read before any lane overwrites it and key[k + M] / key[k + M - N] are at least 227 apart
#pragma GCC ivdep
  for (int k = 0; k < N - M; ++k) {
    const uint32_t y = (key[k] & UP) | (key[k + 1] & LOW);
    key[k] = key[k + M] ^ (y >> 1) ^ ((0u - (y & 1u)) & MAG);
  }
#pragma GCC ivdep
  for (int k = N - M; k < N - 1; ++k) {
    const uint32_t y = (key[k] & UP) | (key[k + 1] & LOW);
    key[k] = key[k + (M - N)] ^ (y >> 1) ^ ((0u - (y & 1u)) & MAG);
  }
  const uint32_t y = (key[N - 1] & UP) | (key[0] & LOW);
  key[N - 1] = key[M - 1] ^ (y >> 1) ^ ((0u - (y & 1u)) & MAG);
  for (int k = 0; k < N; ++k) {
    uint32_t t = key[k];
    t ^= t >> 11;
    t ^= (t << 7) & 0x9d2c5680u;
    t ^= (t << 15) & 0xefc60000u;
    t ^= t >> 18;
    buf[k] = t;
  }
}

RECAD_CLONES
static void mt_temper_only(const uint32_t* __restrict__ key, uint32_t* __restrict__ buf) {
  for (int k = 0; k < 624; ++k) {
    uint32_t t = key[k];
    t ^= t >> 11;
    t ^= (t << 7) & 0x9d2c5680u;
    t ^= (t << 15) & 0xefc60000u;
    t ^= t >> 18;
    buf[k] = t;
  }
}

struct MT {
  uint32_t* key;
  int pos;
  alignas(64) uint32_t buf[624];
  MT(uint32_t* k, int p) : key(k), pos(p) { mt_temper_only(key, buf); }   // outputs pos..623 of the current block
  inline uint32_t next() {
    if (__builtin_expect(pos >= 624, 0)) { mt_refill(key, buf); pos = 0; }
    return buf[pos++];
  }
  // the draws of a Fisher-Yates pass over one power-of-two band: j[i] = random_interval(i) for i = hi, hi-1, .., lo
  // (all share `mask`): every output is stored at the cursor and the cursor moves down only if it is accepted -- no
  // branch on the (random) acceptance
  void fill_band_desc(uint32_t* j, int64_t hi, int64_t lo, uint32_t mask) {
    int64_t i = hi;
    while (i >= lo) {
      if (pos >= 624) { mt_refill(key, buf); pos = 0; }
      int p = pos;
      const int stop = (int)std::min<int64_t>(624, p + (i - lo + 1));
      for (; p < stop; ++p) {
        const uint32_t v = buf[p] & mask;
        j[i] = v;
        i -= (int64_t)v <= i;
      }
      pos = p;
    }
  }
  static inline uint32_t mask_of(uint64_t r) {
    uint64_t mask = r;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    return (uint32_t)mask;
  }
  inline uint64_t masked(uint64_t r) {
    if (r == 0) return 0;
    return masked_with((uint32_t)r, mask_of(r));
  }
  // rejection loop with the first TWO candidates examined without a branch between them: the loop exit of the
  // plain do/while is mispredicted on every rejection (20-50 % of the draws), this form only when both fail
  inline uint32_t masked_with(uint32_t r, uint32_t mask) {
    if (__builtin_expect(pos + 2 <= 624, 1)) {
      const uint32_t v0 = buf[pos] & mask, v1 = buf[pos + 1] & mask;
      const bool ok0 = v0 <= r, ok1 = v1 <= r;
      if (__builtin_expect(ok0 | ok1, 1)) {
        pos += ok0 ? 1 : 2;
        return ok0 ? v0 : v1;
      }
      pos += 2;
    }
    uint32_t v;
    do { v = next() & mask; } while (v > r);
    return v;
  }
};

// growable host scratch, huge-page advised, never zero-filled
template <typename T>
struct Scratch {
  T* p = nullptr;
  int64_t cap = 0;
  T* get(int64_t n) {
    if (n > cap) {
      free(p);
      cap = std::max<int64_t>(n, 1);
      const size_t bytes = (((size_t)cap * sizeof(T)) + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
      void* q = nullptr;
      if (posix_memalign(&q, (size_t)2 << 20, bytes) != 0) { p = nullptr; cap = 0; return nullptr; }
      madvise(q, bytes, MADV_HUGEPAGE);
      p = static_cast<T*>(q);
    }
    return p;
  }
  // no destructor on purpose: the instances are function-local statics, and a daemon prefetch thread may still be
  // inside a sampler call when the process exits (static destructors would pull the memory from under it)
};

// the draws of np.random.shuffle(arange(n)): j[i] = random_interval(i) for i = n-1 .. 1, one power-of-two band at a time
static void shuffle_draws(MT& mt, int64_t n, uint32_t* j_out) {
  for (int64_t i = n - 1; i > 0;) {
    const uint32_t mask = MT::mask_of((uint64_t)i);
    const int64_t band_lo = std::max<int64_t>((int64_t)(mask >> 1) + 1, 1);        // every i in [band_lo, i] has this mask
    mt.fill_band_desc(j_out, i, band_lo, mask);
    i = band_lo - 1;
  }
  if (n > 0) j_out[0] = 0;
}


// Iteration order of the CPython set built by inserting, in ascending order, every item of [0, n_items) that is not
// in the sorted list sp[0..n) (duplicates allowed in sp) into an empty set -- what `set(range(n_items)) - set(iids)`
// returns when it does not take the copy-and-discard path.  hash(int) == int for these values.
static void cpython_set_order(const int64_t* sp, int64_t n, int64_t n_items, std::vector<int64_t>& order) {
  constexpr int kLinearProbes = 9, kPerturbShift = 5;
  std::vector<int64_t> table(8, -1), old;
  size_t mask = 7, fill = 0;
  auto insert_clean = [&](std::vector<int64_t>& t, size_t m, int64_t key) {
    size_t perturb = (size_t)key, i = (size_t)key & m;
    for (;;) {
      if (t[i] < 0) { t[i] = key; return; }
      if (i + kLinearProbes <= m) {
        for (int j = 1; j <= kLinearProbes; ++j)
          if (t[i + (size_t)j] < 0) { t[i + (size_t)j] = key; return; }
      }
      perturb >>= kPerturbShift;
      i = (i * 5 + 1 + perturb) & m;
    }
  };
  int64_t q = 0;
  for (int64_t item = 0; item < n_items; ++item) {
    while (q < n && sp[q] < item) ++q;
    if (q < n && sp[q] == item) continue;
    insert_clean(table, mask, item);          // no dummies, no equal keys: set_add_entry probes exactly like set_insert_clean
    ++fill;
    if (fill * 5 >= mask * 3) {
      const size_t minused = fill > 50000 ? fill * 2 : fill * 4;
      size_t newsize = 8;
      while (newsize <= minused) newsize <<= 1;
      old.swap(table);
      table.assign(newsize, -1);
      mask = newsize - 1;
      for (int64_t key : old)
        if (key >= 0) insert_clean(table, mask, key);
    }
  }
  order.clear();
  for (int64_t key : table)
    if (key >= 0) order.push_back(key);
}

}  // namespace

extern "C" {

int recad_mt19937_pairwise(uint32_t* key, int32_t* pos, int64_t n_users, int64_t n_items, int64_t train_size,
                           const int64_t* allpos_rowptr, const int32_t* allpos_col, int64_t* out, int64_t* n_out) {
  if (!key || !pos || !allpos_rowptr || !out || !n_out || n_users <= 0 || n_items <= 0 || train_size < 0 ||
      n_users > 0xffffffffLL || n_items > 0xffffffffLL) {
    recad::set_error("mt19937_pairwise: bad argument");
    return RECAD_ERR_ARG;
  }
  MT mt(key, *pos);
  // np.random.randint(0, n_users, train_size): ONE vector call, all users drawn first (implicit.py:57)
  int64_t* users = new int64_t[train_size > 0 ? train_size : 1];
  for (int64_t k = 0; k < train_size; ++k) users[k] = (int64_t)mt.masked((uint64_t)n_users - 1);
  int64_t w = 0;
  // The users are known up front, so the two dependent random accesses per sample (row pointer,
  // then the row's items) are software-prefetched: the loop is otherwise DRAM-latency bound.
  constexpr int64_t kAheadPtr = 24, kAheadRow = 12;
  for (int64_t k = 0; k < train_size; ++k) {
    if (k + kAheadPtr < train_size) __builtin_prefetch(allpos_rowptr + users[k + kAheadPtr]);
    if (k + kAheadRow < train_size) {
      const int64_t u1 = users[k + kAheadRow];
      const int64_t a = allpos_rowptr[u1], b = allpos_rowptr[u1 + 1];
      for (int64_t q = a; q < b && q < a + 192; q += 16) __builtin_prefetch(allpos_col + q);
      if (b > a + 192) __builtin_prefetch(allpos_col + (a + b) / 2);
    }
    const int64_t u = users[k];
    const int64_t lo = allpos_rowptr[u], hi = allpos_rowptr[u + 1];
    if (hi == lo) continue;  // implicit.py:63-64
    if (hi - lo >= n_items) {
      delete[] users;
      recad::set_error("mt19937_pairwise: user %lld interacted with every item; negative sampling cannot terminate",
                       (long long)u);
      return RECAD_ERR_ARG;
    }
    const int64_t p = allpos_col[lo + (int64_t)mt.masked((uint64_t)(hi - lo) - 1)];
    int64_t neg;
    do { neg = (int64_t)mt.masked((uint64_t)n_items - 1); } while (std::binary_search(allpos_col + lo, allpos_col + hi, (int32_t)neg));
    out[3 * w] = u; out[3 * w + 1] = p; out[3 * w + 2] = neg;
    ++w;
  }
  delete[] users;
  *n_out = w;
  *pos = mt.pos;
  return RECAD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Per-user membership filter of the large-epoch sampler (recad_mt19937_pairwise_soa).  Checking a negative
// candidate touches ONE OR TWO cache lines of a 1024-bit filter (no false negatives; a "maybe" falls back to the
// exact binary search of the user's sorted list, a "no" accepts the negative without ever reading the list).
// ---------------------------------------------------------------------------------------------------------
// Two 64-byte lines per user, of which a sample normally touches only the FIRST:
//   line 0: word 0 = first entry of the user's row | row length << 40, words 1..7 = 448 filter bits (region A)
//   line 1: 512 filter bits (region B)
// Users with at most kLight positives keep all three probes of an item in region A.  For heavier users probe 1
// is in region A and probes 2, 3 in region B, so a negative candidate whose first probe misses (80-90 % of them)
// is accepted from line 0 alone.  The parse is bound by the cache misses it can keep in flight (about ten line-fill
// buffers per core), hence everything a sample needs -- row bounds and the decisive filter bits -- sits in one line.
constexpr int kFilterWords = 16;
constexpr uint32_t kBitsA = 448;             // region A; region B is the 512 bits that follow (9-bit probes, below)
constexpr int64_t kLight = 32;
static inline uint32_t probe_a(uint32_t item) { return 64u + (uint32_t)(((uint64_t)(item * 0x9E3779B1u) * kBitsA) >> 32); }
static inline void probes_bc(uint32_t item, bool light, uint32_t& b, uint32_t& c) {
  const uint32_t hb = item * 0x85EBCA77u, hc = item * 0xC2B2AE3Du;
  if (light) {
    b = 64u + (uint32_t)(((uint64_t)hb * kBitsA) >> 32);
    c = 64u + (uint32_t)(((uint64_t)hc * kBitsA) >> 32);
  } else {
    b = 512u + (hb >> 23);      // 9 bits: region B
    c = 512u + (hc >> 23);
  }
}

static void parallel_for(int64_t n, int n_threads, const std::function<void(int64_t, int64_t)>& fn) {
  n_threads = (int)std::max<int64_t>(1, std::min<int64_t>(n_threads, (n + 65535) / 65536));
  if (n_threads == 1) { fn(0, n); return; }
  std::vector<std::thread> th;
  const int64_t per = (n + n_threads - 1) / n_threads;
  for (int t = 0; t < n_threads; ++t) {
    const int64_t lo = t * per, hi = std::min(n, lo + per);
    if (lo < hi) th.emplace_back(fn, lo, hi);
  }
  for (auto& t : th) t.join();
}

// Ask for transparent huge pages on a freshly allocated (not yet touched) host buffer: the samplers' random
// accesses into 10^8-byte arrays otherwise pay a TLB miss each.  Best effort (no-op where THP is off).
int recad_host_advise_huge(void* ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) return RECAD_OK;
  const uintptr_t a = ((uintptr_t)ptr + 4095) & ~(uintptr_t)4095;
  const uintptr_t e = ((uintptr_t)ptr + (uintptr_t)bytes) & ~(uintptr_t)4095;
  if (e > a) madvise(reinterpret_cast<void*>(a), e - a, MADV_HUGEPAGE);
  return RECAD_OK;
}

// second level for heavy users (more than kHeavy positives, where the 1024-bit block saturates): 32 bits per
// positive, three probes, stored at the user's own offset of a [nnz] uint32 array => ~0.1 % false positives
constexpr int64_t kHeavy = 96;
static inline uint64_t ext_probe(uint32_t item, int j, uint64_t nbits) {
  const uint32_t h = (item + 0x7F4A7C15u * (uint32_t)(j + 1)) * (j == 0 ? 0xC2B2AE35u : (j == 1 ? 0x27D4EB2Fu : 0x165667B1u));
  return ((uint64_t)h * nbits) >> 32;
}

// users [u_lo, n_users) only: the blocks of the other users are left as they are (an injected dataset copies its parent's
// blocks -- appended fake users do not move anybody's row -- and builds only the new ones)
int recad_pairwise_filter_build_range(const int64_t* allpos_rowptr, const int32_t* allpos_col, int64_t u_lo, int64_t n_users,
                                      uint64_t* filter, uint32_t* ext, int32_t n_threads) {
  if (!allpos_rowptr || !filter || !ext || n_users <= 0 || u_lo < 0 || u_lo > n_users) {
    recad::set_error("pairwise_filter_build: bad argument");
    return RECAD_ERR_ARG;
  }
  if (allpos_rowptr[n_users] >= ((int64_t)1 << 40)) {
    recad::set_error("pairwise_filter_build: more than 2^40 interactions");
    return RECAD_ERR_UNSUPPORTED;
  }
  for (int64_t u = u_lo; u < n_users; ++u)
    if (allpos_rowptr[u + 1] - allpos_rowptr[u] >= ((int64_t)1 << 24)) {
      recad::set_error("pairwise_filter_build: user %lld has 2^24 or more interactions", (long long)u);
      return RECAD_ERR_UNSUPPORTED;
    }
  parallel_for(n_users - u_lo, n_threads, [&](int64_t lo, int64_t hi) {
    for (int64_t u = u_lo + lo; u < u_lo + hi; ++u) {
      uint64_t* f = filter + u * kFilterWords;
      for (int q = 0; q < kFilterWords; ++q) f[q] = 0;
      const int64_t a0 = allpos_rowptr[u], a1 = allpos_rowptr[u + 1];
      f[0] = (uint64_t)a0 | ((uint64_t)(a1 - a0) << 40);
      const bool light = a1 - a0 <= kLight;
      for (int64_t e = a0; e < a1; ++e) {
        const uint32_t item = (uint32_t)allpos_col[e], a = probe_a(item);
        uint32_t b, c;
        probes_bc(item, light, b, c);
        f[a >> 6] |= 1ull << (a & 63);
        f[b >> 6] |= 1ull << (b & 63);
        f[c >> 6] |= 1ull << (c & 63);
      }
      for (int64_t e = a0; e < a1; ++e) ext[e] = 0;
      if (a1 - a0 > kHeavy) {
        const uint64_t nbits = (uint64_t)(a1 - a0) * 32;
        for (int64_t e = a0; e < a1; ++e)
          for (int j = 0; j < 3; ++j) {
            const uint64_t p = ext_probe((uint32_t)allpos_col[e], j, nbits);
            ext[a0 + (p >> 5)] |= 1u << (p & 31);
          }
      }
    }
  });
  return RECAD_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Large-epoch sampler (recad_mt19937_pairwise_soa).  Same samples, same stream consumption as
// recad_mt19937_pairwise (implicit.py:50-74) + the shuffle draws (implicit.py:24-25).  The stream parse is inherently
// sequential (every draw's position depends on all earlier rejections), so everything else is moved off it:
//   * a PRODUCER thread generates the MT19937 output stream into a ring -- the stream does not depend on the parse,
//     so rewinding the parser is just resetting an index (no generator checkpoints), and the parser never runs a twist;
//   * the users are drawn first (implicit.py:57); while they are drawn, helper threads already gather every sample's
//     row LENGTH from a 4-byte-per-user table, so the sequential parser only streams sequential arrays;
//   * the parser draws optimistically (first candidate the mask accepts) block by block; the helpers check block b's
//     candidates against the per-user filter lines while the parser draws block b + 1; a candidate that IS a positive
//     makes the parser redo that sample exactly and redraw ONLY until the new trajectory meets the old one again
//     (same sample, same stream offset: typically a few samples later), bounded by the two blocks in flight;
//   * outputs are three 32-bit arrays (user, index of the positive inside the user's row, negative): the positive
//     ITEM is looked up on the device (recad_samples_expand), where the CSR already lives.
// ---------------------------------------------------------------------------------------------------------
namespace {

struct StreamRing {
  static constexpr uint64_t kWords = (uint64_t)1 << 21;        // 8 MB of outputs in flight
  static constexpr uint64_t kMask = kWords - 1;
  static constexpr int kPad = 64;                              // mirror of the first words behind the end: windows never wrap
  static constexpr int64_t kSnapEvery = 1024;                  // generator snapshots, in twists
  uint32_t* buf = nullptr;
  alignas(64) std::atomic<uint64_t> head{0};                   // outputs produced
  alignas(64) std::atomic<uint64_t> tail{0};                   // lowest output the consumer may still read
  std::atomic<bool> stop{false};
  uint32_t key[624];
  int pos0 = 0;
  std::vector<uint32_t> snaps;                                 // key after s * kSnapEvery twists
  std::thread th;

  bool start(const uint32_t* key_in, int pos_in) {
    void* q = nullptr;
    if (posix_memalign(&q, 4096, (kWords + kPad) * sizeof(uint32_t)) != 0) return false;
    buf = static_cast<uint32_t*>(q);
    memcpy(key, key_in, sizeof(key));
    pos0 = pos_in;
    snaps.assign(key, key + 624);
    th = std::thread([this]() { run(); });
    return true;
  }
  void put(const uint32_t* src, int n) {                       // append n outputs at head (the caller checked the room)
    if (n <= 0 || n > 624) return;
    const uint64_t h = head.load(std::memory_order_relaxed);
    uint64_t i = h & kMask;
    const uint64_t first = std::min<uint64_t>((uint64_t)n, kWords - i);
    memcpy(buf + i, src, first * 4);
    const uint64_t rest = (uint64_t)n - first;
    if (rest > 0 && rest <= 624) memcpy(buf, src + first, rest * 4);
    // mirror: ring words [0, kPad) also live at [kWords, kWords + kPad)
    if (i < (uint64_t)kPad) {
      const uint64_t m = std::min<uint64_t>((uint64_t)n, (uint64_t)kPad - i);
      memcpy(buf + kWords + i, src, m * 4);
    }
    if (rest > 0 && rest <= 624) memcpy(buf + kWords, src + first, std::min<uint64_t>(rest, (uint64_t)kPad) * 4);
    head.store(h + (uint64_t)n, std::memory_order_release);
  }
  void run() {
    alignas(64) uint32_t out[624];
    mt_temper_only(key, out);
    if (pos0 < 624) put(out + pos0, 624 - pos0);
    int64_t twists = 0;
    for (;;) {
      int spins = 0;
      while (head.load(std::memory_order_relaxed) + 624 + kPad > tail.load(std::memory_order_acquire) + kWords) {
        if (stop.load(std::memory_order_relaxed)) return;
        if (++spins > 256) { std::this_thread::yield(); spins = 0; } else { cpu_relax(); }
      }
      if (stop.load(std::memory_order_relaxed)) return;
      mt_refill(key, out);
      ++twists;
      if (twists % kSnapEvery == 0) snaps.insert(snaps.end(), key, key + 624);
      put(out, 624);
    }
  }
  // generator state after `consumed` outputs, in numpy's convention (pos in [0, 624])
  void finish(uint64_t consumed, uint32_t* key_out, int32_t* pos_out) {
    stop.store(true, std::memory_order_relaxed);
    th.join();
    const uint64_t q = (uint64_t)pos0 + consumed;
    int64_t twists = q <= 624 ? 0 : (int64_t)((q - 1) / 624);
    const int64_t s = twists / kSnapEvery;
    memcpy(key_out, snaps.data() + (size_t)s * 624, 624 * sizeof(uint32_t));
    alignas(64) uint32_t scratch[624];
    for (int64_t k = s * kSnapEvery; k < twists; ++k) mt_refill(key_out, scratch);
    *pos_out = (int32_t)(q - (uint64_t)twists * 624);
    free(buf);
    buf = nullptr;
  }
};

// consumer view of the ring
struct StreamReader {
  StreamRing& r;
  uint64_t t = 0;            // next output to consume
  uint64_t avail = 0;        // cached head
  explicit StreamReader(StreamRing& ring) : r(ring) {}
  inline const uint32_t* at(uint64_t i) const { return r.buf + (i & StreamRing::kMask); }
  inline void need(uint64_t n) {                     // outputs [t, t + n) produced?  (n <= kPad for window reads)
    if (__builtin_expect(t + n <= avail, 1)) return;
    for (;;) {
      avail = r.head.load(std::memory_order_acquire);
      if (t + n <= avail) return;
      cpu_relax();
    }
  }
  inline void release(uint64_t upto) { r.tail.store(upto, std::memory_order_release); }
  inline uint32_t masked(uint32_t rr, uint32_t mask) {          // random_interval(rr), rr > 0
    for (;;) {
      need(1);
      const uint32_t v = *at(t++) & mask;
      if (v <= rr) return v;
    }
  }
};

}  // namespace

// sampler_avx512.cpp (built with -mavx512f; entered only when the CPU has it)
uint64_t recad_shuffle_draws_avx512(const uint32_t* src, uint64_t n_words, uint32_t mask, int64_t* i_io, int64_t band_lo,
                                    uint32_t* j_out);
int64_t recad_parse_window_avx512(const uint32_t* ring, uint64_t ring_mask, uint64_t* t_io, uint64_t avail, const uint32_t* lens,
                                  int64_t k0, int64_t k1, uint32_t* rel, uint32_t* negs, uint32_t* tst, int64_t tst_mask,
                                  uint32_t neg_r, uint32_t neg_mask, uint32_t n_items);

int recad_mt19937_pairwise_soa(uint32_t* key, int32_t* pos, int64_t n_users, int64_t n_items, int64_t train_size,
                               const int64_t* allpos_rowptr, const int32_t* allpos_col, const uint64_t* filter,
                               const uint32_t* ext, int32_t n_threads, uint32_t* users, uint32_t* rel, uint32_t* negs,
                               int64_t* n_out, uint32_t* j_out) {
  if (!key || !pos || !allpos_rowptr || !filter || !ext || !users || !rel || !negs || !n_out || n_users <= 0 || n_items <= 0 ||
      train_size < 0 || n_users > 0x7fffffffLL || n_items > 0x7fffffffLL || train_size > 0x7fffffffLL || *pos < 0 || *pos > 624) {
    recad::set_error("mt19937_pairwise_soa: bad argument");
    return RECAD_ERR_ARG;
  }
#if defined(__x86_64__) && defined(__GNUC__)
  const bool use_avx512 = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("bmi") && n_items > 1 &&
                          !(getenv("RECAD_SAMPLER_SCALAR") && atoi(getenv("RECAD_SAMPLER_SCALAR")));
#else
  const bool use_avx512 = false;
#endif
  const bool trace = getenv("RECAD_SAMPLER_TRACE") != nullptr;
  auto t0 = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[sampler2] %s %.3f s\n", what, std::chrono::duration<double>(t1 - t0).count());
    t0 = t1;
  };
  static std::mutex scratch_mutex;                           // one epoch of a stream at a time (they are chained anyway)
  static Scratch<uint32_t> len_buf, deg_buf;
  std::lock_guard<std::mutex> scratch_lock(scratch_mutex);
  uint32_t* len32 = len_buf.get(train_size);
  uint32_t* deg = deg_buf.get(n_users);
  if (!len32 || !deg) {
    recad::set_error("mt19937_pairwise_soa: out of host memory");
    return RECAD_ERR_ARG;
  }
  StreamRing ring;
  if (!ring.start(key, *pos)) {
    recad::set_error("mt19937_pairwise_soa: out of host memory");
    return RECAD_ERR_ARG;
  }
  StreamReader rd(ring);
  auto fail = [&](int rc) { ring.finish(0, key, pos); return rc; };   // leaves key / pos as they were
  // row lengths (4 MB at 10^6 users: cache resident for the gather below); the producer fills the ring meanwhile
  for (int64_t u = 0; u < n_users; ++u) deg[u] = (uint32_t)(allpos_rowptr[u + 1] - allpos_rowptr[u]);
  // ---- helper pool: first the length gather (chunks of the user array as they are drawn), then the block checks
  const int n_help = getenv("RECAD_SAMPLER_HELPERS") ? std::max(1, atoi(getenv("RECAD_SAMPLER_HELPERS")))
                                                     : (int)std::max(1, std::min(n_threads - 4, 8));   // parser, producer, swap thread, caller
  constexpr int64_t kChunk = 1 << 15;
  const int64_t n_chunks = (train_size + kChunk - 1) / kChunk;
  std::atomic<int64_t> users_ready{0};            // users [0, users_ready) are drawn
  std::atomic<int64_t> next_chunk{0}, chunks_done{0};
  std::vector<std::atomic<uint8_t>> chunk_done((size_t)std::max<int64_t>(n_chunks, 1));
  for (auto& c : chunk_done) c.store(0, std::memory_order_relaxed);
  constexpr int64_t kBlock = 512;               // power of two: the offsets ring below is indexed with a mask
  constexpr int64_t kAhead = 16;
  constexpr uint32_t kDropped = 0xffffffffu;
  constexpr int64_t kNoFail = INT64_MAX;
  const uint32_t neg_r = (uint32_t)(n_items - 1), neg_mask = MT::mask_of(neg_r);
  auto is_positive = [&](const uint64_t* f, int64_t lo, int64_t len, uint32_t neg) -> bool {
    const uint32_t a = probe_a(neg);
    if (!((f[a >> 6] >> (a & 63)) & 1ull)) return false;
    uint32_t b, c;
    probes_bc(neg, len <= kLight, b, c);
    if (!((f[b >> 6] >> (b & 63)) & (f[c >> 6] >> (c & 63)) & 1ull)) return false;
    if (len > kHeavy) {
      const uint64_t nbits = (uint64_t)len * 32;
      const uint64_t p0 = ext_probe(neg, 0, nbits), p1 = ext_probe(neg, 1, nbits), p2 = ext_probe(neg, 2, nbits);
      if (!((ext[lo + (p0 >> 5)] >> (p0 & 31)) & (ext[lo + (p1 >> 5)] >> (p1 & 31)) & (ext[lo + (p2 >> 5)] >> (p2 & 31)) & 1u))
        return false;
    }
    return std::binary_search(allpos_col + lo, allpos_col + lo + len, (int32_t)neg);
  };
  auto check = [&](int64_t a0, int64_t a1) -> int64_t {     // first sample of [a0, a1) whose candidate is a positive
    for (int64_t k = a0; k < std::min(a1, a0 + kAhead); ++k) __builtin_prefetch(filter + (int64_t)users[k] * kFilterWords);
    for (int64_t k = a0; k < a1; ++k) {
      if (k + kAhead < a1) __builtin_prefetch(filter + (int64_t)users[k + kAhead] * kFilterWords);
      if (rel[k] == kDropped) continue;
      const uint64_t* f = filter + (int64_t)users[k] * kFilterWords;
      if (__builtin_expect(is_positive(f, (int64_t)(f[0] & (((uint64_t)1 << 40) - 1)), (int64_t)(f[0] >> 40), negs[k]), 0)) return k;
    }
    return kNoFail;
  };
  struct alignas(64) Slot { std::atomic<int64_t> fail; };
  std::vector<Slot> slots((size_t)n_help + 1);
  std::atomic<int64_t> go{0}, done{0};
  std::atomic<bool> quit{false};
  int64_t job_lo = 0, job_hi = 0;
  std::vector<std::thread> helpers;
  for (int t = 1; t <= n_help; ++t)
    helpers.emplace_back([&, t]() {
      // phase 1: lengths
      for (;;) {
        const int64_t c = next_chunk.load(std::memory_order_relaxed);
        if (c >= n_chunks) break;
        const int64_t hi = std::min(train_size, (c + 1) * kChunk);
        if (users_ready.load(std::memory_order_acquire) < hi) {
          if (quit.load(std::memory_order_relaxed)) return;
          cpu_relax();
          continue;
        }
        int64_t mine = c;
        if (!next_chunk.compare_exchange_strong(mine, c + 1, std::memory_order_relaxed)) continue;
        for (int64_t k = c * kChunk; k < hi; ++k) len32[k] = deg[users[k]];
        chunk_done[(size_t)c].store(1, std::memory_order_release);
        chunks_done.fetch_add(1, std::memory_order_release);
      }
      // phase 2: checks
      int64_t seen = 0;
      for (;;) {
        int spins = 0;
        while (go.load(std::memory_order_acquire) == seen) {
          if (quit.load(std::memory_order_relaxed)) return;
          if (++spins > 4000) { std::this_thread::yield(); spins = 0; } else { cpu_relax(); }
        }
        ++seen;
        const int64_t n = job_hi - job_lo, per = (n + n_help - 1) / n_help;
        const int64_t a0 = std::min(job_hi, job_lo + (t - 1) * per), a1 = std::min(job_hi, a0 + per);
        slots[(size_t)t].fail.store(check(a0, a1), std::memory_order_relaxed);
        done.fetch_add(1, std::memory_order_release);
      }
    });
  auto stop_helpers = [&]() {
    quit.store(true, std::memory_order_relaxed);
    for (auto& h : helpers) h.join();
  };
  // ---- users: np.random.randint(0, n_users, train_size), one vector call (implicit.py:57); branch-free cursor
  {
    const uint32_t r = (uint32_t)(n_users - 1), mask = MT::mask_of(r);
    if (r == 0) {
      memset(users, 0, (size_t)train_size * sizeof(uint32_t));
      users_ready.store(train_size, std::memory_order_release);
    } else {
      int64_t k = 0, published = 0;
      while (k < train_size) {
        rd.need(1);
        uint64_t span = std::min<uint64_t>(rd.avail - rd.t, (uint64_t)(train_size - k));
        span = std::min<uint64_t>(span, StreamRing::kWords - (rd.t & StreamRing::kMask));      // contiguous part
        const uint32_t* src = rd.at(rd.t);
        for (uint64_t q = 0; q < span; ++q) {
          const uint32_t v = src[q] & mask;
          users[k] = v;
          k += v <= r;
        }
        rd.t += span;
        rd.release(rd.t);
        if (k - published >= kChunk || k == train_size) {
          users_ready.store(k, std::memory_order_release);
          published = k;
        }
      }
    }
  }
  lap("draw users");
  while (chunks_done.load(std::memory_order_acquire) < n_chunks) cpu_relax();
  lap("wait for the length gather");
  // ---- parse
  std::vector<uint32_t> tst_v((size_t)4 * kBlock);            // stream offset in front of each sample (ring of 4 blocks)
  uint32_t* tst = tst_v.data();
  constexpr int64_t kTstMask = 4 * kBlock - 1;
  int rc = RECAD_OK;
  // optimistic draw of samples [k0, k1): position of the positive, first candidate the mask accepts.  The stream
  // cursor and every pointer live in locals: the loop-carried chain is cursor -> 4 loads -> compares -> selects -> cursor
  auto draw = [&](int64_t k0, int64_t k1) -> int {
    uint64_t t = rd.t, avail = rd.avail;
    const uint32_t* __restrict__ ringbuf = ring.buf;
    const uint32_t* __restrict__ lens = len32;
    uint32_t* __restrict__ rel_ = rel;
    uint32_t* __restrict__ negs_ = negs;
    uint32_t* __restrict__ tst_ = tst;
    const uint32_t nr = neg_r, nm = neg_mask;
    const int64_t tmask = kTstMask;
    int rc_ = RECAD_OK;
    int64_t k = k0;
    while (k < k1) {
      if (use_avx512 && k1 - k >= 8) {
        // 64-word windows of the stream, acceptance masks by vector compares, the chain is shift / tzcnt / add
        if (t + 64 > avail) {
          rd.t = t;
          rd.need(64);
          avail = rd.avail;
        }
        k = recad_parse_window_avx512(ringbuf, StreamRing::kMask, &t, avail, lens, k, k1, rel_, negs_, tst_, tmask, nr, nm,
                                      (uint32_t)std::min<int64_t>(n_items, 0xffffffffLL));
        if (k >= k1) break;
        // sample k is extraordinary (or the stream ran dry): the exact scalar code below takes it
      }
      tst_[k & tmask] = (uint32_t)t;
      const uint32_t len = lens[k];
      if (__builtin_expect(len == 0, 0)) { rel_[k] = kDropped; ++k; continue; }               // implicit.py:63-64
      if (__builtin_expect((int64_t)len >= n_items, 0)) {
        recad::set_error("mt19937_pairwise_soa: user %lld interacted with every item; negative sampling cannot terminate",
                         (long long)users[k]);
        rc_ = RECAD_ERR_ARG;
        break;
      }
      const uint32_t r1 = len - 1, m1 = r1 ? 0xffffffffu >> __builtin_clz(r1) : 0u;
      if (__builtin_expect(t + 4 > avail, 0)) {
        rd.t = t;
        rd.need(4);
        avail = rd.avail;
      }
      const uint32_t* w = ringbuf + (t & StreamRing::kMask);
      const uint32_t o0 = w[0], o1 = w[1], o2 = w[2], o3 = w[3];
      const uint32_t a0 = o0 & m1, a1 = o1 & m1;
      const bool none = r1 == 0, okA0 = a0 <= r1, okA1 = a1 <= r1;
      const int cA = none ? 0 : (okA0 ? 1 : 2);
      const uint32_t x0 = cA == 0 ? o0 : (cA == 1 ? o1 : o2), x1 = cA == 0 ? o1 : (cA == 1 ? o2 : o3);
      const uint32_t b0 = x0 & nm, b1 = x1 & nm;
      const bool okB0 = b0 <= nr, okB1 = b1 <= nr;
      if (__builtin_expect((none | okA0 | okA1) & (okB0 | okB1) & (nr != 0), 1)) {
        rel_[k] = none ? 0u : (okA0 ? a0 : a1);
        negs_[k] = okB0 ? b0 : b1;
        t += (uint64_t)(cA + (okB0 ? 1 : 2));
        ++k;
        continue;
      }
      rd.t = t;
      rel_[k] = r1 ? rd.masked(r1, m1) : 0u;
      negs_[k] = nr ? rd.masked(nr, nm) : 0u;
      t = rd.t;
      avail = rd.avail;
      ++k;
    }
    rd.t = t;
    return rc_;
  };
  int64_t inline_result = kNoFail;
  bool pool_busy = false;
  auto start_check = [&](int64_t lo_, int64_t hi_) {
    if (hi_ - lo_ < 64) { inline_result = check(lo_, hi_); pool_busy = false; return; }
    job_lo = lo_; job_hi = hi_;
    done.store(0, std::memory_order_relaxed);
    go.fetch_add(1, std::memory_order_release);
    pool_busy = true;
  };
  int64_t wait_spins = 0;
  auto finish_check = [&]() -> int64_t {
    if (!pool_busy) return inline_result;
    while (done.load(std::memory_order_acquire) < n_help) { cpu_relax(); ++wait_spins; }
    int64_t first = kNoFail;
    for (int t = 1; t <= n_help; ++t) first = std::min(first, slots[(size_t)t].fail.load(std::memory_order_relaxed));
    pool_busy = false;
    return first;
  };
  int64_t n_fix = 0, n_redrawn = 0, n_dropped = 0;
  rc = draw(0, std::min(train_size, kBlock));
  for (int64_t b0 = 0; b0 < train_size && rc == RECAD_OK; b0 += kBlock) {
    // invariant: [b0, b1) is drawn and rd.t is the offset behind it
    const int64_t b1 = std::min(train_size, b0 + kBlock), n1 = std::min(train_size, b1 + kBlock);
    rd.release(rd.t - (uint64_t)(uint32_t)((uint32_t)rd.t - tst[b0 & kTstMask]));   // block b may still be rewound into
    start_check(b0, b1);
    if (b1 < train_size && (rc = draw(b1, n1))) { finish_check(); break; }      // speculative, under the check of block b
    int64_t k = finish_check();
    while (k != kNoFail) {
      // sample k's candidate is one of its user's positives: redo it exactly from its own offset, then redraw what
      // follows until the new trajectory meets the old one (same sample, same offset) or the drawn region ends
      const uint64_t t_end_old = rd.t;
      rd.t = rd.t - (uint64_t)(uint32_t)((uint32_t)rd.t - tst[k & kTstMask]);
      {
        const int64_t u = users[k];
        const int64_t lo = allpos_rowptr[u], len = allpos_rowptr[u + 1] - lo;
        const uint64_t* f = filter + u * kFilterWords;
        const uint32_t r1 = (uint32_t)(len - 1), m1 = r1 ? 0xffffffffu >> __builtin_clz(r1) : 0u;
        rel[k] = r1 ? rd.masked(r1, m1) : 0u;
        uint32_t neg;
        do { neg = neg_r ? rd.masked(neg_r, neg_mask) : 0u; } while (is_positive(f, lo, len, neg));
        negs[k] = neg;
      }
      ++n_fix;
      int64_t j = k + 1;
      bool met = false;
      for (; j < n1; ++j) {
        if ((uint32_t)rd.t == tst[j & kTstMask]) { met = true; break; }
        if ((rc = draw(j, j + 1))) break;
        ++n_redrawn;
      }
      if (rc) break;
      if (met) rd.t = t_end_old;
      if (k + 1 < b1) {
        start_check(k + 1, b1);
        k = finish_check();
      } else {
        k = kNoFail;
      }
    }
  }
  stop_helpers();
  if (rc) return fail(rc);
  if (trace) fprintf(stderr, "[sampler2] %lld exact redos, %lld samples redrawn, %d helper threads, %lld wait spins\n", (long long)n_fix,
                     (long long)n_redrawn, n_help, (long long)wait_spins);
  lap("parse stream");
  // users without positives are dropped (implicit.py:63-64): compact in place (rare)
  int64_t w = train_size;
  for (int64_t k = 0; k < train_size; ++k) n_dropped += rel[k] == kDropped;
  if (n_dropped) {
    w = 0;
    for (int64_t k = 0; k < train_size; ++k) {
      if (rel[k] == kDropped) continue;
      users[w] = users[k]; rel[w] = rel[k]; negs[w] = negs[k];
      ++w;
    }
    lap("drop users without positives");
  }
  if (j_out) {
    // the draws of np.random.shuffle(arange(w)): j[i] = random_interval(i) for i = w-1 .. 1, band by band
    for (int64_t i = w - 1; i > 0;) {
      const uint32_t mask = MT::mask_of((uint64_t)i);
      const int64_t band_lo = std::max<int64_t>((int64_t)(mask >> 1) + 1, 1);
      while (i >= band_lo) {
        rd.need(1);
        uint64_t span = std::min<uint64_t>(rd.avail - rd.t, (uint64_t)(i - band_lo + 1));
        span = std::min<uint64_t>(span, StreamRing::kWords - (rd.t & StreamRing::kMask));
        const uint32_t* src = rd.at(rd.t);
        const uint64_t q0 = use_avx512 ? recad_shuffle_draws_avx512(src, span, mask, &i, band_lo, j_out) : 0;
        for (uint64_t q = q0; q < span; ++q) {
          const uint32_t v = src[q] & mask;
          j_out[i] = v;
          i -= (int64_t)v <= i;
        }
        rd.t += span;
        rd.release(rd.t);
      }
    }
    if (w > 0) j_out[0] = 0;
    lap("shuffle draws");
  }
  *n_out = w;
  ring.finish(rd.t, key, pos);
  return RECAD_OK;
}

// perm = arange(n) with swap(perm[i], perm[j[i]]) for i = n-1 .. 1, 32-bit (n < 2^31)
int recad_permutation_apply32(int64_t n, const uint32_t* j, int32_t* perm) {
  if (!j || !perm || n < 0 || n > 0x7fffffffLL) {
    recad::set_error("permutation_apply32: bad argument");
    return RECAD_ERR_ARG;
  }
  const auto t0 = std::chrono::steady_clock::now();
  for (int64_t i = 0; i < n; ++i) perm[i] = (int32_t)i;
  constexpr int64_t kAhead = 64;
  for (int64_t i = n - 1; i > 0; --i) {
    if (i > kAhead) __builtin_prefetch(perm + j[i - kAhead], 1);
    std::swap(perm[i], perm[j[i]]);
  }
  if (getenv("RECAD_SAMPLER_TRACE"))
    fprintf(stderr, "[sampler2] shuffle swaps %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  return RECAD_OK;
}

int recad_mt19937_pointwise(uint32_t* key, int32_t* pos, int64_t n_dict_users, const int64_t* user_ids,
                            const int64_t* pos_rowptr, const int64_t* pos_items, const int64_t* pos_sorted,
                            int64_t n_items, int32_t ratio, int64_t* out) {
  if (!key || !pos || !user_ids || !pos_rowptr || !out || n_items <= 0 || ratio < 0 || n_dict_users < 0) {
    recad::set_error("mt19937_pointwise: bad argument");
    return RECAD_ERR_ARG;
  }
  MT mt(key, *pos);
  int64_t w = 0;
  std::vector<int64_t> left_scratch;
  for (int64_t k = 0; k < n_dict_users; ++k) {
    const int64_t lo = pos_rowptr[k], hi = pos_rowptr[k + 1], n = hi - lo, uid = user_ids[k];
    for (int64_t j = lo; j < hi; ++j) { out[3 * w] = uid; out[3 * w + 1] = pos_items[j]; out[3 * w + 2] = 1; ++w; }
    const int64_t n_neg = n * ratio;
    if (n_neg == 0) continue;
    // distinct sorted positives of this user
    const int64_t* sp = pos_sorted + lo;
    int64_t n_distinct = 0;
    for (int64_t j = 0; j < n; ++j) if (j == 0 || sp[j] != sp[j - 1]) ++n_distinct;
    const int64_t n_left = n_items - n_distinct;
    if (n_left <= 0) {
      recad::set_error("mt19937_pointwise: user %lld has no negative item to draw", (long long)uid);
      return RECAD_ERR_ARG;
    }
    const uint32_t rr = (uint32_t)(n_left - 1), mask = MT::mask_of(rr);
    // `list(full_items - set(iids))` (implicit.py:86) is ascending only while CPython takes the copy-and-discard path
    // of set_difference, i.e. while len(full) / 4 > len(set(iids)).  For denser users the difference is BUILT by
    // inserting the surviving items, in ascending order, into a fresh hash table; when that table ends up smaller than
    // n_items the values wrap around it and the list order is the table's slot order (setobject.c, CPython 3.8-3.13:
    // LINEAR_PROBES 9, PERTURB_SHIFT 5, growth to 4 x used (2 x above 50000) when fill * 5 >= mask * 3).
    const bool table_order = !((n_items >> 2) > n_distinct);
    if (table_order) {
      cpython_set_order(sp, n, n_items, left_scratch);
      for (int64_t c = 0; c < n_neg; ++c) {
        const int64_t r = rr ? (int64_t)mt.masked_with(rr, mask) : 0;
        out[3 * w] = uid; out[3 * w + 1] = left_scratch[(size_t)r]; out[3 * w + 2] = 0; ++w;
      }
      continue;
    }
    for (int64_t c = 0; c < n_neg; ++c) {
      const int64_t r = rr ? (int64_t)mt.masked_with(rr, mask) : 0;
      // r-th element of the ascending complement: r + #{distinct positives p_j with p_j - j <= r}
      int64_t t = 0, j_distinct = 0;
      if (n_distinct == n) {
        // count of the non-decreasing sequence sp[j] - j that is <= r: binary search with selects instead of branches
        // (the outcome of every step is a coin flip)
        int64_t a = 0, len = n;
        while (len > 0) {
          const int64_t half = len >> 1, mid = a + half;
          const bool le = sp[mid] - mid <= r;
          a = le ? mid + 1 : a;
          len = le ? len - half - 1 : half;
        }
        t = a;
      } else {
        for (int64_t j = 0; j < n; ++j) {
          if (j > 0 && sp[j] == sp[j - 1]) continue;
          if (sp[j] - j_distinct <= r) ++t; else break;
          ++j_distinct;
        }
      }
      out[3 * w] = uid; out[3 * w + 1] = r + t; out[3 * w + 2] = 0; ++w;
    }
  }
  *pos = mt.pos;
  return RECAD_OK;
}

int recad_mt19937_permutation(uint32_t* key, int32_t* pos, int64_t n, int64_t* perm) {
  if (!key || !pos || !perm || n < 0 || n > 0xffffffffLL) {
    recad::set_error("mt19937_permutation: bad argument");
    return RECAD_ERR_ARG;
  }
  MT mt(key, *pos);
  for (int64_t i = 0; i < n; ++i) perm[i] = i;
  // j = random_interval(i) depends on i only, not on the data: draw kAhead swaps ahead (same stream
  // order) and prefetch perm[j], which is otherwise one DRAM miss per element
  constexpr int kAhead = 32;
  int64_t ring[kAhead];
  int64_t drawn = n - 1;  // next i whose j has not been drawn yet
  for (int q = 0; q < kAhead && drawn > 0; ++q, --drawn) {
    ring[(n - 1 - drawn) % kAhead] = (int64_t)mt.masked((uint64_t)drawn);
    __builtin_prefetch(perm + ring[(n - 1 - drawn) % kAhead], 1);
  }
  for (int64_t i = n - 1; i > 0; --i) {
    const int slot = (int)((n - 1 - i) % kAhead);
    const int64_t j = ring[slot];
    if (drawn > 0) {
      ring[slot] = (int64_t)mt.masked((uint64_t)drawn);
      __builtin_prefetch(perm + ring[slot], 1);
      --drawn;
    }
    std::swap(perm[i], perm[j]);
  }
  *pos = mt.pos;
  return RECAD_OK;
}

// The shuffle in two halves, so that the sequential stream can move on to the next epoch while another thread
// applies the swaps: draw = the data-independent part (j_i = random_interval(i) for i = n-1 .. 1, the ONLY part that
// consumes the stream), apply = the memory-bound part (perm = arange(n); swap(perm[i], perm[j_i]) in the same order).
int recad_mt19937_permutation_draw(uint32_t* key, int32_t* pos, int64_t n, uint32_t* j_out) {
  if (!key || !pos || !j_out || n < 0 || n > 0xffffffffLL) {
    recad::set_error("mt19937_permutation_draw: bad argument");
    return RECAD_ERR_ARG;
  }
  const auto t0 = std::chrono::steady_clock::now();
  MT mt(key, *pos);
  shuffle_draws(mt, n, j_out);
  *pos = mt.pos;
  if (getenv("RECAD_SAMPLER_TRACE"))
    fprintf(stderr, "[sampler] shuffle draws %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  return RECAD_OK;
}

int recad_permutation_apply(int64_t n, const uint32_t* j, int64_t* perm) {
  if (!j || !perm || n < 0) {
    recad::set_error("permutation_apply: bad argument");
    return RECAD_ERR_ARG;
  }
  const auto t0 = std::chrono::steady_clock::now();
  for (int64_t i = 0; i < n; ++i) perm[i] = i;
  constexpr int64_t kAhead = 48;
  for (int64_t i = n - 1; i > 0; --i) {
    if (i > kAhead) __builtin_prefetch(perm + j[i - kAhead], 1);
    std::swap(perm[i], perm[j[i]]);
  }
  if (getenv("RECAD_SAMPLER_TRACE"))
    fprintf(stderr, "[sampler] shuffle swaps %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  return RECAD_OK;
}

// The draws of one AUSH batch on the global generator, in the reference's order: per row F draws of
// random_interval(len - 1) indexing the row's candidate list (np.random.choice(a, size=F, replace=True) ==
// randint(0, len, F), aush.py:64-68), then the Fisher-Yates pass of np.random.shuffle over the batch's ZR pool (the
// (row, selected column) pairs with real == 0 in row-major order, aush.py:113-117); the first floor(P * (1 - ZR_ratio))
// pairs of the shuffled pool leave the mask.
int recad_mt19937_aush_batch(uint32_t* key, int32_t* pos, int64_t B, const int64_t* users, const int64_t* cand_ptr,
                             const int32_t* cand_items, const float* cand_vals, int32_t F, int32_t S, const uint8_t* zero_sel,
                             double zr_ratio, int32_t* cols_out, float* tval_out, float* zr_out) {
  if (!key || !pos || B < 0 || F < 0 || S < 0 || (B && (!users || !cand_ptr || !cand_items || !cols_out)) || (B && S && (!zero_sel || !zr_out))) {
    recad::set_error("mt19937_aush_batch: bad argument");
    return RECAD_ERR_ARG;
  }
  MT mt(key, *pos);
  for (int64_t b = 0; b < B; ++b) {
    const int64_t lo = cand_ptr[users[b]], len = cand_ptr[users[b] + 1] - lo;
    if (len <= 0) {
      recad::set_error("mt19937_aush_batch: user %lld has no filler candidate", (long long)users[b]);   // np.random.choice: 'a' cannot be empty
      return RECAD_ERR_ARG;
    }
    const uint32_t r = (uint32_t)(len - 1), mask = MT::mask_of(r);
    for (int f = 0; f < F; ++f) {
      const int64_t at = lo + (r ? mt.masked_with(r, mask) : 0u);
      const int32_t c = cand_items[at];
      cols_out[b * F + f] = c;
      if (tval_out && cand_vals) {            // input_template carries a rating once per distinct column: a repeat adds 0
        bool seen = false;
        for (int g = 0; g < f; ++g) seen |= cols_out[b * F + g] == c;
        tval_out[b * F + f] = seen ? 0.f : cand_vals[at];
      }
    }
  }
  std::vector<int64_t> pool;
  for (int64_t q = 0; q < B * S; ++q) {
    zr_out[q] = zero_sel[q] ? 1.f : 0.f;
    if (zero_sel[q]) pool.push_back(q);
  }
  const int64_t P = (int64_t)pool.size();
  for (int64_t i = P - 1; i > 0; --i) std::swap(pool[i], pool[(int64_t)mt.masked((uint64_t)i)]);
  const int64_t cut = (int64_t)std::floor((double)P * (1.0 - zr_ratio));
  for (int64_t q = 0; q < cut && q < P; ++q) zr_out[pool[q]] = 0.f;
  *pos = mt.pos;
  return RECAD_OK;
}

}  // extern "C"
