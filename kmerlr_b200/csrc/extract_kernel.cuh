// extract_kernel.cuh -- the extraction kernel (one warp per sequence) and its launcher, shared between
// extract.cu (host flow) and the extract_e*.cu translation units, each of which instantiates the kernel
// for ONE value of E (keys per lane of the register sort): the instantiations compile in parallel.
// See extract.cu for the design.
#pragma once

#include <type_traits>

#include "common.cuh"

namespace kl {
namespace xk {

#ifndef KL_X_OLDPOS
#define KL_X_OLDPOS 1     // 1: position pass with one funnel-shift load per position (lane = positions lane, lane + 32, ...);
                          // 0: a 64-bit window per 16 consecutive positions of a lane (no load / bit reversal per position:
                          // fewer instructions, yet 2.57 vs 2.54 ms at C2 and 6.31 vs 6.37 ms at a quarter of C3)
#endif
#ifndef KL_X_WALK
#define KL_X_WALK 1       // 1: bitmap levels emitted by a walk over the set bits; 0: a slot per position computed from
                          // prefix popcounts (measured slower: 2.90 vs 2.55 ms at C2 -- a numbering gather, three
                          // shared-memory reads and a scattered store per position cost more than the bit loops)
#endif
#ifndef KL_X_TKPRE
#define KL_X_TKPRE 0      // 1: the ticket of the next row group is drawn one group ahead (measured: the register it holds costs more than
                          // the round trip it hides -- 2.275 vs 2.251 ms at C2)
#endif
#ifndef KL_X_TLPIPE
#define KL_X_TLPIPE 1     // the class list of the table levels is read one iteration ahead
#endif
#ifndef KL_X_MARKSKIP
#define KL_X_MARKSKIP 1   // 1: the marks of observed classes stop once the device-wide bitmap covers the numbering set
#endif
constexpr uint32_t SENT = 0xFFFFFFFFu;    // sort key of a position without a valid k-mer (sorts last)
constexpr uint32_t NOKEY = 0xFFFFFFFEu;   // "no previous key" in front of the sorted array
constexpr int KT_MAX = 5;          // levels <= KT_MAX use direct count tables
constexpr int KB_MAX = 8;          // highest level that can use a per-row bitmap
constexpr int KB_DEFAULT = 7;      // ... level 8 does so only when the rows are too long for the register sort
constexpr int MAX_N = 13;          // 2*13 code bits + 4 length bits per position
constexpr int TAB_WORDS = 704;     // (4+16+64+256+1024)/2 = 682 packed u16 pairs, padded to whole rows of 32 (swizzle)
constexpr int OBS_MAX_LEVEL = 8;   // marks of observed classes of levels <= 8 are gathered per block in smem

struct XParams {
  int M, N, op, binarize;
  int t_lo, t_hi;                  // table levels (empty if t_lo > t_hi)
  int b_lo, b_hi;                  // bitmap levels (empty if b_lo > b_hi)
  int s_lo;                        // sorted levels [s_lo, N] (empty if s_lo > N)
  int mark;                        // mark observed classes in the bitmap
  uint32_t level_off[MAX_N + 2];   // dense id of (k, code 0), multiples of 32
  uint32_t bm_off[KB_MAX + 2];     // word offset of level k's bitmap inside the per-warp bitmap area
  uint32_t pf_off[KB_MAX + 2];     // word offset of level k's prefix array (one entry per 4 words)
  uint32_t tl_cnt;                 // classes of the table levels (flat list tl, in (k, code) order)
  int bm_words, pf_words, ts_words;// per-warp shared memory areas, in 32-bit words
  int warp_words;                  // total per-warp shared memory, in 32-bit words
  int obs_words;                   // per-block marks of observed classes: obs_id_words by class id (levels <= OBS_MAX_LEVEL),
  int obs_id_words;                // then one bit per entry of the table-level class list tl
  int64_t stride, n, row0, ovf_stride;   // the launch covers the rows [row0, n)
  const int64_t *len, *blk;
  const uint32_t *bits2;
  const uint16_t *inv16;
  const uint2 *tl;                 // x = byte offset of the code's 16-bit counter in the warp's table | that of its image << 16, y = class id
  uint32_t *st_id, *st_cnt, *rowcnt, *bitmap, *ovf;
  const uint2 *nbx;                // numbering set (all classes of the configuration, or the frozen list)
  int filter;                      // drop ids outside the numbering set
  unsigned long long *stats;       // [0] max_i sum_j v_ij^2, [1] max v_ij
  uint32_t *ticket;                // rows are handed out to the blocks in groups of one row per warp
  int64_t nb_words;                // words of the numbering set / of the bitmap of observed classes
  uint32_t *full;                  // set once every class of the numbering set has been observed: the marks stop
  // binarized rows, for the matrix-free logistic pass (see Implicit in common.cuh)
  uint32_t *lowbits;               // per row: bitmap over the classes of the table levels (nullptr: not wanted)
  int low_words;
  uint32_t *rowdup;                // per row: number of repeat events written at the tail of the row's slots
  int events;                      // record one event (the column) per repeat of a class of a level > KT_MAX
};

__device__ __forceinline__ uint32_t tab_off(int k) {  // sum_{j=1}^{k-1} 4^j
  return ((1u << (2 * k)) - 4u) / 3u;
}


// Index swizzle of the per-warp staging buffers: lanes that write runs of consecutive slots at a stride of
// ~16 (the sorted level: E keys per lane) would all hit two banks; XOR-ing the row number into the bank bits
// spreads them, and a read of 32 consecutive slots stays a permutation of one row (conflict free).
// (Measured: the bank conflicts drop -- ncu counted 1 031 of 1 631 shared-memory wavefronts per C2 row as excess
// before -- but the kernel is not bound by them: 2.60 ms with the swizzle, 2.58 ms without.  Off by default.)
#ifndef KL_X_NOSWZ
#define KL_X_NOSWZ 1
#endif
__host__ __device__ __forceinline__ uint32_t sw(uint32_t j) { return KL_X_NOSWZ ? j : j ^ ((j >> 5) & 31u); }
__host__ __device__ __forceinline__ int sw(int j) { return (int)sw((uint32_t)j); }

template <int E>
void launch_extract(const XParams &P);

#ifdef KL_EXTRACT_KERNEL_IMPL
// ---- bitonic sort of 32*E keys in registers, index = lane*E + r, ascending ----------------------
__device__ __forceinline__ void ce(uint32_t &a, uint32_t &b) {
  uint32_t lo = min(a, b), hi = max(a, b);
  a = lo; b = hi;
}

template <int E>
__device__ __forceinline__ void warp_sort(uint32_t (&K)[E], unsigned lane) {
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
    // first stage of the merge: partner = i ^ (k-1)
    if (k <= E) {
#pragma unroll
      for (int r = 0; r < E; r++) {
        int pr = r ^ (k - 1);
        if (pr > r) ce(K[r], K[pr]);
      }
    } else {
      const int lm = k / E - 1;                       // lane xor mask
      const bool keepmin = (lane & ((k / E) >> 1)) == 0;
#pragma unroll
      for (int r = 0; r < E / 2; r++) {
        uint32_t a = K[r], b = K[E - 1 - r];
        uint32_t va = __shfl_xor_sync(0xffffffffu, b, lm);   // partner's K[E-1-r]
        uint32_t vb = __shfl_xor_sync(0xffffffffu, a, lm);   // partner's K[r]
        K[r] = keepmin ? min(a, va) : max(a, va);
        K[E - 1 - r] = keepmin ? min(b, vb) : max(b, vb);
      }
    }
    // remaining half-cleaners
#pragma unroll
    for (int j = k / 4; j >= 1; j >>= 1) {
      if (j < E) {
#pragma unroll
        for (int r = 0; r < E; r++)
          if ((r & j) == 0) ce(K[r], K[r | j]);
      } else {
        const int lm = j / E;
        const bool keepmin = (lane & lm) == 0;
#pragma unroll
        for (int r = 0; r < E; r++) {
          uint32_t v = __shfl_xor_sync(0xffffffffu, K[r], lm);
          K[r] = keepmin ? min(K[r], v) : max(K[r], v);
        }
      }
    }
  }
}

// ---- the same network on 16-bit keys, two to a register (levels k <= PACK_MAX) -------------------
// P[q] holds the keys at sorted indices lane*E + q (low half) and lane*E + q + E/2 (high half).  Every
// stage at an in-lane distance below E/2, and every cross-lane half-cleaner, pairs low halves with low
// halves and high halves with high halves, so one __vminu2 / __vmaxu2 / shuffle serves two keys.  Only
// the stages that pair the two halves of a lane (distance E/2, and the flips of the in-lane merge of E
// keys and of the cross-lane merges) swap halves with a PRMT.  0xFFFF is the sentinel: under revcomp
// no canonical code of a level k <= 8 is 0xFFFF (TTTTTTTT canonicalises to AAAAAAAA).
constexpr int PACK_MAX = 8;
__device__ __forceinline__ uint32_t swap_halves(uint32_t x) { return __byte_perm(x, 0u, 0x1032); }
__device__ __forceinline__ void ce2(uint32_t &a, uint32_t &b) {
  uint32_t lo = __vminu2(a, b), hi = __vmaxu2(a, b);
  a = lo; b = hi;
}

template <int E>
__device__ __forceinline__ void warp_sort16(uint32_t (&P)[E / 2], unsigned lane) {
  constexpr int H = E / 2;
#pragma unroll
  for (int k = 2; k <= 32 * E; k <<= 1) {
    // first stage of the merge: partner = i ^ (k-1)
    if (k <= H) {
#pragma unroll
      for (int q = 0; q < H; q++) {
        int pq = q ^ (k - 1);
        if (pq > q) ce2(P[q], P[pq]);
      }
    } else if (k == E) {
      // index q pairs with E-1-q (the high half of P[H-1-q]), index q+H with H-1-q (its low half)
#pragma unroll
      for (int q = 0; 2 * q < H; q++) {
        const uint32_t b = swap_halves(P[H - 1 - q]);
        const uint32_t mn = __vminu2(P[q], b), mx = __vmaxu2(P[q], b);
        P[q] = __byte_perm(mn, mx, 0x7610);           // index q: min, index q+H: max
        P[H - 1 - q] = __byte_perm(mn, mx, 0x5432);   // index H-1-q: min, index E-1-q: max
      }
    } else {
      const int lm = k / E - 1;                       // lane xor mask
      const bool keepmin = (lane & ((k / E) >> 1)) == 0;
#pragma unroll
      for (int q = 0; 2 * q < H; q++) {
        uint32_t a = P[q], b = P[H - 1 - q];
        uint32_t va = swap_halves(__shfl_xor_sync(0xffffffffu, b, lm));   // partner's (K[E-1-q], K[H-1-q])
        uint32_t vb = swap_halves(__shfl_xor_sync(0xffffffffu, a, lm));   // partner's (K[H+q], K[q])
        P[q] = keepmin ? __vminu2(a, va) : __vmaxu2(a, va);
        P[H - 1 - q] = keepmin ? __vminu2(b, vb) : __vmaxu2(b, vb);
      }
    }
    // remaining half-cleaners
#pragma unroll
    for (int j = k / 4; j >= 1; j >>= 1) {
      if (j < H) {
#pragma unroll
        for (int q = 0; q < H; q++)
          if ((q & j) == 0) ce2(P[q], P[q | j]);
      } else if (j == H) {
#pragma unroll
        for (int q = 0; q < H; q++) {
          const uint32_t s = swap_halves(P[q]);
          P[q] = __byte_perm(__vminu2(P[q], s), __vmaxu2(P[q], s), 0x7610);
        }
      } else {
        const int lm = j / E;
        const bool keepmin = (lane & lm) == 0;
#pragma unroll
        for (int q = 0; q < H; q++) {
          uint32_t v = __shfl_xor_sync(0xffffffffu, P[q], lm);
          P[q] = keepmin ? __vminu2(P[q], v) : __vmaxu2(P[q], v);
        }
      }
    }
  }
}

// A lane's sorted keys as emit_sorted reads them: key(r) at sorted index lane*E + r, the last one, and the
// mask of run starts (bit r: key(r) differs from the key before it; prevlast: the previous lane's last key).
template <int E>
struct Keys32 {
  const uint32_t (&K)[E];
  __device__ __forceinline__ uint32_t key(int r) const { return K[r]; }
  __device__ __forceinline__ uint32_t last() const { return K[E - 1]; }
  template <class MaskT>
  __device__ __forceinline__ MaskT bounds(uint32_t prevlast, unsigned) const {
    MaskT bnd = (MaskT)(K[0] != prevlast);
#pragma unroll
    for (int r = 1; r < E; r++) bnd |= (MaskT)(K[r] != K[r - 1]) << r;
    return bnd;
  }
};
template <int E>
struct Keys16 {
  static constexpr int H = E / 2;
  const uint32_t (&P)[H];
  __device__ __forceinline__ uint32_t key(int r) const { return r < H ? P[r] & 0xFFFFu : P[r - H] >> 16; }
  __device__ __forceinline__ uint32_t last() const { return P[H - 1] >> 16; }
  template <class MaskT>
  __device__ __forceinline__ MaskT bounds(uint32_t prevlast, unsigned lane) const {
    // __vsetne2 compares both halves at once: bit 0 of the result is index q, bit 16 index q + H
    // (lane 0 starts a run at index 0 whatever the low half of NOKEY compares to)
    const uint32_t s0 = __vsetne2(P[0], __byte_perm(prevlast, P[H - 1], 0x5410)) | (lane == 0 ? 1u : 0u);
    if constexpr (H <= 16) {
      uint32_t acc = s0;
#pragma unroll
      for (int q = 1; q < H; q++) acc |= __vsetne2(P[q], P[q - 1]) << q;
      return (MaskT)((acc & ((1u << H) - 1u)) | ((acc >> 16) << H));
    } else {
      uint32_t lo = s0 & 1u, hi = s0 >> 16;
#pragma unroll
      for (int q = 1; q < H; q++) {
        const uint32_t s = __vsetne2(P[q], P[q - 1]);
        lo |= (s & 1u) << q; hi |= (s >> 16) << q;
      }
      return (MaskT)lo | ((MaskT)hi << H);
    }
  }
};

struct Emitter {
  uint32_t *sid, *scnt;            // this row's slices of the column / count arrays
  uint32_t *obs, *bitmap;          // observed classes: per-block (shared) and global bitmap
  const uint2 *nbx;                // numbering set, per 32 ids: x = member bits, y = column of the first member
  uint32_t obs_bits;               // ids below this are marked in obs
  uint32_t cursor;
  int binarize, mark, filter;      // filter: ids outside the numbering set are dropped (frozen class list)
  unsigned long long sq;           // per lane: sum of squared counts / largest count emitted
  uint32_t vm;
  uint32_t ev;                     // repeat events written so far (binarized rows, downwards from the row's last slot)
  // mark one class id as observed
  __device__ __forceinline__ void mark_id(uint32_t id) {
    if (!mark) return;
    const uint32_t bit = 1u << (id & 31), w = id >> 5;
    if (id < obs_bits) { if (!(obs[w] & bit)) atomicOr(obs + w, bit); }
    else if (!(bitmap[w] & bit)) atomicOr(bitmap + w, bit);
  }
  // OR a word of 32 consecutive class ids (a level <= OBS_MAX_LEVEL) into the block's bitmap
  __device__ __forceinline__ void mark_word(uint32_t word_index, uint32_t bits) {
    if (mark && (bits & ~obs[word_index])) atomicOr(obs + word_index, bits);
  }
  // column of a class id; false when the id is not in the numbering set
  __device__ __forceinline__ bool column(uint32_t id, uint32_t &col) const {
    const uint2 e = __ldg(nbx + (id >> 5));
    const uint32_t bit = 1u << (id & 31);
    col = e.y + __popc(e.x & (bit - 1u));
    return (e.x & bit) != 0u;
  }
  __device__ __forceinline__ void stat(uint32_t cnt) {
    sq += (unsigned long long)cnt * cnt;
    vm = max(vm, cnt);
  }
  // ballot-compacted emission (coalesced stores); col_known >= 0: the column when no class is dropped
  template <bool MARK = true>
  __device__ __forceinline__ unsigned emit(bool flag, uint32_t id, uint32_t cnt, int64_t col_known = -1) {
    uint32_t col = (uint32_t)col_known;
    if (flag && (filter || col_known < 0)) { const bool member = column(id, col); if (filter) flag = member; }
    unsigned em = __ballot_sync(0xffffffffu, flag);
    if (flag) {
      uint32_t pos = cursor + __popc(em & lanemask_lt());
      sid[pos] = col;
      if (!binarize) scnt[pos] = cnt;
      if (MARK) mark_id(id);
      stat(binarize ? 1u : cnt);
    }
    cursor += __popc(em);
    return em;
  }
};

__host__ __device__ constexpr int ext_threads(int E) { return E <= 16 ? 512 : (E == 32 ? 256 : 128); }

// ---- sorted level: the canonical codes of one level, sorted in registers -----------------------------
// K[r] sits at sorted index lane*E + r.  A run (equal keys) is one class, its length the count; a run
// is emitted by the lane holding the position right after it.  Ids and counts go through the warp's
// shared-memory buffer so that the global stores are coalesced.
template <int E, class Keys>
__device__ __forceinline__ void emit_sorted(const Keys &K, unsigned lane, uint32_t *sbuf, Emitter &em,
                                            uint32_t idbase, int events, int64_t stride) {
  using MaskT = typename std::conditional<(E <= 32), uint32_t, unsigned long long>::type;
  uint32_t prevlast = __shfl_up_sync(0xffffffffu, K.last(), 1);
  if (lane == 0) prevlast = NOKEY;
  // bit r of bnd: a run starts at this lane's key r (sorted index lane*E + r)
  const MaskT bnd = K.template bounds<MaskT>(prevlast, lane);
  // a run is emitted by the position right after it: every boundary but sorted index 0
  const MaskT cls = lane == 0 ? (bnd & ~(MaskT)1) : bnd;
  const int c = sizeof(MaskT) == 4 ? __popc((uint32_t)cls) : __popcll(cls);
  const int lastb = bnd ? (int)lane * E + (sizeof(MaskT) == 4 ? 31 - __clz((uint32_t)bnd) : 63 - __clzll(bnd)) : -1;
  int incl = c, mx = lastb;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, incl, o), z = __shfl_up_sync(0xffffffffu, mx, o);
    if (lane >= (unsigned)o) { incl += y; mx = max(mx, z); }
  }
  const int base = incl - c, total = __shfl_sync(0xffffffffu, incl, 31);
  // the last run of the sorted array is the run of SENT keys (a level has fewer valid keys than sort slots): its start
  // is the number of valid keys, and valid keys - classes = repeats of the level
  const int nvalid = __shfl_sync(0xffffffffu, mx, 31);
  int start0 = __shfl_up_sync(0xffffffffu, mx, 1);   // last boundary before this lane's keys
  if (lane == 0) start0 = 0;
  // the runs this lane emits, in sorted order: f(j = entry of the level, r, count).  The run emitted at key r
  // started at the last boundary below r (start0 when this lane has none below r); j counts up from base.
  auto each_run = [&](auto &&f) {
    int j = base;
#pragma unroll
    for (int r = 0; r < E; r++)
      if ((cls >> r) & 1) {
        const MaskT bbelow = bnd & (((MaskT)1 << r) - 1);
        const int st = bbelow ? (int)lane * E + (sizeof(MaskT) == 4 ? 31 - __clz((uint32_t)bbelow) : 63 - __clzll(bbelow))
                              : start0;
        f(j, r, (uint32_t)((int)lane * E + r - st)); j++;
      }
  };
  // round 1: ids
  each_run([&](int j, int r, uint32_t) { sbuf[sw(j)] = idbase + (r == 0 ? prevlast : K.key(r > 0 ? r - 1 : 0)); });
  __syncwarp();
  // binarized rows feeding the matrix-free logistic pass: a run of r > 1 equal keys leaves r - 1 repeat
  // events (the column of its class) at the tail of the row's slots, in sorted order (while sbuf holds the ids)
  auto repeat_events = [&]() {
    uint32_t extra = 0;
    each_run([&](int j, int, uint32_t cnt) {
      uint32_t col;
      if (cnt > 1 && (em.column(sbuf[sw(j)], col) || !em.filter)) extra += cnt - 1;
    });
    uint32_t incl = extra;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (unsigned)o) incl += y;
    }
    const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
    if (tot == 0) return;
    uint32_t *tail = em.sid + stride - 1;
    uint32_t pos = em.ev + incl - extra;
    each_run([&](int j, int, uint32_t cnt) {
      uint32_t col;
      if (cnt > 1 && (em.column(sbuf[sw(j)], col) || !em.filter))
        for (uint32_t x = 1; x < cnt; x++) tail[-(int64_t)(pos++)] = col;
    });
    em.ev += tot;
  };
  if (!em.filter) {
    // no class is dropped: slot i of the buffer is entry i of the level
    // four numbering gathers in flight per lane (each is an L2 round trip)
    for (int i0 = lane; i0 < total; i0 += 128) {
      uint32_t id[4];
      uint2 e[4];
#pragma unroll
      for (int j = 0; j < 4; j++) id[j] = i0 + 32 * j < total ? sbuf[sw(i0 + 32 * j)] : idbase;
#pragma unroll
      for (int j = 0; j < 4; j++) e[j] = __ldg(em.nbx + (id[j] >> 5));
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (i0 + 32 * j < total) {
          em.sid[em.cursor + i0 + 32 * j] = e[j].y + __popc(e[j].x & ((1u << (id[j] & 31)) - 1u));
          em.mark_id(id[j]);
        }
      }
    }
    __syncwarp();
    if (!em.binarize) {
      each_run([&](int j, int, uint32_t cnt) { sbuf[sw(j)] = cnt; em.stat(cnt); });
      __syncwarp();
      for (int i = lane; i < total; i += 32) em.scnt[em.cursor + i] = sbuf[sw(i)];
      __syncwarp();
    } else {
      em.sq += (unsigned long long)c; if (c) em.vm = max(em.vm, 1u);
      if (events && nvalid > total) { repeat_events(); __syncwarp(); }
    }
    em.cursor += (uint32_t)total;
    return;
  }
  // copy out: id -> column; with a frozen class list the ids outside the list are dropped here and the
  // keep decisions (one bit per copy iteration) are replayed for the counts
  unsigned long long keepbits = 0;
  uint32_t kept = 0;
  for (int i0 = 0, it = 0; i0 < total; i0 += 32, it++) {
    const int i = i0 + (int)lane;
    bool keep = false; uint32_t col = 0, id = 0;
    if (i < total) { id = sbuf[sw(i)]; keep = em.column(id, col) || !em.filter; }
    const unsigned km = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      em.sid[em.cursor + kept + __popc(km & lanemask_lt())] = col;
      em.mark_id(id);
      keepbits |= 1ull << it;
    }
    kept += __popc(km);
  }
  __syncwarp();
  // round 2: counts = distance to the previous boundary
  if (!em.binarize) {
    each_run([&](int j, int, uint32_t cnt) { sbuf[sw(j)] = cnt; });
    __syncwarp();
    uint32_t k2 = 0;
    for (int i0 = 0, it = 0; i0 < total; i0 += 32, it++) {
      const int i = i0 + (int)lane;
      const bool keep = (keepbits >> it) & 1ull;
      const unsigned km = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const uint32_t cnt = sbuf[sw(i)];
        em.scnt[em.cursor + k2 + __popc(km & lanemask_lt())] = cnt;
        em.stat(cnt);
      }
      k2 += __popc(km);
    }
    __syncwarp();
  } else {
    em.sq += __popcll(keepbits); if (keepbits) em.vm = max(em.vm, 1u);
    if (events && nvalid > total) { repeat_events(); __syncwarp(); }
  }
  em.cursor += kept;
}


// A lane's view of its stretch of a row: 32 consecutive bases starting at p0, once with the first base in the
// low bits (fwd: the k-mer starting at base x is the low 2k bits of fwd >> 2x, and the complement of those
// bits is its reverse complement in code order) and once digit-reversed, first base in the two top bits (rev:
// a shift and a mask give the forward code, first base most significant), + one "not usable" bit per base
// (not ACGT, or past the end of the row).
struct XWindow {
  unsigned long long fwd, rev;
  uint32_t inv;
  __device__ __forceinline__ void load(const uint32_t *__restrict__ b2, const uint16_t *__restrict__ iv, int L, int p0) {
    if (p0 >= L) { fwd = rev = 0ull; inv = 0xFFFFFFFFu; return; }
    const int wi = p0 >> 4, sh = p0 & 15;
    const uint32_t w0 = __ldg(b2 + wi), w1 = __ldg(b2 + wi + 1), w2 = __ldg(b2 + wi + 2);
    const uint32_t lo = __funnelshift_r(w0, w1, 2 * sh), hi = __funnelshift_r(w1, w2, 2 * sh);
    fwd = ((unsigned long long)hi << 32) | lo;
    rev = ((unsigned long long)swap_pairs(__brev(lo)) << 32) | swap_pairs(__brev(hi));
    const unsigned long long iw = (unsigned long long)__ldg(iv + wi) | ((unsigned long long)__ldg(iv + wi + 1) << 16) |
                                  ((unsigned long long)__ldg(iv + wi + 2) << 32);
    inv = (uint32_t)(iw >> sh);
    const int left = L - p0;
    if (left < 32) inv |= 0xFFFFFFFFu << left;
  }
};

// ---- the extraction kernel: one warp per sequence ------------------------------------------------
// E = keys per lane of the register sort (0: no sorted levels, sequences of any length)
// OPT: the strand operation when it is known at compile time (1 = revcomp, the common case), -1 = P.op
// EV: binarized rows that also leave their table-level class bitmap and repeat events (XParams::events)
// PK: revcomp with N <= PACK_MAX: the sorted levels take the 16-bit network (warp_sort16)
template <int E, int OPT, bool EV, bool PK>
__global__ void __launch_bounds__(ext_threads(E), 2) extract_kernel(const XParams P) {
  static_assert(!PK || (E >= 2 && OPT == 1), "the 16-bit sort keys need revcomp and two keys per lane");
  constexpr int EE = E > 0 ? E : 1;
  extern __shared__ __align__(16) uint32_t smem[];
  const unsigned lane = lane_id();
  const int warp_in_block = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  // block: [observed classes]; per warp: [bitmaps][prefix][count tables | sort buffer][dup count + dups]
  uint32_t *obs = smem;
  uint32_t *bm = smem + P.obs_words + (size_t)warp_in_block * P.warp_words;
  uint32_t *pf = bm + P.bm_words;
  uint32_t *tab = pf + P.pf_words;
  uint32_t *dupn = tab + P.ts_words;
  const int64_t gwarp = (int64_t)blockIdx.x * wpb + warp_in_block;
  uint32_t *ovf = P.ovf ? P.ovf + gwarp * P.ovf_stride : nullptr;
  const int N = P.N, M = P.M, op = OPT >= 0 ? OPT : P.op;
  const bool two = op != 0;
  const uint32_t maskN = (1u << (2 * N)) - 1u;
  const bool has_tab = P.t_lo <= P.t_hi, has_bm = P.b_lo <= P.b_hi, has_sort = E > 0 && P.s_lo <= N;
  const bool single_sorted = has_sort && P.s_lo == N && op != 2;   // (complement: the image is not a window image)

  // shared memory starts clean; every row leaves its bitmaps clean again
  for (int i = threadIdx.x; i < P.obs_words; i += blockDim.x) obs[i] = 0;
  for (int i = lane; i < P.bm_words; i += 32) bm[i] = 0;
  if (lane == 0) dupn[0] = 0;
  __syncthreads();

  // The body of this loop is ~150 KB of unrolled code, several times the SM's instruction cache, and
  // the kernel is bound by instruction fetch (ncu: the GPC instruction cache at 88 % of its request
  // rate).  The warps of a block therefore start every row together: a fetched line then serves
  // many warps (measured 3.03 -> 2.73 ms at C2).  More barriers inside the row, 1024-thread blocks and
  // a compact re-rolled body were all measured slower.  A warp past the last row runs an empty row.
  // Groups of rows (one row per warp) are handed out through a ticket counter: the blocks that run
  // faster take more groups.
  uint32_t *s_ticket = smem + P.obs_words + P.bm_words + P.pf_words + P.ts_words + 1;   // warp 0's spare word
  // Marks of the observed classes: on real inputs every class of the configuration has shown up after the first few
  // thousand rows of the launch, and from then on a mark is a shared-memory (levels > OBS_MAX_LEVEL: L2) read per
  // emitted entry that never changes anything.  After 4, 8, 16, ... groups of rows a block therefore flushes its
  // marks and looks whether the device-wide bitmap covers the numbering set; once it does (P.full) nobody marks.
  auto flush_marks = [&]() {
    for (int i = threadIdx.x; i < P.obs_id_words; i += blockDim.x) {
      const uint32_t w = obs[i];
      if (w && (w & ~P.bitmap[i])) atomicOr(P.bitmap + i, w);
    }
    if (P.t_lo <= P.t_hi)
      for (uint32_t j = threadIdx.x; j < P.tl_cnt; j += blockDim.x)
        if ((obs[P.obs_id_words + (j >> 5)] >> (j & 31)) & 1u) {
          const uint32_t id = __ldg(P.tl + j).y;
          if (!((P.bitmap[id >> 5] >> (id & 31)) & 1u)) atomicOr(P.bitmap + (id >> 5), 1u << (id & 31));
        }
  };
  int mk = P.mark;
  uint32_t groups = 0, next_check = KL_X_MARKSKIP ? 4u : 0xFFFFFFFFu;
  if (mk) mk = __syncthreads_or(threadIdx.x == 0 && *(volatile uint32_t *)P.full == 0u) ? 1 : 0;
  // (the ticket of the NEXT group is drawn while this one is worked on: the atomic's round trip is off the path)
#if KL_X_TKPRE
  uint32_t tk = threadIdx.x == 0 ? atomicAdd(P.ticket, 1u) : 0u;
#endif
  for (;;) {
    __syncthreads();
#if KL_X_TKPRE
    if (threadIdx.x == 0) *s_ticket = tk;
#else
    if (threadIdx.x == 0) *s_ticket = atomicAdd(P.ticket, 1u);
#endif
    __syncthreads();
    const int64_t row0 = P.row0 + (int64_t)*s_ticket * wpb;
    if (row0 >= P.n) break;
#if KL_X_TKPRE
    if (threadIdx.x == 0) tk = atomicAdd(P.ticket, 1u);
#endif
    const int64_t row = row0 + warp_in_block;
    const bool active = row < P.n;
    const int L = active ? (int)P.len[row] : 0;
    const int64_t blk0 = active ? P.blk[row] : 0;
    const uint32_t *b2 = P.bits2 + blk0 * 4;
    const uint16_t *iv16 = P.inv16 + blk0 * 4;
    if (has_tab)
      for (int i = lane; i < TAB_WORDS; i += 32) tab[i] = 0;
    __syncwarp();

#if KL_X_OLDPOS
    // ---- pass over the positions: lane handles the start positions p = lane, lane + 32, ... ----------
    // The N bases starting at p are 2N consecutive bits of the packed words (first base in the low
    // bits): one funnel shift.  Read that way the k-mer starting at p is the LOW 2k bits, its
    // reverse complement (first base most significant, the code order) is the complement of those
    // bits and its forward code is their digit reversal -- no rolling state, no warm-up.
    const int steps = (L + 31) / 32;
    uint32_t FWL[EE];                 // (forward code << 4) | valid length, per position of this lane
#pragma unroll
    for (int r = 0; r < EE; r++) FWL[r] = 0;
    {
      auto visit = [&](int p) -> uint32_t {
        const int wi = p >> 4, sh = p & 15;
        const uint32_t e = __funnelshift_r(__ldg(b2 + wi), __ldg(b2 + wi + 1), 2 * sh) & maskN;
        const uint32_t ivb = (((uint32_t)__ldg(iv16 + wi) | ((uint32_t)__ldg(iv16 + wi + 1) << 16)) >> sh) |
                             (1u << min(N, L - p));       // the sequence ends: no k-mer reaches past L
        const int len_f = __ffs(ivb) - 1;                 // valid bases from p on (<= N)
        const uint32_t FW = swap_pairs(__brev(e)) >> (32 - 2 * N);
        const uint32_t S2 = op == 1 ? (~e) & maskN : e;   // image of the window under revcomp / reverse
        if (len_f >= M) {
          // table levels: one count at the deepest table level this suffix reaches
          if (has_tab) {
            int kk = len_f < P.t_hi ? len_f : P.t_hi;
            if (kk >= P.t_lo) {
              uint32_t idx = tab_off(kk) + (FW >> (2 * (N - kk)));
              atomicAdd(tab + sw(idx >> 1), 1u << (16 * (idx & 1)));
            }
          }
          // bitmap levels: canonical code = min(prefix, image)
          if (has_bm) {
#pragma unroll
            for (int j = 0; j < KB_MAX - KT_MAX; j++) {
              const int k = P.b_lo + j;
              if (k > P.b_hi || len_f < k) break;
              const uint32_t mk = (1u << (2 * k)) - 1u;
              uint32_t c = FW >> (2 * (N - k));
              if (op == 1 || op == 3) c = min(c, S2 & mk);
              else if (op == 2) c = min(c, (~c) & mk);
              const uint32_t bit = 1u << (c & 31);
              const uint32_t old = atomicOr(bm + P.bm_off[k] + (c >> 5), bit);
              if ((old & bit) && (!P.binarize || EV)) {
                ovf[atomicAdd(dupn, 1u)] = ((uint32_t)k << 26) | c;     // the warp's list of repeats (L2)
              }
            }
          }
        }
        // one sorted level (s_lo == N): keep the CANONICAL code of the full window, the key of that level
        const uint32_t keep = (single_sorted && two) ? min(FW, S2) : FW;
        return (keep << 4) | (uint32_t)len_f;
      };
      if (E > 0) {
#pragma unroll
        for (int i = 0; i < EE; i++) {
          const int p = i * 32 + (int)lane;
          if (p < L) FWL[i] = visit(p);
        }
      } else {
        for (int i = 0; i < steps; i++) {
          const int p = i * 32 + (int)lane;
          if (p < L) visit(p);
        }
      }
    }
    __syncwarp();

    const int spl = (L + 31) >> 5, p0 = (int)lane * spl;
#else
    // ---- pass over the positions: lane owns the start positions [lane spl, (lane + 1) spl) ----------------
    // Its stretch is read once per 16 positions as a 64-bit window of packed bases (XWindow): the k-mer
    // starting at base x of the window is a shift and a mask -- no rolling state, no warm-up, no load or
    // bit reversal per position.
    const int spl = (L + 31) >> 5;    // start positions per lane
    const int p0 = (int)lane * spl;
    uint32_t FWL[EE];                 // (forward code << 4) | valid length, per position of this lane
#pragma unroll
    for (int r = 0; r < EE; r++) FWL[r] = 0;
    {
      const uint32_t tab_top = has_tab ? tab_off(P.t_hi) : 0u;
      auto visit = [&](const XWindow &W, int x) -> uint32_t {
        const int len_f = __ffs((W.inv >> x) | (1u << N)) - 1;                 // valid bases from here on (<= N)
        const uint32_t e = (uint32_t)(W.fwd >> (2 * x)) & maskN;
        const uint32_t FW = (uint32_t)(W.rev >> (64 - 2 * (x + N))) & maskN;
        const uint32_t S2 = op == 1 ? (~e) & maskN : e;   // image of the window under revcomp / reverse
        if (len_f >= M) {
          // table levels: one count at the deepest table level this suffix reaches
          if (has_tab) {
            uint32_t idx;
            if (len_f >= P.t_hi) idx = tab_top + (FW >> (2 * (N - P.t_hi)));
            else idx = len_f >= P.t_lo ? tab_off(len_f) + (FW >> (2 * (N - len_f))) : 0xFFFFFFFFu;
            if (idx != 0xFFFFFFFFu) atomicAdd(tab + sw(idx >> 1), 1u << (16 * (idx & 1)));
          }
          // bitmap levels: canonical code = min(prefix, image)
          if (has_bm) {
#pragma unroll
            for (int j = 0; j < KB_MAX - KT_MAX; j++) {
              const int k = P.b_lo + j;
              if (k > P.b_hi || len_f < k) break;
              const uint32_t mk = (1u << (2 * k)) - 1u;
              uint32_t c = FW >> (2 * (N - k));
              if (op == 1 || op == 3) c = min(c, S2 & mk);
              else if (op == 2) c = min(c, (~c) & mk);
              const uint32_t bit = 1u << (c & 31);
              const uint32_t old = atomicOr(bm + P.bm_off[k] + (c >> 5), bit);
              if ((old & bit) && (!P.binarize || EV)) {
                ovf[atomicAdd(dupn, 1u)] = ((uint32_t)k << 26) | c;     // the warp's list of repeats (L2)
              }
            }
          }
        }
        // one sorted level (s_lo == N): keep the CANONICAL code of the full window, the key of that level
        const uint32_t keep = (single_sorted && two) ? min(FW, S2) : FW;
        return (keep << 4) | (uint32_t)len_f;
      };
      XWindow W;
      if (E > 0) {
#pragma unroll
        for (int i = 0; i < EE; i++) {
          if ((i & 15) == 0 && i < spl) W.load(b2, iv16, L, p0 + i);
          if (i < spl && p0 + i < L) FWL[i] = visit(W, i & 15);
        }
      } else {
        for (int i = 0; i < spl && p0 + i < L; i++) {
          if ((i & 15) == 0) W.load(b2, iv16, L, p0 + i);
          visit(W, i & 15);
        }
      }
    }
    __syncwarp();

#endif
    Emitter em;
    em.sid = P.st_id + row * P.stride; em.scnt = P.st_cnt + (P.binarize ? 0 : row * P.stride);
    em.obs = obs; em.bitmap = P.bitmap; em.obs_bits = (uint32_t)P.obs_id_words * 32u;
    em.nbx = P.nbx; em.filter = P.filter;
    em.cursor = 0; em.binarize = P.binarize; em.mark = mk;
    em.sq = 0; em.vm = 0;
    em.ev = 0;

    // ---- table levels ---------------------------------------------------------------------------
    if (has_tab) {
      // a k-mer count is the sum of its 4 extensions plus the suffixes that end right after it
      for (int k = P.t_hi - 1; k >= P.t_lo; k--) {
        const uint32_t nk = 1u << (2 * k), toff = tab_off(k), coff = tab_off(k + 1);
#if KL_X_NOSWZ
        // a lane takes the two parents that share a word: their 8 children are four consecutive words
        for (uint32_t u2 = lane; u2 < nk / 2; u2 += 32) {
          const uint2 a = *reinterpret_cast<const uint2 *>(tab + (coff >> 1) + 4 * u2);
          const uint2 b = *reinterpret_cast<const uint2 *>(tab + (coff >> 1) + 4 * u2 + 2);
          const uint32_t s0 = (a.x & 0xFFFFu) + (a.x >> 16) + (a.y & 0xFFFFu) + (a.y >> 16);
          const uint32_t s1 = (b.x & 0xFFFFu) + (b.x >> 16) + (b.y & 0xFFFFu) + (b.y >> 16);
          tab[(toff >> 1) + u2] += s0 | (s1 << 16);
        }
#else
        for (uint32_t u = lane; u < nk; u += 32) {
          uint32_t c0 = coff + 4 * u;                 // 4 children = two aligned words
          uint32_t w0 = tab[sw(c0 >> 1)], w1 = tab[sw(c0 >> 1) ^ 1u];   // (the swizzle keeps an even / odd pair together)
          uint32_t sum = (w0 & 0xFFFFu) + (w0 >> 16) + (w1 & 0xFFFFu) + (w1 >> 16);
          uint32_t idx = toff + u;
          if (sum) atomicAdd(tab + sw(idx >> 1), sum << (16 * (idx & 1)));
        }
#endif
        __syncwarp();
      }
      // walk the classes of the table levels in (k, code) order: count = code + image
      uint32_t mylow = 0, mylow2 = 0;                      // lane w: words w and w + 32 of the row's table-level class bitmap
      uint2 e_next = lane < P.tl_cnt ? __ldg(P.tl + lane) : make_uint2(0u, 0u);
      for (uint32_t base = 0; base < P.tl_cnt; base += 32) {
        const uint32_t j = base + lane;
        uint32_t id = 0, cnt = 0;
#if KL_X_TLPIPE
        const uint2 e = e_next;
        if (j + 32 < P.tl_cnt) e_next = __ldg(P.tl + j + 32);
#else
        const uint2 e = j < P.tl_cnt ? __ldg(P.tl + j) : e_next;
#endif
        if (j < P.tl_cnt) {
          const unsigned char *tb = reinterpret_cast<const unsigned char *>(tab);
          cnt = (uint32_t)*reinterpret_cast<const unsigned short *>(tb + (e.x & 0xFFFFu)) +
                (uint32_t)*reinterpret_cast<const unsigned short *>(tb + (e.x >> 16));
          id = e.y;
        }
        // without a frozen list the numbering set is ALL classes: the j-th class of the list is column j
        const unsigned kept = em.emit<false>(cnt > 0, id, cnt, P.filter ? -1 : (int64_t)j);
        // marks of the table levels: one word per 32 list entries (translated to class ids when the block ends)
        if (mk && lane == 0 && (kept & ~obs[P.obs_id_words + (base >> 5)])) atomicOr(obs + P.obs_id_words + (base >> 5), kept);
        if (EV && lane == ((base >> 5) & 31u)) { if (base < 1024u) mylow = kept; else mylow2 = kept; }
      }
      if (EV && P.lowbits && active) {
        if ((int)lane < P.low_words) P.lowbits[row * P.low_words + lane] = mylow;
        if ((int)lane + 32 < P.low_words) P.lowbits[row * P.low_words + lane + 32] = mylow2;
      }
      __syncwarp();
    }

#if KL_X_WALK
    // ---- bitmap levels: walk the bitmap 128 words at a time (4 consecutive words per lane) ---------
    if (has_bm) {
      for (int k = P.b_lo; k <= P.b_hi; k++) {
        const int W = 1 << (2 * k - 5);
        uint32_t *bk = bm + P.bm_off[k];
        uint32_t *pk = pf + P.pf_off[k];
        const uint32_t gword = P.level_off[k] >> 5;
        for (int it = 0; it * 128 < W; it++) {
          const int wi = it * 128 + (int)lane * 4;
          uint4 w4 = make_uint4(0, 0, 0, 0);
          if (wi < W) w4 = *reinterpret_cast<const uint4 *>(bk + wi);
          // numbering of the lane's 4 words: member bits and column of the first member (coalesced loads)
          uint2 nx[4];
#pragma unroll
          for (int j = 0; j < 4; j++) nx[j] = wi < W ? __ldg(P.nbx + gword + wi + j) : make_uint2(0u, 0u);
          if (P.filter && wi < W) {
            // frozen class list: classes outside the list vanish here, before any slot is assigned
            w4.x &= nx[0].x; w4.y &= nx[1].x; w4.z &= nx[2].x; w4.w &= nx[3].x;
            *reinterpret_cast<uint4 *>(bk + wi) = w4;
          }
          if (w4.x | w4.y | w4.z | w4.w) {
            em.mark_word(gword + wi, w4.x); em.mark_word(gword + wi + 1, w4.y);
            em.mark_word(gword + wi + 2, w4.z); em.mark_word(gword + wi + 3, w4.w);
          }
          const uint32_t c = __popc(w4.x) + __popc(w4.y) + __popc(w4.z) + __popc(w4.w);
          uint32_t incl = c;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += y;
          }
          const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
          if (wi < W) pk[wi >> 2] = em.cursor + incl - c;   // slot of this lane's first class
          const uint32_t ws[4] = {w4.x, w4.y, w4.z, w4.w};
          if (tot <= (uint32_t)P.ts_words) {
            // ids through the warp's shared buffer: coalesced global stores of the columns
            uint32_t pos = incl - c;
#pragma unroll
            for (int j = 0; j < 4; j++) {
              uint32_t w = ws[j];
              while (w) {
                const uint32_t below = (w & (0u - w)) - 1u;            // bits under the lowest set bit
                tab[sw(pos++)] = nx[j].y + __popc(nx[j].x & below);     // its column
                w &= w - 1;
              }
            }
            __syncwarp();
            for (uint32_t i = lane; i < tot; i += 32) {
              em.sid[em.cursor + i] = tab[sw(i)];
              if (!P.binarize) em.scnt[em.cursor + i] = 1;
            }
            __syncwarp();
          } else {
            uint32_t pos = em.cursor + incl - c;
#pragma unroll
            for (int j = 0; j < 4; j++) {
              uint32_t w = ws[j];
              while (w) {
                const uint32_t below = (w & (0u - w)) - 1u;
                w &= w - 1;
                em.sid[pos] = nx[j].y + __popc(nx[j].x & below);
                if (!P.binarize) em.scnt[pos] = 1;
                pos++;
              }
            }
          }
          em.sq += c; if (c) em.vm = max(em.vm, 1u);        // every class of the chunk enters with count 1
          em.cursor += tot;
        }
      }
#else
    // ---- bitmap levels ---------------------------------------------------------------------------------
    // (1) one pass over the words of the level's bitmap (4 consecutive words per lane): frozen-list filter,
    // marks of the observed classes, popcounts -> the slot of the first class of every PAIR of words (u16);
    // (2) every position computes the slot of its class from that prefix and two popcounts, and puts the
    // column there (repeats of a class write the same value to the same slot) -- no loop over set bits;
    // (3) the staged columns leave in coalesced stores.
    if (has_bm) {
      for (int k = P.b_lo; k <= P.b_hi; k++) {
        const int W = 1 << (2 * k - 5);
        uint32_t *bk = bm + P.bm_off[k];
        unsigned short *pk = reinterpret_cast<unsigned short *>(pf + P.pf_off[k]);
        const uint32_t gword = P.level_off[k] >> 5;
        uint32_t run = 0;                                     // classes of the words before this chunk
        for (int it = 0; it * 128 < W; it++) {
          const int wi = it * 128 + (int)lane * 4;
          uint4 w4 = make_uint4(0, 0, 0, 0);
          if (wi < W) w4 = *reinterpret_cast<const uint4 *>(bk + wi);
          if (P.filter && wi < W) {
            // frozen class list: classes outside the list vanish here, before any slot is assigned
            w4.x &= __ldg(P.nbx + gword + wi).x; w4.y &= __ldg(P.nbx + gword + wi + 1).x;
            w4.z &= __ldg(P.nbx + gword + wi + 2).x; w4.w &= __ldg(P.nbx + gword + wi + 3).x;
            *reinterpret_cast<uint4 *>(bk + wi) = w4;
          }
          if (w4.x | w4.y | w4.z | w4.w) {
            em.mark_word(gword + wi, w4.x); em.mark_word(gword + wi + 1, w4.y);
            em.mark_word(gword + wi + 2, w4.z); em.mark_word(gword + wi + 3, w4.w);
          }
          const uint32_t c01 = __popc(w4.x) + __popc(w4.y), c = c01 + __popc(w4.z) + __popc(w4.w);
          uint32_t incl = c;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (unsigned)o) incl += y;
          }
          if (wi < W) {
            const uint32_t first = run + incl - c;
            *reinterpret_cast<uint32_t *>(pk + (wi >> 1)) = first | ((first + c01) << 16);   // pairs (wi, wi+1), (wi+2, wi+3)
          }
          run += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
        const uint32_t tot = run;
        const bool staged = tot <= (uint32_t)P.ts_words;
        const uint32_t mk = (1u << (2 * k)) - 1u;
        auto place = [&](const XWindow &V, int x) {
          if (__ffs((V.inv >> x) | (1u << N)) - 1 < k) return;          // no valid k-mer starts here
          uint32_t c = (uint32_t)(V.rev >> (64 - 2 * (x + k))) & mk;
          if (op == 1) c = min(c, ~(uint32_t)(V.fwd >> (2 * x)) & mk);
          else if (op == 3) c = min(c, (uint32_t)(V.fwd >> (2 * x)) & mk);
          else if (op == 2) c = min(c, (~c) & mk);
          const uint32_t wd = c >> 5, bit = 1u << (c & 31), wv = bk[wd];
          if (!(wv & bit)) return;                                      // class dropped by the frozen list
          uint32_t slot = pk[wd >> 1] + __popc(wv & (bit - 1u));
          if (wd & 1u) slot += __popc(bk[wd - 1]);
          uint32_t col;
          em.column(P.level_off[k] + c, col);
          if (staged) tab[sw(slot)] = col; else em.sid[em.cursor + slot] = col;
        };
        {
          XWindow V;
          if (E > 0) {
#pragma unroll
            for (int i = 0; i < EE; i++) {
              if ((i & 15) == 0 && i < spl) V.load(b2, iv16, L, p0 + i);
              if (i < spl && p0 + i < L) place(V, i & 15);
            }
          } else {
            for (int i = 0; i < spl && p0 + i < L; i++) {
              if ((i & 15) == 0) V.load(b2, iv16, L, p0 + i);
              place(V, i & 15);
            }
          }
        }
        __syncwarp();
        for (uint32_t i = lane; i < tot; i += 32) {
          if (staged) em.sid[em.cursor + i] = tab[sw(i)];
          if (!P.binarize) em.scnt[em.cursor + i] = 1;
        }
        __syncwarp();
        if (lane == 0) {
          dupn[4 + k - P.b_lo] = em.cursor;                             // row slot of the level's first class (repeats below)
          em.sq += tot;                                                 // every class of the level enters with count 1
        }
        if (tot) em.vm = max(em.vm, 1u);
        em.cursor += tot;
      }
#endif
      __syncwarp();
      __threadfence_block();
      // repeats: add one to the count of the class, found by its rank in the bitmap
      if (!P.binarize) {
        const uint32_t nd = dupn[0];
        for (uint32_t i = lane; i < nd; i += 32) {
          const uint32_t e = ovf[i];
          const uint32_t k = e >> 26, c = e & 0x3FFFFFFu, wi = c >> 5;
          const uint32_t *bk = bm + P.bm_off[k];
          if (!((bk[wi] >> (c & 31)) & 1u)) continue;       // class dropped by the frozen list
#if KL_X_WALK
          uint32_t slot = pf[P.pf_off[k] + (wi >> 2)] + __popc(bk[wi] & ((1u << (c & 31)) - 1u));
          for (uint32_t j = wi & ~3u; j < wi; j++) slot += __popc(bk[j]);
#else
          uint32_t slot = dupn[4 + k - P.b_lo] + reinterpret_cast<const unsigned short *>(pf + P.pf_off[k])[wi >> 1] +
                          __popc(bk[wi] & ((1u << (c & 31)) - 1u));
          if (wi & 1u) slot += __popc(bk[wi - 1]);
#endif
          const uint32_t old = atomicAdd(em.scnt + slot, 1u);
          em.sq += 2ull * old + 1ull;                       // (old+1)^2 - old^2
          em.vm = max(em.vm, old + 1u);
        }
        __syncwarp();
        if (lane == 0) dupn[0] = 0;
      } else if (EV) {
        // binarized rows: every repeat becomes one event = the column of its class, in a deterministic
        // order (the list order depends on which lane lost the atomicOr): rank by (column, list index)
        const uint32_t nd = dupn[0];
        for (uint32_t i = lane; i < nd; i += 32) {
          const uint32_t e = ovf[i];
          const uint32_t k = e >> 26, c = e & 0x3FFFFFFu;
          uint32_t col = NOCOL;
          if ((bm[P.bm_off[k] + (c >> 5)] >> (c & 31)) & 1u) em.column(P.level_off[k] + c, col);   // else: dropped by the frozen list
          ovf[i] = col;
        }
        __syncwarp();
        uint32_t mine = 0;
        for (uint32_t i = lane; i < nd; i += 32) {
          const uint32_t key = ovf[i];
          if (key == NOCOL) continue;
          uint32_t rank = 0;
          for (uint32_t j = 0; j < nd; j++) {
            const uint32_t kj = ovf[j];
            rank += (kj < key || (kj == key && j < i)) ? 1u : 0u;
          }
          em.sid[P.stride - 1 - (int64_t)rank] = key;
          mine++;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
        em.ev = mine;
        __syncwarp();
        if (lane == 0) dupn[0] = 0;
      }
      for (int i = (int)lane * 4; i < P.bm_words; i += 128) *reinterpret_cast<uint4 *>(bm + i) = make_uint4(0, 0, 0, 0);
      __syncwarp();
    }

    // ---- sorted levels: one register sort of the canonical codes per level ---------------------------
    if (has_sort) {
      for (int k = P.s_lo; k <= N; k++) {
        auto key = [&](uint32_t f) -> uint32_t {
          uint32_t c = (f >> 4) >> (2 * (N - k));
          if (two && !single_sorted) c = min(c, kmer_op(c, k, op));
          return (int)(f & 15u) >= k ? c : SENT;
        };
        if constexpr (PK) {
          // 16-bit keys, two to a register (the low 16 bits of SENT are the sentinel 0xFFFF)
          uint32_t K2[E / 2];
#pragma unroll
          for (int q = 0; q < E / 2; q++) K2[q] = __byte_perm(key(FWL[q]), key(FWL[q + E / 2]), 0x5410);
          warp_sort16<E>(K2, lane);
          emit_sorted<E>(Keys16<E>{K2}, lane, tab, em, P.level_off[k], EV ? 1 : 0, P.stride);
        } else {
          uint32_t K[EE];
#pragma unroll
          for (int r = 0; r < EE; r++) K[r] = key(FWL[r]);
          warp_sort<EE>(K, lane);
          emit_sorted<EE>(Keys32<EE>{K}, lane, tab, em, P.level_off[k], EV ? 1 : 0, P.stride);
        }
      }
    }
    // row statistics (exact integers): what the step size and the fixed-point scale of the gradient need
    {
      unsigned long long sq = em.sq; uint32_t vm = em.vm;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        vm = max(vm, __shfl_xor_sync(0xffffffffu, vm, o));
      }
      if (lane == 0 && active) {
        P.rowcnt[row] = em.cursor;
        if (EV) P.rowdup[row] = em.ev;
        if (sq > P.stats[0]) atomicMax(P.stats, sq);
        if ((unsigned long long)vm > P.stats[1]) atomicMax(P.stats + 1, (unsigned long long)vm);
      }
    }
    if (mk && ++groups == next_check) {
      next_check *= 2;
      __syncthreads();
      flush_marks();
      __threadfence();
      __syncthreads();
      int missing = 0;
      for (int64_t i = threadIdx.x; i < P.nb_words; i += blockDim.x)
        missing |= (__ldg(P.nbx + i).x & ~*(volatile const uint32_t *)(P.bitmap + i)) != 0u;
      if (!__syncthreads_or(missing)) {
        mk = 0;
        if (threadIdx.x == 0) *(volatile uint32_t *)P.full = 1u;
      } else if (__syncthreads_or(threadIdx.x == 0 && *(volatile uint32_t *)P.full != 0u)) {
        mk = 0;
      }
    }
  }
  // flush the block's observed classes
  __syncthreads();
  if (mk) flush_marks();
}

template <int E, int OPT, bool EV, bool PK>
void launch_extract_op(const XParams &P) {
  // warps per block: the choice that keeps the most warps resident per SM (the block shares one
  // bitmap of observed classes, every warp brings its own working set)
  KL_CUDA(cudaFuncSetAttribute((extract_kernel<E, OPT, EV, PK>), cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  int best_wpb = 0, best_per_sm = 0;
  for (int wpb = ext_threads(E) / 32; wpb >= 1; wpb--) {
    size_t smem = ((size_t)P.obs_words + (size_t)wpb * P.warp_words) * sizeof(uint32_t);
    if (smem > (size_t)227 * 1024) continue;
    int per_sm = 0;
    KL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (extract_kernel<E, OPT, EV, PK>), 32 * wpb, smem));
    if (per_sm * wpb > best_per_sm * best_wpb) { best_wpb = wpb; best_per_sm = per_sm; }
  }
  KL_REQUIRE(best_wpb > 0, "sequence too long for the shared-memory working set of one warp");
  const int wpb = best_wpb;
  size_t smem = ((size_t)P.obs_words + (size_t)wpb * P.warp_words) * sizeof(uint32_t);
  int64_t blocks = (int64_t)ctx().sm_count * best_per_sm;
  int64_t need = (P.n - P.row0 + wpb - 1) / wpb;
  if (blocks > need) blocks = need;
  if (blocks < 1) blocks = 1;
  KL_LAUNCH((extract_kernel<E, OPT, EV, PK>), (unsigned)blocks, 32 * wpb, smem, P);
}

template <int E>
void launch_extract(const XParams &P) {
  if constexpr (E >= 2) {
    if (P.op == 1 && P.N <= PACK_MAX) {
      if (P.events) launch_extract_op<E, 1, true, true>(P);
      else launch_extract_op<E, 1, false, true>(P);
      return;
    }
  }
  if (P.events) {
    if (P.op == 1) launch_extract_op<E, 1, true, false>(P);
    else launch_extract_op<E, -1, true, false>(P);
  } else {
    if (P.op == 1) launch_extract_op<E, 1, false, false>(P);
    else launch_extract_op<E, -1, false, false>(P);
  }
}

#endif  // KL_EXTRACT_KERNEL_IMPL

}  // namespace xk
}  // namespace kl
