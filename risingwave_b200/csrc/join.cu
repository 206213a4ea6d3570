// join.cu -- streaming two-sided incremental HashJoin on sm_100a.
//
// Replaces (reference, Rust):
//   HashJoinExecutor::eq_join_oneside      src/stream/src/executor/hash_join.rs:925-1062
//   handle_match_rows / handle_match_row   hash_join.rs:1072-1357
//   JoinChunkBuilder (output-op rules)     src/stream/src/executor/join/builder.rs:158-316
//   JoinHashMap / JoinEntryState           src/stream/src/executor/join/hash_join.rs:169-830
//   join-type predicates                   src/stream/src/executor/join/mod.rs:103-169
//
// HBM layout per side:
//   record       : { u32 link (next row of the same key | DEAD bit), u32 null mask (bit c = column c
//                  is NULL), u32 seq (arrival order), u32 degree } + the row's columns packed at
//                  naturally aligned offsets; stride is a multiple of 16 B (Nexmark bid / auction:
//                  16 + 4*8 = 48 B).
//   hash index   : open addressing over BUCKETS, linear probing, power-of-two capacity, load <= 1/2;
//                  bucket = key word(s) | (live count << 32 | overflow head row) | ONE INLINE RECORD.
//                  Key64 + 48 B record = 64 B: a probe of a key with one row (bid -> auction) is ONE
//                  64-byte random access that returns key, count and the row; an insert into a
//                  fresh key is one 64-byte read-modify-write.  (Random 64 B transactions are what
//                  bounds this workload: measured 42 G random loads/s, 22 G random RMW/s on B200,
//                  profiles/r1_ubench_atomics.txt.)
//   overflow store: further rows of a key go to an append-only array of records chained through
//                  `link` from the bucket's head.
// Two execution paths:
//   * inner fast path (no degrees): ONE fused kernel per batch -- probe the other side, emit the
//     matches with tile-scan compaction, append the row to the own side; a second kernel applies
//     own-side deletes (it exits immediately when the batch has none).
//   * generic path (all 8 join types, degrees, append-only optimisation, mixed +/- on one key):
//     the batch is grouped by join key (scratch hash table + radix sort) and ONE thread walks each
//     key's rows in input order -- state of different keys is disjoint, so this is exactly the
//     reference's sequential semantics with the parallelism taken across keys.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <thread>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace rw {

#define J_EMPTY 0x8000000000000000ull
#define J_NIL 0x7fffffffu
#define J_DEAD 0x80000000u
#define J_MAX_OUT (2 * RW_MAX_COLS)
#define J_HDR 16
// bucket state word W (64 bit, follows the key word(s)):
//   bits  0..30  head of the overflow chain (row id, J_NIL = none)
//   bits 31..32  state of the inline record: 0 = never used, 1 = live, 2 = dead (reusable)
//   bits 33..63  live row count of the key (inline + overflow)
// Every own-side mutation of a bucket is ONE compare-and-swap on W (or one 128-bit CAS on key|W
// when the bucket is claimed): random atomics are the scarce resource (22 G/s on B200).
#define W_EMPTY 0x7fffffffull
#define W_COUNT_ONE (1ull << 33)
#define W_IL_LIVE (1ull << 31)
#define W_IL_DEAD (2ull << 31)
#define W_IL_MASK (3ull << 31)
__device__ __host__ __forceinline__ uint32_t W_head(uint64_t W) { return (uint32_t)(W & 0x7fffffffull); }
__device__ __host__ __forceinline__ uint32_t W_istate(uint64_t W) { return (uint32_t)((W >> 31) & 3ull); }
__device__ __host__ __forceinline__ uint32_t W_count(uint64_t W) { return (uint32_t)(W >> 33); }

#define JERR_DOUBLE_DELETE 1u
#define JERR_OUT_CAPACITY 2u
#define JERR_APPEND_ONLY_MULTI 4u
#define JERR_STORE_CAPACITY 8u
#define JERR_BAD_COUNT 16u

struct JoinPlanDev {
  int T;
  int n_keys;
  int key_col[2][RW_MAX_KEYS];
  int null_safe[RW_MAX_KEYS];
  int n_cols[2];
  int col_type[2][RW_MAX_COLS];
  int col_width[2][RW_MAX_COLS];
  int col_off[2][RW_MAX_COLS];  // byte offset of the column inside a record
  int stride[2];
  int bhdr;        // bytes of a bucket before its inline record: (KW + 1) * 8
  int bstride[2];  // bucket bytes: bhdr + stride, rounded up to 16
  int n_pk[2];
  int pk_col[2][RW_MAX_COLS];
  int n_out;
  int out_type[J_MAX_OUT];
  int out_width[J_MAX_OUT];
  int n_map[2];
  int map_in[2][J_MAX_OUT];
  int map_out[2][J_MAX_OUT];
  int need_degree[2];
  int append_only_optimize;
  int cond_cmp, cond_lhs, cond_rhs;
  int single_key, KW, SW;
  int strict;
};

struct JoinSideDev {
  uint8_t* recs;     // overflow record store
  uint8_t* buckets;  // hash index with inline records
  uint64_t cap;
  uint2* pools;      // per-warp row-id pools of the overflow store {next, end} (join_inner_q4_kernel)
  uint64_t rec_cap;  // records the overflow store can hold
  int stride;
  int bstride;
};

struct JoinStatus {
  unsigned long long out_rows;   // rows reserved in the output
  unsigned long long n_store;    // rows appended to the own side by this push
  unsigned long long n_del;      // visible delete rows seen by this push
  unsigned long long null_mask;  // bit k: output column k received a NULL; bit 63: invisible rows exist
  unsigned long long n_keys[2];  // distinct keys ever claimed per side
  unsigned int err;
  unsigned int pad;
  unsigned long long n_in;       // rows of the input chunk as the kernel saw them (device-resident row count)
  unsigned long long log_next[2];  // unified table: log ids handed out per side (copied from the device counters)
  unsigned long long n_dead[2];    // unified table: dead log records per side
  unsigned long long n_defer;      // unified table: bit 0 = the hot kernel deferred rows to the tail kernel, bit 1 = some are whole (sentinel-key) rows
};

struct JoinOutDev {
  uint8_t* ops;
  uint8_t* vis;                 // written by the generic path only
  void* col[J_MAX_OUT];
  uint8_t* valid[J_MAX_OUT];    // kept at 1; only NULLs are written (0)
  int64_t capacity;
  const uint8_t* heap[2];       // varlen payload: the sides' byte heaps (handles in varlen output columns point here)
};

// join/mod.rs:103-169
__device__ __host__ __forceinline__ bool jt_is_outer_side(int T, int S) { return T == RW_JOIN_FULL_OUTER || (T == RW_JOIN_LEFT_OUTER && S == 0) || (T == RW_JOIN_RIGHT_OUTER && S == 1); }
__device__ __host__ __forceinline__ bool jt_outer_side_null(int T, int S) { return T == RW_JOIN_FULL_OUTER || (T == RW_JOIN_LEFT_OUTER && S == 1) || (T == RW_JOIN_RIGHT_OUTER && S == 0); }
__device__ __host__ __forceinline__ bool jt_forward_exactly_once(int T, int S) { return ((T == RW_JOIN_LEFT_SEMI || T == RW_JOIN_LEFT_ANTI) && S == 0) || ((T == RW_JOIN_RIGHT_SEMI || T == RW_JOIN_RIGHT_ANTI) && S == 1); }
__device__ __host__ __forceinline__ bool jt_only_forward_matched_side(int T, int S) { return ((T == RW_JOIN_LEFT_SEMI || T == RW_JOIN_LEFT_ANTI) && S == 1) || ((T == RW_JOIN_RIGHT_SEMI || T == RW_JOIN_RIGHT_ANTI) && S == 0); }
__device__ __host__ __forceinline__ bool jt_is_semi(int T) { return T == RW_JOIN_LEFT_SEMI || T == RW_JOIN_RIGHT_SEMI; }
__device__ __host__ __forceinline__ bool jt_is_anti(int T) { return T == RW_JOIN_LEFT_ANTI || T == RW_JOIN_RIGHT_ANTI; }
__device__ __host__ __forceinline__ bool jt_forward_if_not_matched(int T, int S) { return (jt_is_anti(T) && jt_forward_exactly_once(T, S)) || jt_is_outer_side(T, S); }

// ------------------------------------------------------------------ records
struct RecHdr {
  uint32_t link, nullmask, seq, degree;
};
__device__ __forceinline__ uint8_t* rec_ptr(const JoinSideDev& s, uint32_t row) { return s.recs + (uint64_t)row * s.stride; }
__device__ __forceinline__ RecHdr* rec_hdr(const JoinSideDev& s, uint32_t row) { return (RecHdr*)rec_ptr(s, row); }

__device__ __forceinline__ uint64_t rec_key_word(const uint8_t* rec, int off, int width, int type) {
  ColRef cr;
  cr.data = rec + off;
  cr.valid_bits = nullptr;
  cr.valid_bytes = nullptr;
  cr.type = type;
  cr.width = width;
  return load_key_word(cr, 0);
}

__device__ __forceinline__ void prefetch_l2(const void* ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }

// copy one datum of `width` bytes
__device__ __forceinline__ void copy_bytes(void* dst, const void* src, int width) {
  switch (width) {
    case 1: *(uint8_t*)dst = *(const uint8_t*)src; break;
    case 2: *(uint16_t*)dst = *(const uint16_t*)src; break;
    case 4: *(uint32_t*)dst = *(const uint32_t*)src; break;
    case 8: *(uint64_t*)dst = *(const uint64_t*)src; break;
    default: *(ulonglong2*)dst = *(const ulonglong2*)src; break;
  }
}

// ------------------------------------------------------------------ key helpers
__device__ __forceinline__ bool chunk_key(const JoinPlanDev* p, int S, const DevChunk& ch, int64_t r, uint64_t* kw,
                                          uint32_t* nm) {
  uint32_t m = 0;
  bool never = false;
  for (int k = 0; k < p->n_keys; k++) {
    const ColRef& c = ch.cols[p->key_col[S][k]];
    if (col_is_null(c, r)) {
      m |= 1u << k;
      kw[k] = 0;
      if (!p->null_safe[k]) never = true;  // hash_join.rs:985-999
    } else {
      kw[k] = load_key_word(c, r);
    }
  }
  *nm = m;
  return never;
}

__device__ __forceinline__ uint64_t key_hash(const JoinPlanDev* p, const uint64_t* kw, uint32_t nm) {
  uint64_t h = 0x9e3779b97f4a7c15ull ^ nm;
  for (int k = 0; k < p->n_keys; k++) h = mix64(h ^ kw[k]) + 0x9e3779b97f4a7c15ull;
  return h;
}

// Key64 tables: the probe sequence of a key starts at an EVEN bucket, i.e. at a 128-byte aligned pair
// of 64-byte buckets, and continues bucket by bucket.  The quad-cooperative kernel fetches the whole
// pair with one 32-byte load per lane: the second probe of a collision costs no second trip to HBM.
__device__ __forceinline__ uint64_t home64(uint64_t key, uint64_t mask) { return mix64(key) & mask & ~1ull; }

// bucket = [key word(s)] [state word W] [inline record]
__device__ __forceinline__ uint8_t* bkt(const JoinSideDev& s, int64_t b) { return s.buckets + (uint64_t)b * s.bstride; }
__device__ __forceinline__ unsigned long long* bkt_W(const JoinSideDev& s, const JoinPlanDev* p, int64_t b) {
  return (unsigned long long*)(bkt(s, b) + p->KW * 8);
}
__device__ __forceinline__ uint8_t* bkt_inline(const JoinSideDev& s, const JoinPlanDev* p, int64_t b) { return bkt(s, b) + p->bhdr; }

// 128-bit compare-and-swap (sm_90+): claims an empty Key64 bucket, key and state word at once
__device__ __forceinline__ bool cas128(void* addr, ulonglong2 expect, ulonglong2 desired, ulonglong2* found) {
  unsigned long long o0, o1;
  asm volatile(
      "{\n .reg .b128 c, d, o;\n mov.b128 c, {%2, %3};\n mov.b128 d, {%4, %5};\n atom.global.cas.b128 o, [%6], c, d;\n mov.b128 {%0, %1}, o;\n}"
      : "=l"(o0), "=l"(o1)
      : "l"(expect.x), "l"(expect.y), "l"(desired.x), "l"(desired.y), "l"(addr)
      : "memory");
  found->x = o0;
  found->y = o1;
  return o0 == expect.x && o1 == expect.y;
}

// own-side append of one row to bucket b whose key is already claimed.  Returns true if the row got
// the bucket's inline record (caller writes it there); otherwise the caller supplies an overflow row
// id to `w_push_overflow`.  One CAS on W either way.
__device__ __forceinline__ bool w_claim_inline(unsigned long long* Wp) {
  unsigned long long cur = __ldcg(Wp);
  while (W_istate(cur) != 1u) {
    const unsigned long long nw = ((cur & ~W_IL_MASK) | W_IL_LIVE) + W_COUNT_ONE;
    const unsigned long long old = atomicCAS(Wp, cur, nw);
    if (old == cur) return true;
    cur = old;
  }
  return false;
}
__device__ __forceinline__ uint32_t w_push_overflow(unsigned long long* Wp, uint32_t row) {
  unsigned long long cur = __ldcg(Wp);
  while (true) {
    const unsigned long long nw = ((cur & ~0x7fffffffull) | (unsigned long long)row) + W_COUNT_ONE;
    const unsigned long long old = atomicCAS(Wp, cur, nw);
    if (old == cur) return W_head(cur);
    cur = old;
  }
}

// visit every live record of bucket b: the inline record first, then the overflow chain.
// `f(rec)` returns false to stop.
template <class F>
__device__ __forceinline__ void for_each_live(const JoinSideDev& s, const JoinPlanDev* p, int64_t b, F f) {
  // state / link words are read through L2 (ld.cg): another thread of the same kernel may change them
  const unsigned long long W = __ldcg(bkt_W(s, p, b));
  if (W_istate(W) == 1u) {
    if (!f(bkt_inline(s, p, b))) return;
  }
  uint32_t m = W_head(W);
  while (m != J_NIL) {
    uint8_t* rec = rec_ptr(s, m);
    const uint32_t lk = __ldcg(&((const RecHdr*)rec)->link);
    if (!(lk & J_DEAD)) {
      if (!f(rec)) return;
    }
    m = lk & 0x7fffffffu;
  }
}

// find the slot of a key (read-only). returns -1 if absent; *hc = (count << 32 | head) of the slot.
__device__ __forceinline__ int64_t js_find(const JoinSideDev& s, const JoinPlanDev* p, const uint64_t* kw, uint32_t nm,
                                           uint64_t* hc) {
  const uint64_t mask = s.cap - 1;
  if (p->single_key) {
    int64_t side = -1;
    if (nm) side = (int64_t)s.cap;                         // NULL key side slot (null-safe equality)
    else if (kw[0] == J_EMPTY) side = (int64_t)s.cap + 1;
    if (side >= 0) { *hc = __ldcg((const unsigned long long*)(bkt(s, side) + 8)); return side; }
    uint64_t idx = home64(kw[0], mask);
    while (true) {
      const ulonglong2 sl = __ldcg((const ulonglong2*)bkt(s, (int64_t)idx));  // key + head/count in one 128-bit load
      if (sl.x == kw[0]) { *hc = sl.y; return (int64_t)idx; }
      if (sl.x == J_EMPTY) return -1;
      idx = (idx + 1) & mask;
    }
  }
  uint64_t h = key_hash(p, kw, nm);
  uint64_t tag = (h & ~0xFFFFull) | ((uint64_t)nm << 8) | 1ull;
  uint64_t idx = (h >> 17) & mask;
  while (true) {
    const unsigned long long* ptr = (const unsigned long long*)bkt(s, (int64_t)idx);
    unsigned long long cur = __ldcg(ptr);
    if (cur == 0ull) return -1;
    if ((cur & ~2ull) == tag) {
      while (cur & 2ull) cur = *(volatile const unsigned long long*)ptr;
      bool eq = true;
      for (int k = 0; k < p->n_keys; k++) eq = eq && (__ldcg(ptr + 1 + k) == kw[k]);
      if (eq) { *hc = __ldcg(ptr + p->KW); return (int64_t)idx; }
    }
    idx = (idx + 1) & mask;
  }
}

__device__ __forceinline__ int64_t js_find_or_insert(const JoinSideDev& s, const JoinPlanDev* p, const uint64_t* kw,
                                                     uint32_t nm, bool* created) {
  const uint64_t mask = s.cap - 1;
  if (p->single_key) {
    if (nm) return (int64_t)s.cap;
    if (kw[0] == J_EMPTY) return (int64_t)s.cap + 1;
    uint64_t idx = home64(kw[0], mask);
    while (true) {
      unsigned long long* ptr = (unsigned long long*)bkt(s, (int64_t)idx);
      unsigned long long cur = __ldcg(ptr);
      if (cur == kw[0]) return (int64_t)idx;
      if (cur == J_EMPTY) {
        unsigned long long old = atomicCAS(ptr, (unsigned long long)J_EMPTY, (unsigned long long)kw[0]);
        if (old == J_EMPTY) { *created = true; return (int64_t)idx; }
        if (old == kw[0]) return (int64_t)idx;
      }
      idx = (idx + 1) & mask;
    }
  }
  uint64_t h = key_hash(p, kw, nm);
  uint64_t tag = (h & ~0xFFFFull) | ((uint64_t)nm << 8) | 1ull;
  uint64_t idx = (h >> 17) & mask;
  while (true) {
    unsigned long long* ptr = (unsigned long long*)bkt(s, (int64_t)idx);
    unsigned long long cur = __ldcg(ptr);
    if (cur == 0ull) {
      unsigned long long old = atomicCAS(ptr, 0ull, (unsigned long long)(tag | 2ull));
      if (old == 0ull) {
        for (int k = 0; k < p->n_keys; k++) __stcg(ptr + 1 + k, (unsigned long long)kw[k]);
        __threadfence();
        atomicExch(ptr, (unsigned long long)tag);
        *created = true;
        return (int64_t)idx;
      }
      cur = old;
    }
    if ((cur & ~2ull) == tag) {
      while (cur & 2ull) cur = *(volatile unsigned long long*)ptr;
      bool eq = true;
      for (int k = 0; k < p->n_keys; k++) eq = eq && (__ldcg(ptr + 1 + k) == kw[k]);
      if (eq) return (int64_t)idx;
    }
    idx = (idx + 1) & mask;
  }
}

__global__ void join_init_slots_kernel(uint8_t* buckets, uint64_t cap, int bstride, int KW, int single_key) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap + 2; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t* s = (uint64_t*)(buckets + i * bstride);
    s[0] = single_key ? J_EMPTY : 0ull;
    for (int k = 1; k < KW; k++) s[k] = 0;
    s[KW] = W_EMPTY;                                   // overflow head = NIL, inline never used, count = 0
  }
}

// ------------------------------------------------------------------ emission
// JoinStreamChunkBuilder::{append_row, append_row_update, append_row_matched}  builder.rs:84-148
// (ur < 0: update side NULL-padded; mrec == nullptr: matched side NULL-padded)
__device__ __forceinline__ void emit_row(const JoinOutDev& o, const JoinPlanDev* p, JoinStatus* st, int64_t orow, uint8_t op,
                                         int S, const DevChunk& ch, int64_t ur, const uint8_t* mrec) {
  o.ops[orow] = op;
  unsigned long long nullbits = 0;
  const int n_u = p->n_map[S], n_m = p->n_map[1 - S];
  for (int i = 0; i < n_u; i++) {
    const int ic = p->map_in[S][i], oc = p->map_out[S][i];
    bool nul = true;
    if (ur >= 0) {
      const ColRef& c = ch.cols[ic];
      nul = col_is_null(c, ur);
      if (!nul) copy_bytes((uint8_t*)o.col[oc] + orow * c.width, (const uint8_t*)c.data + ur * c.width, c.width);
    }
    if (nul) { o.valid[oc][orow] = 0; nullbits |= 1ull << oc; }
  }
  const uint32_t mnm = mrec ? ((const RecHdr*)mrec)->nullmask : 0xffffffffu;
  for (int i = 0; i < n_m; i++) {
    const int ic = p->map_in[1 - S][i], oc = p->map_out[1 - S][i];
    const bool nul = (mnm >> ic) & 1;
    if (!nul) {
      const int w = p->col_width[1 - S][ic];
      copy_bytes((uint8_t*)o.col[oc] + orow * w, mrec + p->col_off[1 - S][ic], w);
    } else {
      o.valid[oc][orow] = 0;
      nullbits |= 1ull << oc;
    }
  }
  if (nullbits) atomicOr(&st->null_mask, nullbits);
}

// check_join_condition (hash_join.rs:1362-1384) restricted to one integer comparison
__device__ __forceinline__ bool cond_ok(const JoinPlanDev* p, int S, const DevChunk& ch, int64_t ur, const uint8_t* mrec) {
  if (p->cond_cmp == RW_CMP_NONE) return true;
  const int nl = p->n_cols[0];
  int64_t v[2];
  const int idx[2] = {p->cond_lhs, p->cond_rhs};
  for (int t = 0; t < 2; t++) {
    const bool left = idx[t] < nl;
    const int local = left ? idx[t] : idx[t] - nl;
    const int side = left ? 0 : 1;
    if (side == S) {
      if (col_is_null(ch.cols[local], ur)) return false;
      v[t] = load_i64(ch.cols[local], ur);
    } else {
      if ((((const RecHdr*)mrec)->nullmask >> local) & 1) return false;
      v[t] = (int64_t)rec_key_word(mrec, p->col_off[side][local], p->col_width[side][local], p->col_type[side][local]);
    }
  }
  switch (p->cond_cmp) {
    case RW_CMP_LT: return v[0] < v[1];
    case RW_CMP_LE: return v[0] <= v[1];
    case RW_CMP_GT: return v[0] > v[1];
    case RW_CMP_GE: return v[0] >= v[1];
    case RW_CMP_EQ: return v[0] == v[1];
    default: return v[0] != v[1];
  }
}

// does the stored record carry the same pk as chunk row r ?  (pk = deduped_pk_indices; the join key
// is equal by construction: join/hash_join.rs:710-713)
__device__ __forceinline__ bool pk_equal(const JoinPlanDev* p, int S, const uint8_t* rec, const DevChunk& ch, int64_t r) {
  const uint32_t nmask = ((const RecHdr*)rec)->nullmask;
  for (int i = 0; i < p->n_pk[S]; i++) {
    const int c = p->pk_col[S][i];
    const bool n1 = (nmask >> c) & 1, n2 = col_is_null(ch.cols[c], r);
    if (n1 != n2) return false;
    if (n1) continue;
    const int w = p->col_width[S][c];
    if (w == 16) {
      const uint64_t* a = (const uint64_t*)(rec + p->col_off[S][c]);
      const uint64_t* b = (const uint64_t*)ch.cols[c].data + r * 2;
      if (a[0] != b[0] || a[1] != b[1]) return false;
    } else if (rec_key_word(rec, p->col_off[S][c], w, p->col_type[S][c]) != load_key_word(ch.cols[c], r)) {
      return false;
    }
  }
  return true;
}

// write chunk row r into the record `row`
__device__ __forceinline__ void rec_write(const JoinPlanDev* p, int S, uint8_t* rec, const DevChunk& ch, int64_t r,
                                          uint32_t link, uint32_t seq, uint32_t degree) {
  uint32_t nm = 0;
  for (int c = 0; c < p->n_cols[S]; c++) {
    const ColRef& cr = ch.cols[c];
    if (col_is_null(cr, r)) nm |= 1u << c;
    else copy_bytes(rec + p->col_off[S][c], (const uint8_t*)cr.data + r * cr.width, cr.width);
  }
  uint4 h;
  h.x = link;
  h.y = nm;
  h.z = seq;
  h.w = degree;
  *(uint4*)rec = h;
}

// =============================================================================== generic path
struct JoinScratch {
  uint64_t* sortkey;      // [n]  gid << 32 | row
  uint64_t* sortkey_alt;  // [n]
  uint64_t* packed;       // [n]  store_flag << 40 | out bound
  uint64_t* offs;         // [n]  exclusive scan of packed
  int64_t* match_slot;    // [n]
  int32_t* gtable;        // [gcap] batch-local key -> representative row
  uint64_t gcap;
};

// G1: per row -- never-match rule, probe of the other side's index, output bound, batch-local group id
__global__ void __launch_bounds__(256) join_prepare_kernel(const JoinPlanDev* __restrict__ p, int S, DevChunk ch,
                                                            JoinSideDev other, JoinScratch sc) {
  const int T = p->T;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < ch.n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint8_t op = ch.ops[r];
    if (!row_visible(ch, r, op)) {
      sc.sortkey[r] = 0xFFFFFFFF00000000ull | (uint64_t)r;
      sc.packed[r] = 0;
      sc.match_slot[r] = -1;
      continue;
    }
    uint64_t kw[RW_MAX_KEYS];
    uint32_t nm;
    const bool never = chunk_key(p, S, ch, r, kw, &nm);
    const bool ins = (op == RW_OP_INSERT || op == RW_OP_UPDATE_INSERT);
    uint32_t gid;
    int64_t ms = -1;
    uint64_t bound;
    if (never) {
      gid = 0x80000000u | (uint32_t)r;  // singleton group
      bound = jt_forward_if_not_matched(T, S) ? 1 : 0;
    } else {
      uint64_t hc = 0;
      ms = js_find(other, p, kw, nm, &hc);
      const uint64_t m = ms >= 0 ? W_count(hc) : 0;
      uint64_t per_match;
      if (T == RW_JOIN_INNER) per_match = 1;
      else if (jt_is_semi(T) || jt_is_anti(T)) per_match = jt_forward_exactly_once(T, S) ? 0 : 1;
      else per_match = jt_outer_side_null(T, S) ? 2 : 1;
      const uint64_t fwd = (jt_forward_if_not_matched(T, S) || (jt_is_semi(T) && jt_forward_exactly_once(T, S))) ? 1 : 0;
      bound = per_match * m + fwd;
      // batch-local grouping: claim a scratch slot with this row as representative, or join the
      // group whose representative carries an equal key
      const uint64_t gmask = sc.gcap - 1;
      uint64_t gi = key_hash(p, kw, nm) & gmask;
      while (true) {
        int cur = sc.gtable[gi];
        if (cur < 0) {
          int old = atomicCAS(sc.gtable + gi, -1, (int)r);
          if (old < 0) break;
          cur = old;
        }
        uint64_t kw2[RW_MAX_KEYS];
        uint32_t nm2;
        chunk_key(p, S, ch, cur, kw2, &nm2);
        bool eq = (nm2 == nm);
        for (int k = 0; k < p->n_keys; k++) eq = eq && (kw2[k] == kw[k]);
        if (eq) break;
        gi = (gi + 1) & gmask;
      }
      gid = (uint32_t)gi;
    }
    sc.sortkey[r] = ((uint64_t)gid << 32) | (uint64_t)r;
    sc.packed[r] = ((uint64_t)((ins && !never) ? 1 : 0) << 40) | bound;
    sc.match_slot[r] = ms;
  }
}

__global__ void join_totals_kernel(const uint64_t* packed, const uint64_t* offs, int64_t n, JoinStatus* st) {
  if (n > 0) {
    uint64_t tot = offs[n - 1] + packed[n - 1];
    st->out_rows = tot & ((1ull << 40) - 1);
    st->n_store = tot >> 40;
  } else {
    st->out_rows = 0;
    st->n_store = 0;
  }
}

__global__ void fill_i32_kernel(int32_t* p, uint64_t n, int32_t v) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}

// G4: one thread per join key of the batch, rows in input order (exact sequential semantics per key)
__global__ void __launch_bounds__(128) join_serial_kernel(const JoinPlanDev* __restrict__ p, int S, DevChunk ch,
                                                           JoinSideDev own, JoinSideDev other, JoinScratch sc,
                                                           const uint64_t* __restrict__ sorted, JoinOutDev o,
                                                           JoinStatus* st, uint32_t store_base, uint32_t seq_base,
                                                           int64_t out_base) {
  const int T = p->T;
  const bool fwd_once = jt_forward_exactly_once(T, S);
  const bool fwd_unmatched = jt_forward_if_not_matched(T, S);
  const bool fwd_matched = jt_is_semi(T) && fwd_once;
  const bool only_matched = jt_only_forward_matched_side(T, S);
  const bool side_null = jt_outer_side_null(T, S);
  const bool other_deg = p->need_degree[1 - S] != 0;
  const bool own_deg = p->need_degree[S] != 0;
  unsigned int new_keys = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < ch.n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t sk = sorted[i];
    const uint32_t gid = (uint32_t)(sk >> 32);
    if (gid == 0xFFFFFFFFu) continue;                               // invisible rows
    if (i > 0 && (uint32_t)(sorted[i - 1] >> 32) == gid) continue;  // not a group start
    int64_t own_slot = -2;  // lazily resolved
    for (int64_t j = i; j < ch.n && (uint32_t)(sorted[j] >> 32) == gid; j++) {
      const int64_t r = (int64_t)(sorted[j] & 0xFFFFFFFFull);
      const uint8_t op = ch.ops[r];
      const bool ins = (op == RW_OP_INSERT || op == RW_OP_UPDATE_INSERT);
      const uint8_t jop = ins ? RW_OP_INSERT : RW_OP_DELETE;
      const uint64_t pk = sc.packed[r];
      const int64_t bound = (int64_t)(pk & ((1ull << 40) - 1));
      const int64_t obase = out_base + (int64_t)(sc.offs[r] & ((1ull << 40) - 1));
      const uint32_t store_row = store_base + (uint32_t)(sc.offs[r] >> 40);
      int64_t w = 0;  // rows written so far for r
      const bool room = obase + bound <= o.capacity;
      if (!room) atomicOr(&st->err, JERR_OUT_CAPACITY);
      if (gid & 0x80000000u) {  // CacheResult::NeverMatch (hash_join.rs:1126-1135): forwarded, never stored
        if (fwd_unmatched && room) emit_row(o, p, st, obase + w++, jop, S, ch, r, nullptr);
        continue;
      }
      const int64_t ms = sc.match_slot[r];
      uint32_t degree = 0;
      uint8_t* ao_rec = nullptr;
      if (ms >= 0) {
        for_each_live(other, p, ms, [&](uint8_t* mrec) -> bool {
          RecHdr* mh = (RecHdr*)mrec;
          if (cond_ok(p, S, ch, r, mrec)) {
            degree++;
            uint32_t md = other_deg ? mh->degree : 0;
            if (ins && !fwd_once && room) {  // with_match_on_insert (builder.rs:184-231): m.degree BEFORE the increment
              if (jt_is_anti(T)) { if (md == 0 && only_matched) emit_row(o, p, st, obase + w++, RW_OP_DELETE, S, ch, -1, mrec); }
              else if (jt_is_semi(T)) { if (md == 0 && only_matched) emit_row(o, p, st, obase + w++, RW_OP_INSERT, S, ch, -1, mrec); }
              else if (md == 0 && side_null) {
                emit_row(o, p, st, obase + w++, RW_OP_DELETE, S, ch, -1, mrec);
                emit_row(o, p, st, obase + w++, RW_OP_INSERT, S, ch, r, mrec);
              } else emit_row(o, p, st, obase + w++, RW_OP_INSERT, S, ch, r, mrec);
            }
            if (other_deg) { md = ins ? md + 1 : md - 1; mh->degree = md; }  // update_degree (join/hash_join.rs:355-380)
            if (!ins && !fwd_once && room) {  // with_match_on_delete (builder.rs:233-284): m.degree AFTER the decrement
              if (jt_is_anti(T)) { if (md == 0 && only_matched) emit_row(o, p, st, obase + w++, RW_OP_INSERT, S, ch, -1, mrec); }
              else if (jt_is_semi(T)) { if (md == 0 && only_matched) emit_row(o, p, st, obase + w++, RW_OP_DELETE, S, ch, -1, mrec); }
              else if (md == 0 && side_null) {
                emit_row(o, p, st, obase + w++, RW_OP_DELETE, S, ch, r, mrec);
                emit_row(o, p, st, obase + w++, RW_OP_INSERT, S, ch, -1, mrec);
              } else emit_row(o, p, st, obase + w++, RW_OP_DELETE, S, ch, r, mrec);
            }
          }
          if (p->append_only_optimize) {  // hash_join.rs:1339-1345 (regardless of the condition)
            if (ao_rec) atomicOr(&st->err, JERR_APPEND_ONLY_MULTI);
            ao_rec = mrec;
          }
          return true;
        });
      }
      // forward rows depending on join types (hash_join.rs:1198-1210)
      if (room) {
        if (degree == 0) { if (fwd_unmatched) emit_row(o, p, st, obase + w++, jop, S, ch, r, nullptr); }
        else if (fwd_matched) emit_row(o, p, st, obase + w++, jop, S, ch, r, nullptr);
        if (w < bound) atomicOr(&st->null_mask, 1ull << 63);
        for (; w < bound; w++) {  // unused reserved rows become invisible holes
          o.ops[obase + w] = RW_OP_INSERT;
          o.vis[obase + w] = 0;
        }
      }
      // append-only optimisation (hash_join.rs:1222-1228): drop the matched row, do not store u
      if (p->append_only_optimize && ao_rec) {
        unsigned long long* Wo = bkt_W(other, p, ms);
        if (ao_rec == bkt_inline(other, p, ms)) *Wo = ((*Wo & ~W_IL_MASK) | W_IL_DEAD) - W_COUNT_ONE;
        else { ((RecHdr*)ao_rec)->link |= J_DEAD; *Wo -= W_COUNT_ONE; }
        continue;
      }
      // own-side state (hash_join.rs:1230-1242; JoinHashMap::insert / delete join/hash_join.rs:591-681)
      if (own_slot == -2) {
        uint64_t kw[RW_MAX_KEYS];
        uint32_t nm;
        uint64_t hc;
        chunk_key(p, S, ch, r, kw, &nm);
        bool created = false;
        own_slot = ins ? js_find_or_insert(own, p, kw, nm, &created) : js_find(own, p, kw, nm, &hc);
        if (created) new_keys++;
      }
      if (ins) {
        unsigned long long* Wp = bkt_W(own, p, own_slot);
        const unsigned long long W = *Wp;
        if (W_istate(W) != 1u) {  // the bucket's inline record is free: the row lives in the bucket
          rec_write(p, S, bkt_inline(own, p, own_slot), ch, r, 0u, seq_base + (uint32_t)r, own_deg ? degree : 0);
          *Wp = ((W & ~W_IL_MASK) | W_IL_LIVE) + W_COUNT_ONE;
        } else {
          rec_write(p, S, rec_ptr(own, store_row), ch, r, W_head(W), seq_base + (uint32_t)r, own_deg ? degree : 0);
          *Wp = ((W & ~0x7fffffffull) | (unsigned long long)store_row) + W_COUNT_ONE;
        }
      } else {
        bool found = false;
        if (own_slot >= 0) {
          unsigned long long* Wp = bkt_W(own, p, own_slot);
          uint8_t* irec = bkt_inline(own, p, own_slot);
          for_each_live(own, p, own_slot, [&](uint8_t* mrec) -> bool {
            if (!pk_equal(p, S, mrec, ch, r)) return true;
            if (mrec == irec) *Wp = ((*Wp & ~W_IL_MASK) | W_IL_DEAD) - W_COUNT_ONE;
            else { ((RecHdr*)mrec)->link |= J_DEAD; *Wp -= W_COUNT_ONE; }
            found = true;
            return false;
          });
        } else {
          own_slot = -2;  // the key may be created by a later insert of this group
        }
        if (!found && p->strict) atomicOr(&st->err, JERR_DOUBLE_DELETE);
      }
    }
  }
  if (new_keys) atomicAdd(&st->n_keys[S], (unsigned long long)new_keys);
}

// =============================================================================== inner fast path
// One fused kernel per batch.  A tile is JF_BLOCK * JF_R consecutive rows, thread t owning rows
// t, t + JF_BLOCK, ... (coalesced column loads; JF_R independent slot probes and record gathers in
// flight per thread).  Phase 1 probes the other side's index (128-bit slot loads).  Phase 2 is a
// tile-wide scan (warp shuffles + one shared-memory pass) of the match counts and of the own-side
// store flags; one atomicAdd per tile reserves the output range / the record ids.  Phase 3 walks
// the matched chains and emits (warp-coalesced column stores).  Phase 4 appends the rows to the own
// side (record write, slot claim, head exchange).  With `PROBE_ONLY` phases 1-3 run alone: the
// host uses it to redo the emission after an output-capacity overflow (phases 1-3 never touch
// operator state, and phase 4 only touches the OWN side, so the redo is exact).
#define JF_BLOCK 256
#define JF_R 1
template <bool PROBE_ONLY>
__global__ void __launch_bounds__(JF_BLOCK, 8) join_inner_fused_kernel(const JoinPlanDev* __restrict__ p, int S, DevChunk ch,
                                                                        JoinSideDev own, JoinSideDev other, JoinOutDev o,
                                                                        JoinStatus* st, uint32_t store_base, uint64_t seq_base) {
  __shared__ unsigned long long s_cnt[JF_R][JF_BLOCK / 32];
  __shared__ unsigned int s_sto[JF_R][JF_BLOCK / 32];
  __shared__ unsigned long long s_out_base;
  __shared__ unsigned int s_store_base;
  const int lane = lane_id(), wid = threadIdx.x >> 5;
  const int64_t tile_rows = (int64_t)JF_BLOCK * JF_R;
  const int64_t n_tiles = (ch.n + tile_rows - 1) / tile_rows;
  unsigned int new_keys = 0, n_del = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t base = tile * tile_rows;
    uint32_t head[JF_R], cnt[JF_R];
    uint8_t op[JF_R];
    bool store[JF_R];
    // ---- phase 1: probe the other side's index
#pragma unroll
    for (int k = 0; k < JF_R; k++) {
      const int64_t r = base + (int64_t)k * JF_BLOCK + threadIdx.x;
      head[k] = J_NIL; cnt[k] = 0; op[k] = 0; store[k] = false;
      if (r < ch.n) {
        op[k] = ch.ops[r];
        if (row_visible(ch, r, op[k])) {
          uint64_t kw[RW_MAX_KEYS];
          uint32_t nm;
          const bool ins = (op[k] == RW_OP_INSERT || op[k] == RW_OP_UPDATE_INSERT);
          if (!chunk_key(p, S, ch, r, kw, &nm)) {
            store[k] = ins;
            if (!ins) n_del++;
            if (!PROBE_ONLY && ins && p->single_key && !nm)  // the own-side bucket is claimed in phase 4: start fetching it
              prefetch_l2(bkt(own, (int64_t)home64(kw[0], own.cap - 1)));
            uint64_t hc;
            const int64_t b = js_find(other, p, kw, nm, &hc);
            if (b >= 0) {
              head[k] = (uint32_t)b;  // bucket index of the matched key
              cnt[k] = W_count(hc);
              const uint32_t oh = W_head(hc);
              if (cnt[k] > 1 && oh != J_NIL) prefetch_l2(rec_ptr(other, oh));
            }
          }
        } else {
          op[k] = 0;
        }
      }
    }
    if (p->cond_cmp != RW_CMP_NONE) {  // a non-equi condition filters matches: count by walking
#pragma unroll
      for (int k = 0; k < JF_R; k++) {
        if (cnt[k] == 0) continue;
        const int64_t r = base + (int64_t)k * JF_BLOCK + threadIdx.x;
        uint32_t c = 0;
        for_each_live(other, p, (int64_t)head[k], [&](uint8_t* mrec) -> bool {
          if (cond_ok(p, S, ch, r, mrec)) c++;
          return true;
        });
        cnt[k] = c;
      }
    }
    // ---- phase 2: tile scan of the match counts (row order = k-major), one reservation per tile
    unsigned long long incl[JF_R];
#pragma unroll
    for (int k = 0; k < JF_R; k++) {
      unsigned long long v = cnt[k];
      for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
      }
      incl[k] = v;
      if (lane == 31) s_cnt[k][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long run = 0;
      for (int k = 0; k < JF_R; k++)
        for (int w = 0; w < JF_BLOCK / 32; w++) { unsigned long long t = s_cnt[k][w]; s_cnt[k][w] = run; run += t; }
      s_out_base = run ? atomicAdd(&st->out_rows, run) : 0ull;
    }
    __syncthreads();
    // ---- phase 3: emit
#pragma unroll
    for (int k = 0; k < JF_R; k++) {
      if (cnt[k] == 0) continue;
      const int64_t r = base + (int64_t)k * JF_BLOCK + threadIdx.x;
      int64_t pos = (int64_t)(s_out_base + s_cnt[k][wid] + incl[k] - cnt[k]);
      if (pos + cnt[k] > o.capacity) { atomicOr(&st->err, JERR_OUT_CAPACITY); continue; }
      const uint8_t oop = (op[k] == RW_OP_INSERT || op[k] == RW_OP_UPDATE_INSERT) ? RW_OP_INSERT : RW_OP_DELETE;
      uint32_t left = cnt[k];
      for_each_live(other, p, (int64_t)head[k], [&](uint8_t* mrec) -> bool {
        if (cond_ok(p, S, ch, r, mrec)) { emit_row(o, p, st, pos++, oop, S, ch, r, mrec); left--; }
        return left != 0;
      });
    }
    // ---- phase 4: append to the own side.  4a: claim the bucket and try its inline record (one
    // 64 B read-modify-write for a key's first row); 4b: rows that lost go to the overflow store,
    // whose ids are reserved with one atomicAdd per tile.
    if (!PROBE_ONLY) {
      int64_t own_b[JF_R];
      bool overflow[JF_R];
#pragma unroll
      for (int k = 0; k < JF_R; k++) {
        overflow[k] = false;
        own_b[k] = -1;
        if (!store[k]) continue;
        const int64_t r = base + (int64_t)k * JF_BLOCK + threadIdx.x;
        uint64_t kw[RW_MAX_KEYS];
        uint32_t nm;
        chunk_key(p, S, ch, r, kw, &nm);
        bool created = false;
        const int64_t b = js_find_or_insert(own, p, kw, nm, &created);
        if (created) new_keys++;
        own_b[k] = b;
        // (inner join: no degrees -- the degree word carries the high half of the 64-bit arrival number)
        if (w_claim_inline(bkt_W(own, p, b)))
          rec_write(p, S, bkt_inline(own, p, b), ch, r, 0u, (uint32_t)(seq_base + (uint64_t)r), (uint32_t)((seq_base + (uint64_t)r) >> 32));
        else overflow[k] = true;
      }
      unsigned int sincl[JF_R];
#pragma unroll
      for (int k = 0; k < JF_R; k++) {
        unsigned int sv = overflow[k] ? 1u : 0u;
        for (int d = 1; d < 32; d <<= 1) {
          unsigned int ts = __shfl_up_sync(0xffffffffu, sv, d);
          if (lane >= d) sv += ts;
        }
        sincl[k] = sv;
        if (lane == 31) s_sto[k][wid] = sv;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned int srun = 0;
        for (int k = 0; k < JF_R; k++)
          for (int w = 0; w < JF_BLOCK / 32; w++) { unsigned int ts = s_sto[k][w]; s_sto[k][w] = srun; srun += ts; }
        s_store_base = srun ? (unsigned int)atomicAdd(&st->n_store, (unsigned long long)srun) : 0u;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < JF_R; k++) {
        if (!overflow[k]) continue;
        const int64_t r = base + (int64_t)k * JF_BLOCK + threadIdx.x;
        const uint32_t row = store_base + s_store_base + s_sto[k][wid] + sincl[k] - 1;
        const uint32_t old = w_push_overflow(bkt_W(own, p, own_b[k]), row);
        rec_write(p, S, rec_ptr(own, row), ch, r, old, (uint32_t)(seq_base + (uint64_t)r), (uint32_t)((seq_base + (uint64_t)r) >> 32));
      }
    }
    __syncthreads();
  }
  if (!PROBE_ONLY) {
    for (int d = 16; d > 0; d >>= 1) {
      new_keys += __shfl_xor_sync(0xffffffffu, new_keys, d);
      n_del += __shfl_xor_sync(0xffffffffu, n_del, d);
    }
    if (lane == 0 && new_keys) atomicAdd(&st->n_keys[S], (unsigned long long)new_keys);
    if (lane == 0 && n_del) atomicAdd(&st->n_del, (unsigned long long)n_del);
  }
}

// ------------------------------------------------------------------ Key64 / all-8-byte-columns specialisation
// The generic fused kernel pays ~1800 warp instructions per 32 rows on runtime-typed loops whose
// loads depend on each other (plan -> column pointer -> datum -> store).  Nexmark-shaped joins have a
// single 8-byte key and only 8-byte columns, for which everything can be straight-line code:
//   * the WHOLE other-side bucket (key | head/count | inline record) is fetched with 16-byte loads
//     issued together, before the key is even compared (one HBM round trip per probe);
//   * the update row's columns are loaded once (coalesced) and reused for emission and for the
//     own-side record;
//   * the own-side record is written with 16-byte stores into the bucket's inline record.
// Rows it cannot take (key == EMPTY sentinel, matched record with NULLs, keys with several rows)
// fall through to the same helpers the generic kernel uses.
#define W8_MAXC 8
#define Q4_MAX_GRID (148 * 8)  // blocks of JF_BLOCK threads; one row-id pool per warp
struct W8Plan {
  int n_u, n_m;            // columns of the update / matched side (all 8 bytes wide)
  int key_col;             // key column of the update side
  int8_t u_out[W8_MAXC];   // output column fed by update column c (-1 = not projected)
  int8_t m_out[W8_MAXC];   // output column fed by matched column c
};

// the overflow chain only (the inline record was handled by the caller)
template <class F>
__device__ __forceinline__ void for_each_overflow_live(const JoinSideDev& s, uint32_t head, F f) {
  uint32_t m = head & 0x7fffffffu;
  while (m != J_NIL) {
    uint8_t* rec = rec_ptr(s, m);
    const uint32_t lk = __ldcg(&((const RecHdr*)rec)->link);
    if (!(lk & J_DEAD)) {
      if (!f(rec)) return;
    }
    m = lk & 0x7fffffffu;
  }
}

// Output convention of this kernel ("positional"): the first match of input row r is written to
// output row out_base + r -- no scan, no block barrier, warps never wait for each other; a row
// without a match (or an invisible input row) leaves an invisible output row.  Further matches of a
// row (keys with several rows on the other side) are appended behind the n positional rows with a
// warp-aggregated atomicAdd.  A StreamChunk with invisible rows is a legal chunk; for the
// bid -> auction probe (every bid matches exactly one auction) the output is dense and in input order.
// JoinStatus.out_rows counts the EXTRA rows; JoinStatus.pad = 1 when some row matched;
// null_mask bit 63 = some positional row is invisible.
template <bool PROBE_ONLY>
__global__ void __launch_bounds__(JF_BLOCK, 4) join_inner_w8p_kernel(const JoinPlanDev* __restrict__ p, W8Plan w, int S, DevChunk ch,
                                                                      JoinSideDev own, JoinSideDev other, JoinOutDev o, JoinStatus* st,
                                                                      uint32_t store_base, uint64_t seq_base, int64_t out_base) {
  const int lane = lane_id();
  const uint64_t omask = other.cap - 1, wmask = own.cap - 1;
  unsigned int new_keys = 0, n_del = 0;
  bool any_match = false, any_hole = false;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < ch.n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint8_t op = ch.ops[r];
    if (op == 0) { o.vis[out_base + r] = 0; any_hole = true; continue; }
    const bool ins = (op == RW_OP_INSERT || op == RW_OP_UPDATE_INSERT);
    if (!ins) n_del++;
    uint64_t uv[W8_MAXC], mv[W8_MAXC];
#pragma unroll
    for (int c = 0; c < W8_MAXC; c++)
      if (c < w.n_u) uv[c] = __ldg((const unsigned long long*)ch.cols[c].data + r);
    const uint64_t key = __ldg((const unsigned long long*)ch.cols[w.key_col].data + r);
    bool fast = key != J_EMPTY, ilive = false;
    uint32_t cnt = 0, ohead = J_NIL;
    int64_t ob = -1;
    // ---- probe: the whole 64-byte bucket of the other side in one round trip
    if (fast) {
      if (!PROBE_ONLY && ins) prefetch_l2(bkt(own, (int64_t)home64(key, wmask)));
      uint64_t idx = home64(key, omask);
      while (true) {
        const uint8_t* bp = bkt(other, (int64_t)idx);
        const ulonglong2 h0 = __ldcg((const ulonglong2*)bp);          // key | head/count
        const uint4 mh = __ldcg((const uint4*)(bp + 16));             // inline record header
        ulonglong2 m2[W8_MAXC / 2];
#pragma unroll
        for (int c = 0; c < W8_MAXC / 2; c++)
          if (2 * c < w.n_m) m2[c] = __ldcg((const ulonglong2*)(bp + 32 + 16 * c));
        if (h0.x == key) {
          ob = (int64_t)idx;
          cnt = W_count(h0.y);
          ohead = W_head(h0.y);
          ilive = W_istate(h0.y) == 1u;
          if (ilive && mh.y != 0) { ilive = false; fast = false; }  // NULLs in the matched record: generic emission
#pragma unroll
          for (int c = 0; c < W8_MAXC / 2; c++) { mv[2 * c] = m2[c].x; mv[2 * c + 1] = m2[c].y; }
          break;
        }
        if (h0.x == J_EMPTY) break;
        idx = (idx + 1) & omask;
      }
    } else {
      uint64_t kw[1] = {key}, hc = 0;
      ob = js_find(other, p, kw, 0, &hc);
      if (ob >= 0) { cnt = W_count(hc); ohead = W_head(hc); }
    }
    // ---- emit
    const uint8_t oop = ins ? RW_OP_INSERT : RW_OP_DELETE;
    if (cnt == 0) {
      o.vis[out_base + r] = 0;
      any_hole = true;
    } else {
      any_match = true;
      o.vis[out_base + r] = 1;
      int64_t pos = out_base + r;
      uint32_t left = cnt;
      // extra matches go behind the positional rows
      int64_t xpos = 0;
      if (cnt > 1) {
        const unsigned m = __activemask();
        // lanes converged here may need different amounts: reserve individually but with one atomic per lane group
        xpos = out_base + ch.n + (int64_t)atomicAdd(&st->out_rows, (unsigned long long)(cnt - 1));
        (void)m;
        if (xpos + (cnt - 1) > o.capacity) { atomicOr(&st->err, JERR_OUT_CAPACITY); left = 1; }
      }
      bool first = true;
      auto place = [&]() -> int64_t {
        if (first) { first = false; return pos; }
        o.vis[xpos] = 1;
        return xpos++;
      };
      if (fast && ilive) {
        const int64_t q = place();
        o.ops[q] = oop;
#pragma unroll
        for (int c = 0; c < W8_MAXC; c++)
          if (c < w.n_u && w.u_out[c] >= 0) ((uint64_t*)o.col[w.u_out[c]])[q] = uv[c];
#pragma unroll
        for (int c = 0; c < W8_MAXC; c++)
          if (c < w.n_m && w.m_out[c] >= 0) ((uint64_t*)o.col[w.m_out[c]])[q] = mv[c];
        left--;
        if (left)
          for_each_overflow_live(other, ohead, [&](uint8_t* mrec) -> bool {
            emit_row(o, p, st, place(), oop, S, ch, r, mrec);
            return --left != 0;
          });
      } else {
        for_each_live(other, p, ob, [&](uint8_t* mrec) -> bool {
          emit_row(o, p, st, place(), oop, S, ch, r, mrec);
          return --left != 0;
        });
      }
    }
    // ---- append to the own side: bucket claim, then the bucket's inline record or the overflow store
    if (!PROBE_ONLY && ins) {
      // one 128-bit CAS claims an empty bucket together with its inline record; an existing key
      // costs one 64-bit CAS on its state word
      bool created = false, inline_won = false;
      int64_t wb;
      if (key != J_EMPTY) {
        uint64_t idx = home64(key, wmask);
        while (true) {
          ulonglong2* bp = (ulonglong2*)bkt(own, (int64_t)idx);
          ulonglong2 cur = __ldcg(bp);
          if (cur.x == J_EMPTY) {
            ulonglong2 want, found;
            want.x = key;
            want.y = (W_EMPTY | W_IL_LIVE) + W_COUNT_ONE;
            if (cas128(bp, cur, want, &found)) { created = true; inline_won = true; break; }
            cur = found;
          }
          if (cur.x == key) break;
          if (cur.x != J_EMPTY) idx = (idx + 1) & wmask;
        }
        wb = (int64_t)idx;
      } else {
        uint64_t kw[1] = {key};
        wb = js_find_or_insert(own, p, kw, 0, &created);
      }
      if (created) new_keys++;
      unsigned long long* Wp = bkt_W(own, p, wb);
      if (!inline_won) inline_won = w_claim_inline(Wp);
      uint8_t* rec;
      uint32_t link = 0u;
      if (inline_won) {
        rec = bkt_inline(own, p, wb);
      } else {
        // overflow row: id from a warp-aggregated reservation
        const unsigned m = __activemask();
        const int leader = __ffs(m) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(&st->n_store, (unsigned long long)__popc(m));
        base = __shfl_sync(m, base, leader);
        const uint32_t row = store_base + (uint32_t)base + __popc(m & ((1u << lane) - 1));
        link = w_push_overflow(Wp, row);
        rec = rec_ptr(own, row);
      }
      uint4 hh;
      hh.x = link; hh.y = 0u; hh.z = (uint32_t)(seq_base + (uint64_t)r); hh.w = (uint32_t)((seq_base + (uint64_t)r) >> 32);
      *(uint4*)rec = hh;
#pragma unroll
      for (int c = 0; c < W8_MAXC / 2; c++)
        if (2 * c < w.n_u) {
          ulonglong2 v;
          v.x = uv[2 * c];
          v.y = (2 * c + 1 < w.n_u) ? uv[2 * c + 1] : 0ull;
          *(ulonglong2*)(rec + 16 + 16 * c) = v;
        }
    }
  }
  unsigned long long flags = (any_hole ? (1ull << 63) : 0ull);
  const bool warp_match = __any_sync(0xffffffffu, any_match);
  for (int d = 16; d > 0; d >>= 1) {
    flags |= __shfl_xor_sync(0xffffffffu, flags, d);
    new_keys += __shfl_xor_sync(0xffffffffu, new_keys, d);
    n_del += __shfl_xor_sync(0xffffffffu, n_del, d);
  }
  if (lane == 0) {
    if (flags && (__ldcg(&st->null_mask) & flags) != flags) atomicOr(&st->null_mask, flags);
    if (warp_match && __ldcg(&st->pad) == 0u) st->pad = 1u;  // "some row matched" (plain store: all writers store 1)
    if (!PROBE_ONLY && new_keys) atomicAdd(&st->n_keys[S], (unsigned long long)new_keys);
    if (!PROBE_ONLY && n_del) atomicAdd(&st->n_del, (unsigned long long)n_del);
  }
}

// a chunk whose row count lives on the device (e.g. the output of the exchange): clamp the capacity
__device__ __forceinline__ int64_t chunk_rows(const DevChunk& ch, JoinStatus* st, bool report) {
  if (!ch.n_dev) return ch.n;
  const int64_t n = *ch.n_dev;
  if (n < 0 || n > ch.n) {
    if (report) atomicOr(&st->err, JERR_BAD_COUNT);
    return 0;
  }
  if (report) st->n_in = (unsigned long long)n;
  return n;
}

// ------------------------------------------------------------------ quad-cooperative Key64 kernel (<= 4 + 4 columns)
// tools/ubench_bucket.cu (profiles/r1_ubench_bucket.txt): what a random bucket access costs is the
// number of memory INSTRUCTIONS that touch the line, not its bytes -- one thread reading a 64-byte
// bucket with 4 x LDG.128 takes 90 us per 2^20 rows, four lanes reading 16 bytes each in ONE
// instruction take 25 us (the price of a single 16-byte load); a record written with three 16-byte
// stores costs 89 us cold but ~17 us once the claiming CAS has pulled the line into L2.
// So a row is owned by a QUAD of lanes and a warp works on 8 rows:
//   lane q of the quad loads piece q of the other side's bucket   [key|W] [rec hdr] [col0,col1] [col2,col3]
//   lanes 0,1 hold the update row's columns (0,1) / (2,3) and write them to the output,
//   lanes 2,3 hold the matched columns and write those -- two store instructions emit the row;
//   lane 0 claims the own-side bucket with one speculative 128-bit CAS issued BEFORE the probe
//   resolves (both random accesses are in flight together); lanes 1..3 then write the record
//   (header, columns) with one 16-byte store each into the line the CAS just brought in.
// Rows the quad cannot finish this way (sentinel key, several matches, match not in the inline
// record, NULLs in the matched record) are finished by lane 0 with the generic helpers.
// Output convention: positional, exactly as join_inner_w8p_kernel.
struct U256 { uint64_t a, b, c, d; };
// one 32-byte load (LDG.E.256, sm_100), L2 only
__device__ __forceinline__ U256 ld256_cg(const void* ptr) {
  U256 v;
  asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v.a), "=l"(v.b), "=l"(v.c), "=l"(v.d) : "l"(ptr));
  return v;
}
__device__ __forceinline__ uint64_t shfl64m(unsigned mask, uint64_t v, int src) {
  return (uint64_t)__shfl_sync(mask, (unsigned long long)v, src);
}

template <bool PROBE_ONLY, int MINB>
__global__ void __launch_bounds__(JF_BLOCK, MINB) join_inner_q4_kernel(const JoinPlanDev* __restrict__ p, W8Plan w, int S, DevChunk ch,
                                                                     JoinSideDev own, JoinSideDev other, JoinOutDev o, JoinStatus* st,
                                                                     uint32_t store_base, uint64_t seq_base, int64_t out_base, uint32_t pool_chunk) {
  // (kept in a register: writing ch.n would force a local-memory copy of the whole parameter struct)
  const int64_t n_rows = chunk_rows(ch, st, blockIdx.x == 0 && threadIdx.x == 0);
  const int lane = lane_id(), q = lane & 3, qlead = lane & ~3;
  // Overflow row ids come from a per-warp pool that persists across launches: one atomicAdd on the
  // shared counter hands a warp `pool_chunk` ids.  (One atomicAdd per 8 rows on that single address
  // was measured at +0.3 ms per 2^20 rows -- same-address atomics serialise in one L2 slice.)
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  uint32_t pool_next = 0, pool_end = 0;
  if (!PROBE_ONLY) {
    const uint2 pl = own.pools[warp_global];
    pool_next = pl.x;
    pool_end = pl.y;
  }
  const uint32_t pool_next0 = pool_next, pool_end0 = pool_end;
  const uint64_t omask = other.cap - 1, wmask = own.cap - 1;
  unsigned int new_keys = 0, n_del = 0;
  bool any_match = false, any_hole = false;
  // column roles of this lane
  const int ca = 2 * (q & 1), cb = ca + 1;
  const unsigned long long* pa = ca < w.n_u ? (const unsigned long long*)ch.cols[ca].data : nullptr;
  const unsigned long long* pb = cb < w.n_u ? (const unsigned long long*)ch.cols[cb].data : nullptr;
  const unsigned long long* pk = (const unsigned long long*)ch.cols[w.key_col].data;
  int oc0, oc1;
  if (q < 2) {
    oc0 = ca < w.n_u ? w.u_out[ca] : -1;
    oc1 = cb < w.n_u ? w.u_out[cb] : -1;
  } else {
    oc0 = ca < w.n_m ? w.m_out[ca] : -1;
    oc1 = cb < w.n_m ? w.m_out[cb] : -1;
  }
  uint64_t* po0 = oc0 >= 0 ? (uint64_t*)o.col[oc0] : nullptr;
  uint64_t* po1 = oc1 >= 0 ? (uint64_t*)o.col[oc1] : nullptr;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t groups = (n_rows + 7) >> 3;
  ulonglong2 cas_empty, cas_want;
  cas_empty.x = J_EMPTY;
  cas_empty.y = W_EMPTY;
  cas_want.y = (W_EMPTY | W_IL_LIVE) + W_COUNT_ONE;
  // All shuffles use the full-warp mask and sit in warp-uniform control flow: a shuffle with a
  // per-quad mask splits the warp into eight separately issued groups (measured: 2.8x slower).
  // Software pipeline: the (sequential) column loads of the warp's NEXT group are issued right after
  // the random accesses of the current one, so they are out of the dependent chain
  // ops -> key -> bucket / CAS -> chain CAS that bounds this latency-bound kernel.
  uint8_t n_op = 0;
  uint64_t n_key = J_EMPTY, n_va = 0ull, n_vb = 0ull;
  auto fetch = [&](int64_t g2) {
    const int64_t r2 = g2 * 8 + (lane >> 2);
    n_op = 0;
    if (g2 < groups && r2 < n_rows) {
      n_op = ch.ops[r2];
      n_key = __ldg(pk + r2);
      if (pa) n_va = __ldg(pa + r2);
      if (pb) n_vb = __ldg(pb + r2);
    }
  };
  fetch(warp_global);
  for (int64_t g = warp_global; g < groups; g += nwarps) {
    const int64_t r = g * 8 + (lane >> 2);
    const bool in = r < n_rows;
    const uint8_t op = n_op;
    const uint64_t key = n_key, va = n_va, vb = n_vb;
    const int64_t pos = out_base + r;
    const bool act = op != 0;
    if (in && !act) {  // invisible input row
      if (q == 0) o.vis[pos] = 0;
      any_hole = true;
    }
    const bool ins = act && (op == RW_OP_INSERT || op == RW_OP_UPDATE_INSERT);
    if (act && !ins && q == 0) n_del++;
    const bool keyok = act && key != J_EMPTY;
    const uint64_t hsh = mix64(key);
    // ---- own side: speculative claim, in flight together with the probe
    const bool do_ins = !PROBE_ONLY && ins;
    // (the result `cf` is only looked at after the probe: comparing it here would make the warp
    // wait for the atomic before the probe load is even issued)
    ulonglong2 cf;
    cf.x = 0; cf.y = 0;
    uint64_t widx = hsh & wmask & ~1ull;
    if (do_ins && keyok && q == 0) {
      cas_want.x = key;
      cas128(own.buckets + widx * 64, cas_empty, cas_want, &cf);
    }
    fetch(g + nwarps);
    // ---- probe: the quad fetches the 128-byte bucket PAIR, one 32-byte load per lane
    //   lane 0: A.key A.W A.hdr   lane 1: A.cols 0..3   lane 2: B.key B.W B.hdr   lane 3: B.cols 0..3
    // the warp iterates until its longest probe sequence ends (finished quads idle)
    bool found = false, need = keyok;
    uint64_t idx = hsh & omask & ~1ull;
    int sel = 0;  // 0: matched bucket A, 2: bucket B
    U256 pv;
    pv.a = 0; pv.b = 0; pv.c = 0; pv.d = 0;
    while (__any_sync(0xffffffffu, need)) {
      if (need) pv = ld256_cg(other.buckets + idx * 64 + 32 * q);
      const uint64_t kA = shfl64m(0xffffffffu, pv.a, qlead), kB = shfl64m(0xffffffffu, pv.a, qlead + 2);
      if (need) {
        if (kA == key) { found = true; sel = 0; need = false; }
        else if (kB == key) { found = true; sel = 2; need = false; }
        else if (kA == J_EMPTY || kB == J_EMPTY) need = false;  // an empty bucket ends the probe sequence
        else idx = (idx + 2) & omask;
      }
    }
    const int hl = qlead + sel;  // lane holding key | W | record header of the matched bucket
    const uint64_t W = shfl64m(0xffffffffu, pv.b, hl);
    const uint32_t mnull = __shfl_sync(0xffffffffu, (uint32_t)(pv.c >> 32), hl);  // rec hdr: link | nullmask
    // matched columns: lane 2 writes (0,1), lane 3 writes (2,3)
    const uint64_t m0 = shfl64m(0xffffffffu, pv.a, hl + 1), m1 = shfl64m(0xffffffffu, pv.b, hl + 1);
    const uint64_t m2 = shfl64m(0xffffffffu, pv.c, hl + 1), m3 = shfl64m(0xffffffffu, pv.d, hl + 1);
    const uint64_t ma = q == 3 ? m2 : m0, mb = q == 3 ? m3 : m1;
    // ---- emit
    uint32_t cnt = found ? W_count(W) : 0u;
    if (cnt == 1u && W_istate(W) == 1u && mnull == 0u) {
      any_match = true;
      if (q == 0) o.ops[pos] = ins ? RW_OP_INSERT : RW_OP_DELETE;
      if (q == 1) o.vis[pos] = 1;
      if (po0) po0[pos] = q < 2 ? va : ma;
      if (po1) po1[pos] = q < 2 ? vb : mb;
    } else if (act && q == 0) {
      int64_t ob = found ? (int64_t)idx + (sel >> 1) : -1;
      if (!keyok) {
        uint64_t kw[1] = {key}, hc = 0;
        ob = js_find(other, p, kw, 0, &hc);
        cnt = ob >= 0 ? W_count(hc) : 0u;
      }
      if (cnt == 0u) {
        o.vis[pos] = 0;
        any_hole = true;
      } else {
        any_match = true;
        o.vis[pos] = 1;
        const uint8_t oop = ins ? RW_OP_INSERT : RW_OP_DELETE;
        uint32_t left = cnt;
        int64_t xpos = 0;
        if (cnt > 1u) {
          xpos = out_base + n_rows + (int64_t)atomicAdd(&st->out_rows, (unsigned long long)(cnt - 1));
          if (xpos + (cnt - 1) > o.capacity) { atomicOr(&st->err, JERR_OUT_CAPACITY); left = 1; }
        }
        bool first = true;
        for_each_live(other, p, ob, [&](uint8_t* mrec) -> bool {
          int64_t at = pos;
          if (!first) { o.vis[xpos] = 1; at = xpos++; }
          first = false;
          emit_row(o, p, st, at, oop, S, ch, r, mrec);
          return --left != 0;
        });
      }
    }
    // ---- append to the own side
    uint64_t recp = 0;
    uint32_t link = 0u;
    bool need_ovf = false;
    unsigned long long Wcur = 0ull;
    unsigned long long* Wp = nullptr;
    if (do_ins && q == 0) {
      bool created = false, inline_won = false;
      if (keyok) {
        while (true) {
          if (cf.x == J_EMPTY && cf.y == W_EMPTY) { created = true; inline_won = true; break; }  // the CAS took the bucket
          if (cf.x == key) { Wcur = cf.y; break; }
          widx = (widx + 1) & wmask;  // bucket held by another key
          cas128(own.buckets + widx * 64, cas_empty, cas_want, &cf);
        }
        Wp = (unsigned long long*)(own.buckets + widx * 64 + 8);
      } else {
        uint64_t kw[1] = {key};
        widx = (uint64_t)js_find_or_insert(own, p, kw, 0, &created);
        Wp = (unsigned long long*)(own.buckets + widx * 64 + 8);
        Wcur = __ldcg(Wp);
      }
      if (created) new_keys++;
      if (!inline_won) {
        while (W_istate(Wcur) != 1u) {  // the inline record is free (never used, or its row was deleted)
          const unsigned long long nw = ((Wcur & ~W_IL_MASK) | W_IL_LIVE) + W_COUNT_ONE;
          const unsigned long long old = atomicCAS(Wp, Wcur, nw);
          if (old == Wcur) { inline_won = true; break; }
          Wcur = old;
        }
      }
      if (inline_won) recp = (uint64_t)(own.buckets + widx * 64 + 16);
      else need_ovf = true;
    }
    if (!PROBE_ONLY) {
      const unsigned bal = __ballot_sync(0xffffffffu, need_ovf);
      if (bal) {  // warp-uniform: ids for the rows that go to the overflow store
        const uint32_t k = __popc(bal), left = pool_end - pool_next;
        uint32_t nb = 0;
        if (left < k) {  // refill; the remainder of the old chunk is used up first
          if (lane == 0) {
            nb = store_base + (uint32_t)atomicAdd(&st->n_store, (unsigned long long)pool_chunk);
            if ((uint64_t)nb + pool_chunk > own.rec_cap) { atomicOr(&st->err, JERR_STORE_CAPACITY); nb = 0xffffffffu; }
          }
          nb = __shfl_sync(0xffffffffu, nb, 0);
        }
        const uint32_t i = __popc(bal & ((1u << lane) - 1u));
        const uint32_t row = i < left ? pool_next + i : nb + (i - left);
        const bool bad = left < k && nb == 0xffffffffu;
        if (left < k) {
          pool_next = bad ? 0u : nb + (k - left);
          pool_end = bad ? 0u : nb + pool_chunk;
        } else {
          pool_next += k;
        }
        if (need_ovf && !(bad && i >= left)) {
          while (true) {  // one CAS pushes the row on the key's chain
            const unsigned long long nw = ((Wcur & ~0x7fffffffull) | (unsigned long long)row) + W_COUNT_ONE;
            const unsigned long long old = atomicCAS(Wp, Wcur, nw);
            if (old == Wcur) break;
            Wcur = old;
          }
          link = W_head(Wcur);
          recp = (uint64_t)rec_ptr(own, row);
        }
      }
      recp = shfl64m(0xffffffffu, recp, qlead);
      link = __shfl_sync(0xffffffffu, link, qlead);
      if (do_ins && q != 0 && recp) {
        ulonglong2 v;
        if (q == 1) {  // RecHdr {link, nullmask = 0, seq, degree = 0}
          v.x = (unsigned long long)link;
          v.y = (unsigned long long)(seq_base + (uint64_t)r);  // {seq, degree} = the 64-bit arrival number
        } else {       // lane 2: columns 0,1   lane 3: columns 2,3
          v.x = va;
          v.y = vb;
        }
        *(ulonglong2*)(recp + 16 * (q - 1)) = v;
      }
    }
  }
  if (!PROBE_ONLY && lane == 0 && (pool_next != pool_next0 || pool_end != pool_end0)) own.pools[warp_global] = make_uint2(pool_next, pool_end);
  unsigned long long flags = (any_hole ? (1ull << 63) : 0ull);
  const bool warp_match = __any_sync(0xffffffffu, any_match);
  for (int d = 16; d > 0; d >>= 1) {
    flags |= __shfl_xor_sync(0xffffffffu, flags, d);
    new_keys += __shfl_xor_sync(0xffffffffu, new_keys, d);
    n_del += __shfl_xor_sync(0xffffffffu, n_del, d);
  }
  if (lane == 0) {
    if (flags && (__ldcg(&st->null_mask) & flags) != flags) atomicOr(&st->null_mask, flags);
    if (warp_match && __ldcg(&st->pad) == 0u) st->pad = 1u;
    if (!PROBE_ONLY && new_keys) atomicAdd(&st->n_keys[S], (unsigned long long)new_keys);
    if (!PROBE_ONLY && n_del) atomicAdd(&st->n_del, (unsigned long long)n_del);
  }
}

// own-side deletes of the fast path (after the fused kernel; exits at once when the batch has none).
// Sequential rule: the delete at chunk position r removes the live record with equal pk that
// arrived most recently BEFORE r (64-bit arrival numbers, see the kernel).
// status block -> pinned host memory (UVA), tagged so the host can tell a fresh copy from a stale one;
// then the per-push counters are zeroed for the next push (reset bit 0: n_store / n_del / null_mask,
// bit 1: out_rows / pad of the positional kernels).
__device__ __forceinline__ void join_status_publish(JoinStatus* st, JoinStatus* host, unsigned long long tag, int reset) {
  const JoinStatus s = *st;
  *host = s;
  *(unsigned long long*)(host + 1) = tag;
  __threadfence_system();
  if (reset & 1) { st->n_store = 0ull; st->n_del = 0ull; st->null_mask = 0ull; st->n_defer = 0ull; }
  if (reset & 2) { st->out_rows = 0ull; st->pad = 0u; st->n_in = 0ull; }
}

__global__ void __launch_bounds__(256) join_inner_delete_kernel(const JoinPlanDev* __restrict__ p, int S, DevChunk ch,
                                                                 JoinSideDev own, JoinStatus* st, uint64_t seq_base,
                                                                 JoinStatus* status_host, unsigned long long tag, int reset) {
  const int64_t n_rows = chunk_rows(ch, st, false);
  if (*(volatile unsigned long long*)&st->n_del == 0ull) {
    // nothing to delete (the usual case): this launch doubles as the status read-back
    if (status_host && blockIdx.x == 0 && threadIdx.x == 0) join_status_publish(st, status_host, tag, reset);
    return;
  }
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    const uint8_t op = ch.ops[r];
    if (!row_visible(ch, r, op) || !(op == RW_OP_DELETE || op == RW_OP_UPDATE_DELETE)) continue;
    uint64_t kw[RW_MAX_KEYS];
    uint32_t nm;
    if (chunk_key(p, S, ch, r, kw, &nm)) continue;  // never-match rows were never stored
    uint64_t hc;
    const int64_t slot = js_find(own, p, kw, nm, &hc);
    bool found = false;
    if (slot >= 0) {
      while (!found) {
        // 64-bit arrival numbers ({seq, degree} of the record header; the inner join keeps no degrees): rows this
        // very chunk inserted at positions >= r are excluded, every other live pk-equal row arrived before r; the
        // newest wins.  (A 32-bit wrap-aware age, the first version, lost deletes after 2^31 rows.)
        uint8_t* best = nullptr;
        uint64_t best_seq = 0;
        for_each_live(own, p, slot, [&](uint8_t* mrec) -> bool {
          const RecHdr* mh = (const RecHdr*)mrec;
          const uint64_t sq = (uint64_t)mh->seq | ((uint64_t)mh->degree << 32);
          const bool later = sq >= seq_base + (uint64_t)r && sq < seq_base + (uint64_t)n_rows;
          if (!later && (!best || sq > best_seq) && pk_equal(p, S, mrec, ch, r)) {
            best = mrec;
            best_seq = sq;
          }
          return true;
        });
        if (!best) break;
        unsigned long long* Wp = bkt_W(own, p, slot);
        if (best == bkt_inline(own, p, slot)) {
          unsigned long long cur = __ldcg(Wp);
          while (W_istate(cur) == 1u) {  // live -> dead, count - 1, in one CAS
            const unsigned long long old = atomicCAS(Wp, cur, ((cur & ~W_IL_MASK) | W_IL_DEAD) - W_COUNT_ONE);
            if (old == cur) { found = true; break; }
            cur = old;
          }
        } else {
          const uint32_t old = atomicOr(&((RecHdr*)best)->link, J_DEAD);
          if (!(old & J_DEAD)) {
            atomicAdd(Wp, 0ull - W_COUNT_ONE);
            found = true;
          }
        }
      }
    }
    if (!found && p->strict) atomicOr(&st->err, JERR_DOUBLE_DELETE);
  }
}

// ------------------------------------------------------------------ growth helpers
__global__ void join_rehash_kernel(const uint8_t* ob, uint64_t ocap, uint8_t* nb, uint64_t ncap, int bstride, int KW,
                                   int single_key, int n_keys) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < ocap + 2; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t* s = (const uint64_t*)(ob + i * bstride);
    uint64_t dst;
    if (i >= ocap) {
      dst = ncap + (i - ocap);
    } else {
      const uint64_t w0 = s[0];
      if (single_key ? (w0 == J_EMPTY) : (w0 == 0)) continue;
      const uint64_t mask = ncap - 1;
      uint64_t idx;
      if (single_key) {
        idx = home64(w0, mask);
        while (atomicCAS((unsigned long long*)(nb + idx * bstride), (unsigned long long)J_EMPTY, (unsigned long long)w0) != J_EMPTY) idx = (idx + 1) & mask;
      } else {
        uint32_t nm = (uint32_t)((w0 >> 8) & 0xff);
        uint64_t h = 0x9e3779b97f4a7c15ull ^ nm;
        for (int k = 0; k < n_keys; k++) h = mix64(h ^ s[1 + k]) + 0x9e3779b97f4a7c15ull;
        idx = (h >> 17) & mask;
        while (atomicCAS((unsigned long long*)(nb + idx * bstride), 0ull, (unsigned long long)w0) != 0ull) idx = (idx + 1) & mask;
      }
      dst = idx;
    }
    uint64_t* d = (uint64_t*)(nb + dst * bstride);
    for (int k = (i >= ocap ? 0 : 1); k < bstride / 8; k++) d[k] = s[k];  // rest of the header + the inline record
  }
}

static inline size_t align_up_j(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace rw

#include "join_uni.cuh"

namespace rw {
// varlen payload handles (see "varlen payload columns" below)
#define VH_LEN_MAX ((1u << 22) - 1u)
__device__ __host__ __forceinline__ uint64_t vh_make(int heap, uint32_t len, uint64_t off) { return ((uint64_t)heap << 62) | ((uint64_t)len << 40) | off; }
__device__ __host__ __forceinline__ uint64_t vh_off(uint64_t h) { return h & ((1ull << 40) - 1); }
__device__ __host__ __forceinline__ uint32_t vh_len(uint64_t h) { return (uint32_t)((h >> 40) & VH_LEN_MAX); }
__device__ __host__ __forceinline__ int vh_heap(uint64_t h) { return (int)(h >> 62); }
}  // namespace rw

// =============================================================================== eliminate_adjacent_noop_update
// StreamChunk::eliminate_adjacent_noop_update (src/common/src/array/stream_chunk.rs:331-392), applied by
// JoinChunkBuilder::post_process to every chunk the join yields: walking the visible rows of a chunk, a Delete-then-
// Insert (or Insert-then-Delete) pair of EQUAL rows is hidden, and the walk restarts after the pair.  In a maximal run
// of consecutive such pairs  e1 e2 e3 ...  (edges between neighbouring visible rows) the greedy walk therefore takes
// e1, e3, e5 ...: an edge is taken iff the number of eligible edges directly before it is even -- which every row can
// decide for itself.  Chunks are the `chunk_size`-row cuts of the device output (rwgpu_out::finalize cuts there).
namespace rw {
struct NoopScratch {
  int32_t* nxt;   // next visible row inside the chunk, -1 if none
  int32_t* prv;   // previous visible row inside the chunk, -1 if none
  uint8_t* elig;  // the edge (row, nxt[row]) is an eliminable pair
};

// (null_cols: bit k = output column k holds NULLs in this call -- the validity bytes of the others are all 1 and are not
// read; columns are compared from the last one: in a retraction pair the update side's payload differs first)
__device__ __forceinline__ bool out_rows_equal(const JoinOutDev& o, const JoinPlanDev* p, int64_t a, int64_t b, unsigned long long null_cols) {
  for (int k = p->n_out - 1; k >= 0; k--) {
    if ((null_cols >> k) & 1ull) {
      const bool na = o.valid[k][a] == 0, nb = o.valid[k][b] == 0;
      if (na != nb) return false;
      if (na) continue;
    }
    const int w = p->out_width[k];
    const uint8_t* x = (const uint8_t*)o.col[k] + a * w;
    const uint8_t* y = (const uint8_t*)o.col[k] + b * w;
    if (p->out_type[k] == RW_T_VARCHAR || p->out_type[k] == RW_T_BYTEA) {  // handles: compare the bytes they name
      const uint64_t hx = *(const uint64_t*)x, hy = *(const uint64_t*)y;
      if (hx == hy) continue;
      const uint32_t len = vh_len(hx);
      if (len != vh_len(hy)) return false;
      const uint8_t* bx = o.heap[vh_heap(hx) - 1] + vh_off(hx);
      const uint8_t* by = o.heap[vh_heap(hy) - 1] + vh_off(hy);
      for (uint32_t i = 0; i < len; i++) if (bx[i] != by[i]) return false;
      continue;
    }
    switch (w) {
      case 1: if (*x != *y) return false; break;
      case 2: if (*(const uint16_t*)x != *(const uint16_t*)y) return false; break;
      case 4: if (*(const uint32_t*)x != *(const uint32_t*)y) return false; break;
      case 8: if (*(const uint64_t*)x != *(const uint64_t*)y) return false; break;
      default: if (((const uint64_t*)x)[0] != ((const uint64_t*)y)[0] || ((const uint64_t*)x)[1] != ((const uint64_t*)y)[1]) return false; break;
    }
  }
  return true;
}

// flag[0] = something was hidden, flag[1] = some edge is eligible (the two passes behind this one exit at once otherwise)
__global__ void noop_edges_kernel(JoinOutDev o, const JoinPlanDev* __restrict__ p, int64_t n, int chunk_size, NoopScratch sc, unsigned long long null_cols,
                                  unsigned int* flag) {
  bool any = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    sc.elig[i] = 0;
    sc.nxt[i] = -1;
    sc.prv[i] = -1;
    if (!o.vis[i]) continue;
    int64_t end = (i / chunk_size + 1) * (int64_t)chunk_size;
    if (end > n) end = n;
    int64_t j = i + 1;
    while (j < end && !o.vis[j]) j++;
    if (j >= end) continue;
    sc.nxt[i] = (int32_t)j;
    const uint8_t a = o.ops[i], b = o.ops[j];
    const bool a_del = a == RW_OP_DELETE || a == RW_OP_UPDATE_DELETE, b_del = b == RW_OP_DELETE || b == RW_OP_UPDATE_DELETE;
    if (a_del != b_del && out_rows_equal(o, p, i, j, null_cols)) { sc.elig[i] = 1; any = true; }
  }
  if (any) flag[1] = 1u;
}
__global__ void noop_prev_kernel(int64_t n, int chunk_size, NoopScratch sc, const unsigned int* flag) {
  if (*(volatile const unsigned int*)(flag + 1) == 0u) return;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t j = sc.nxt[i];
    if (j >= 0) sc.prv[j] = (int32_t)i;
  }
}
__global__ void noop_take_kernel(JoinOutDev o, int64_t n, NoopScratch sc, unsigned int* hid) {
  if (*(volatile unsigned int*)(hid + 1) == 0u) return;
  bool any = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!sc.elig[i]) continue;
    int before = 0;  // eligible edges directly before this one
    for (int32_t q = sc.prv[i]; q >= 0 && sc.elig[q]; q = sc.prv[q]) before++;
    if (before & 1) continue;
    o.vis[i] = 0;
    o.vis[sc.nxt[i]] = 0;
    any = true;
  }
  if (any) *hid = 1u;
}
// "Normalize update pairs that became partially invisible" (stream_chunk.rs:377-389)
__global__ void noop_normalize_kernel(JoinOutDev o, int64_t n, int chunk_size, const unsigned int* hid) {
  if (*(volatile const unsigned int*)hid == 0u) return;  // nothing was hidden: no pair lost a half
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x) {
    if ((i + 1) % chunk_size == 0) continue;  // the pair would straddle two chunks
    if (o.ops[i] == RW_OP_UPDATE_DELETE && o.ops[i + 1] == RW_OP_UPDATE_INSERT) {
      const bool dv = o.vis[i] != 0, iv = o.vis[i + 1] != 0;
      if (dv && !iv) o.ops[i] = RW_OP_DELETE;
      else if (!dv && iv) o.ops[i + 1] = RW_OP_INSERT;
    }
  }
}
}  // namespace rw

// =============================================================================== varlen payload columns
// A varchar / bytea column (BytesArray{offset, bitmap, data}, src/common/src/array/bytes_array.rs:30-34) travels through
// the join as PAYLOAD.  When a chunk enters, the bytes of its visible rows are INTERNED into the side's byte heap in
// HBM and the column becomes a column of 8-byte handles
//     bits 0..39 heap offset | bits 40..61 length (< 4 MiB) | bits 62..63 heap id (1 = left, 2 = right)
// which every join kernel treats like any other 8-byte column (stored in buckets / logs, gathered into the output).
// When a result leaves, the handles of a varlen output column are turned back into offsets[n + 1] + bytes: lengths ->
// exclusive scan -> gather.  The heap is append-only (a deleted row's bytes stay until the operator is rebuilt).
namespace rw {

// bytes: base pointer such that value r is bytes[offs[r] .. offs[r+1])
__global__ void __launch_bounds__(256) varlen_intern_kernel(const uint8_t* bytes, const uint32_t* offs, const uint8_t* ops, const uint64_t* vis_bits,
                                                            const uint64_t* valid_bits, int64_t n, uint8_t* heap, unsigned long long* heap_next,
                                                            uint64_t heap_cap, int heap_id, uint64_t* handles, unsigned int* err) {
  const int lane = threadIdx.x & 31;
  for (int64_t r0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) & ~31ll; r0 < n; r0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = r0 + lane;
    uint32_t len = 0, o0 = 0;
    bool live = false;
    if (r < n) {
      live = ops[r] != 0 && bit_get(vis_bits, r) && bit_get(valid_bits, r);
      if (live) { o0 = offs[r]; len = offs[r + 1] - o0; }
    }
    if (len > VH_LEN_MAX) { atomicOr(err, 1u); len = 0; live = false; }
    const uint32_t need = (len + 7u) & ~7u;
    uint32_t incl = need;
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned long long base = 0;
    if (lane == 0 && total) base = atomicAdd(heap_next, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (r >= n) continue;
    uint64_t hd = 0;
    if (live) {
      const unsigned long long at = base + (incl - need);
      if (at + need > heap_cap) { atomicOr(err, 2u); }
      else {
        for (uint32_t i = 0; i < len; i++) heap[at + i] = bytes[o0 + i];
        hd = vh_make(heap_id, len, at);
      }
    }
    handles[r] = hd;
  }
}

__global__ void varlen_lens_kernel(const uint64_t* handles, const uint8_t* vis, const uint8_t* valid, int64_t n, uint32_t* lens) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const bool live = (!vis || vis[r]) && (!valid || valid[r]);
    lens[r] = live ? vh_len(handles[r]) : 0u;
  }
}
__global__ void varlen_total_kernel(const uint32_t* lens, uint32_t* offs, int64_t n) { offs[n] = n ? offs[n - 1] + lens[n - 1] : 0u; }
__global__ void varlen_gather_kernel(const uint64_t* handles, const uint32_t* offs, int64_t n, const uint8_t* heap_l, const uint8_t* heap_r, uint8_t* out) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t len = offs[r + 1] - offs[r];
    if (!len) continue;
    const uint64_t hd = handles[r];
    const uint8_t* src = (vh_heap(hd) == 1 ? heap_l : heap_r) + vh_off(hd);
    uint8_t* dst = out + offs[r];
    for (uint32_t i = 0; i < len; i++) dst[i] = src[i];
  }
}
}  // namespace rw

// =============================================================================== state persistence
// The join's persistent state is, per side, the set of stored input rows (the reference writes every stored row to the
// side's StateTable, JoinHashMap::insert join/hash_join.rs:591-625, pk = join key | deduped input pk; degrees live in a
// second table and are a function of the two row sets).  The snapshot kernels walk every key's chain and emit the live
// rows in the side's INPUT schema; restore replays them as inserts with the output discarded -- the incremental
// algorithm itself re-derives the degrees.
namespace rw {
struct SnapOut {
  void* col[RW_MAX_COLS];
  uint8_t* valid[RW_MAX_COLS];
  unsigned long long* n_rows;
  unsigned int* has_null;
  int64_t capacity;
};

__device__ __forceinline__ void snap_emit_uni(const SnapOut& o, int n_cols, const uint64_t* c, uint32_t nmask) {
  const unsigned long long row = atomicAdd(o.n_rows, 1ull);
  if ((int64_t)row >= o.capacity) return;
  for (int k = 0; k < n_cols; k++) {
    const bool nul = (nmask >> k) & 1u;
    o.valid[k][row] = nul ? 0 : 1;
    if (nul) o.has_null[k] = 1u;
    ((uint64_t*)o.col[k])[row] = c[k];
  }
}

__global__ void __launch_bounds__(256) uni_snapshot_kernel(UniDev t, int S, int n_cols, SnapOut o) {
  for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < t.cap + 2; b += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = *(const unsigned long long*)ub(t, (int64_t)b);
    if (b < t.cap && key == J_EMPTY) continue;
    uint32_t m;
    if (S == t.is) {
      const unsigned long long WI = *ub_WI(t, (int64_t)b);
      if (W_istate(WI) == 1u) snap_emit_uni(o, n_cols, ub_cols(t, (int64_t)b), (uint32_t)(*ub_IH(t, (int64_t)b) & 0xffull));
      m = W_head(WI);
    } else {
      m = *ub_chead(t, (int64_t)b);
    }
    while (m != U_NIL) {
      const UniRec* rec = urec(t, S, m);
      if (!(rec->link & J_DEAD)) snap_emit_uni(o, n_cols, rec->c, rec->nullmask);
      m = rec->link & 0x7fffffffu;
    }
  }
}

__global__ void __launch_bounds__(256) join_snapshot_kernel(const JoinPlanDev* __restrict__ p, int S, JoinSideDev s, SnapOut o) {
  for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < s.cap + 2; b += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t w0 = *(const uint64_t*)bkt(s, (int64_t)b);
    if (b < s.cap && (p->single_key ? w0 == J_EMPTY : w0 == 0ull)) continue;
    for_each_live(s, p, (int64_t)b, [&](uint8_t* rec) -> bool {
      const unsigned long long row = atomicAdd(o.n_rows, 1ull);
      if ((int64_t)row < o.capacity) {
        const uint32_t nmask = ((const RecHdr*)rec)->nullmask;
        for (int k = 0; k < p->n_cols[S]; k++) {
          const bool nul = (nmask >> k) & 1u;
          o.valid[k][row] = nul ? 0 : 1;
          if (nul) o.has_null[k] = 1u;
          const int w = p->col_width[S][k];
          if (!nul) copy_bytes((uint8_t*)o.col[k] + row * w, rec + p->col_off[S][k], w);
        }
      }
      return true;
    });
  }
}
// two-table layout: rows of side S whose key column `key_pos` is below the watermark leave the state
__global__ void __launch_bounds__(256) join_clean_kernel(const JoinPlanDev* __restrict__ p, JoinSideDev s, int key_pos, long long wm) {
  for (uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; b < s.cap + 2; b += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t* w = (const uint64_t*)bkt(s, (int64_t)b);
    long long kv;
    if (p->single_key) {
      if (b == s.cap) continue;  // NULL key
      if (b < s.cap && w[0] == J_EMPTY) continue;
      kv = b == s.cap + 1 ? (long long)J_EMPTY : (long long)w[0];
    } else {
      if (b >= s.cap || w[0] == 0ull) continue;
      if ((w[0] >> (8 + key_pos)) & 1ull) continue;  // NULL in this key column
      kv = (long long)w[1 + key_pos];
    }
    if (kv >= wm) continue;
    unsigned long long* Wp = bkt_W(s, p, (int64_t)b);
    *Wp = W_EMPTY | (W_istate(*Wp) ? W_IL_DEAD : 0ull);
  }
}
}  // namespace rw

// =============================================================================== host handle
using namespace rw;

// unified table: a side's log as a list of 2^22-record segments behind a device table of pointers (join_uni.cuh)
struct SegLog {
  std::vector<DevBuf> segs;
  DevBuf table;  // U_MAX_SEGS device pointers
  // ONE segment is allocated ahead of need by a helper thread (a 200 MB cudaMalloc takes 1.5-2 ms on the GPU boxes:
  // on the push path the GPU would idle for ten steps' worth of time)
  std::thread worker;
  std::mutex mu;
  DevBuf spare;
  bool spare_ready = false, worker_running = false;
  uint64_t stalls = 0, prefetched = 0;  // segments allocated on the push path / taken from the helper
  SegLog() = default;
  SegLog(const SegLog&) = delete;
  ~SegLog() { if (worker.joinable()) worker.join(); }
  uint64_t cap() const { return (uint64_t)segs.size() << U_SEG_SHIFT; }
  void prefetch() {
    {
      std::lock_guard<std::mutex> g(mu);
      if (worker_running || spare_ready || segs.size() >= U_MAX_SEGS) return;
      worker_running = true;
    }
    if (worker.joinable()) worker.join();
    int dev = 0;
    cudaGetDevice(&dev);
    worker = std::thread([this, dev]() {
      cudaSetDevice(dev);
      DevBuf b;
      const cudaError_t e = b.reserve((size_t)U_SEG_RECS * 48);
      std::lock_guard<std::mutex> g(mu);
      if (e == cudaSuccess) { spare = std::move(b); spare_ready = true; } else { cudaGetLastError(); }
      worker_running = false;
    });
  }
  // make room for `rows` records: new segments are allocated and their pointers appended ON `st` (stream order puts
  // the table update before every kernel launched afterwards; existing entries never change)
  int ensure(uint64_t rows, cudaStream_t st) {
    if (!table.p) {
      RW_CUDA(table.reserve(U_MAX_SEGS * sizeof(void*)));
      RW_CUDA(cudaMemsetAsync(table.p, 0, U_MAX_SEGS * sizeof(void*), st));
    }
    while (cap() < rows) {
      if (segs.size() >= U_MAX_SEGS) return fail(RW_ERR_OOM, "join side exceeds 2^31 log rows");
      DevBuf sg;
      if (worker.joinable()) worker.join();  // (a running helper finishes sooner than a second allocation would)
      {
        std::lock_guard<std::mutex> g(mu);
        if (spare_ready) { sg = std::move(spare); spare_ready = false; prefetched++; }
      }
      if (!sg.p) {
        cudaError_t e = sg.reserve((size_t)U_SEG_RECS * 48);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(RW_ERR_OOM, std::string("join log segment: ") + cudaGetErrorString(e)); }
        stalls++;
      }
      void* ptr = sg.p;
      // (the pointer is copied from a pageable temporary: cudaMemcpyAsync stages it before returning)
      RW_CUDA(cudaMemcpyAsync(table.as<uint8_t>() + segs.size() * sizeof(void*), &ptr, sizeof(void*), cudaMemcpyHostToDevice, st));
      segs.push_back(std::move(sg));
    }
    return RW_OK;
  }
};

struct JoinSideHost {
  int n_cols = 0;
  std::vector<int> types;
  SegLog log;          // unified table: the side's row log
  GrowBuf recs;        // overflow record store (grows in place)
  DevBuf slots;        // bucket array
  DevBuf pools;        // per-warp row-id pools of join_inner_q4_kernel
  int stride = 0, bstride = 0;
  uint64_t row_cap = 0;   // records allocated
  uint64_t n_rows = 0;    // records handed out (incl. dead ones)
  uint64_t slot_cap = 0;
  uint64_t keys_upper = 0;
};

// one push between its launch and its collection
struct JoinPending {
  int S = 0, set = 0, grid = 0;
  DevChunk ch;            // the caller keeps the chunk's buffers valid until the push is collected
  cudaStream_t st = nullptr;
  int64_t out_base = 0;
  bool plain = true, counted = false, sync_done = false;
  uint32_t pool_chunk = 0;
  uint64_t seq_base = 0, ids_before = 0, keys_before = 0;
  unsigned long long tag = 0;
  int64_t rows = 0;               // sync_done: the result of a push that was completed at launch time
  unsigned long long nullm = 0;
};

struct rwgpu_join {
  JoinPlanDev plan;
  DevBuf plan_dev, status;
  PinnedBuf status_host;
  JoinSideHost side[2];
  cudaStream_t stream = nullptr, s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_h2d[8] = {nullptr}, ev_main[8] = {nullptr};
  std::vector<int> out_types;
  int chunk_size = 1024;
  bool fast_inner = false;
  bool w8_ok[2] = {false, false};  // per update side: Key64 + all-8-byte columns specialisation usable
  bool q4_ok = false;              // both sides: 3..4 columns, 64-byte buckets -> quad-cooperative kernel
  W8Plan w8[2];
  // unified table (join_uni.cuh): Key64 inner join, <= 4 eight-byte columns per side -- ONE bucket array for both sides
  bool uni = false;
  int uni_is = 1;                  // inline side
  DevBuf uni_buckets, uni_counters;  // counters: log_next[2], n_dead[2], scratch
  uint64_t uni_cap = 0, uni_keys = 0, uni_keys_exact = 0;  // uni_keys: upper bound while pushes are outstanding
  uint64_t uni_dead[2] = {0, 0};
  uint64_t compactions = 0;
  DevBuf uni_wk_entry, uni_wk_mask;  // worklist of the rows the hot kernel defers (join_uni.cuh UniWork)
  int64_t uni_wk_cap = 0;
  // launch / collect split (rwgpu_join_push_device_async / rwgpu_join_collect): pushes enqueued but not collected
  JoinPending pending[2];
  int n_pending = 0;
  cudaEvent_t pend_ev[2] = {nullptr, nullptr};
  cudaStream_t last_st = nullptr;
  cudaEvent_t order_ev = nullptr;
  // watermark-driven state cleaning, applied at the next barrier
  bool wm_pending[2] = {false, false};
  int wm_key_pos[2] = {0, 0};
  int64_t wm_value[2] = {0, 0};
  uint64_t wm_cleanings = 0;
  uint64_t launches = 0;
  uint64_t seq = 0;
  unsigned long long status_tag = 0;
  unsigned long long call_null_mask = 0;  // null_mask accumulated over the sub-batches of one API call
  bool out_rows_cumulative = false;       // the device out_rows counter was left non-zero by the scan-based kernel
  KernelProf prof;
  // scratch (generic path)
  DevBuf sk, sk_alt, packed, offs, mslot, gtable, cub_tmp;
  int64_t scratch_rows = 0;
  uint64_t gcap = 0;
  size_t cub_bytes = 0;
  // output (device)
  // two output sets: the rows of push s can still be read while push s + 1 is computed (launch / collect split);
  // the synchronous entry points only ever use the current one
  struct OutSet {
    DevBuf out_ops, out_vis, out_col[J_MAX_OUT], out_valid[J_MAX_OUT], out_bits[J_MAX_OUT], out_visbits;
    int64_t out_cap = 0;
    unsigned long long valid_dirty = 0;  // columns whose valid bytes hold zeros from the previous push
  } oset[2];
  int cur = 0;
  OutSet& os() { return oset[cur]; }
  // host staging
  DevBuf up;
  PinnedBuf up_host;
  // launch / collect split for HOST chunks (rwgpu_join_push_async / rwgpu_join_collect_out): per output set, the device
  // staging of the input, the pinned output block and what collect still has to copy
  struct HostPending {
    bool active = false, sync_done = false;
    rwgpu_out* out = nullptr;      // sync_done: the finished result; else the block the copies land in
    rw_chunk in;                   // the caller's chunk (its buffers stay valid until collect: rwgpu.h)
    std::vector<rw_column> in_cols;
    std::vector<int> alias_src;
    int64_t n = 0, host_cap = 0;
    bool alias_ok = false;
  } hpend[2];
  DevBuf up2[2];
  PinnedBuf up2_host[2];
  cudaEvent_t ev_up2[2] = {nullptr, nullptr};
  cudaStream_t s_out[2] = {nullptr, nullptr};  // one copy-out stream per output set: collecting push s must not wait for
                                               // the copies of push s+1, which are already queued when s is collected
  std::shared_ptr<PinnedPool> pool = std::make_shared<PinnedPool>();
  std::vector<rw_column> dev_view_cols[2];  // per output set
  DevBuf noop_nxt, noop_prv, noop_elig, noop_flag;  // eliminate_adjacent_noop_update scratch
  // varlen payload (see varlen_intern_kernel): per-side byte heaps, per input column handle staging, per output column bytes
  std::vector<int> var_in[2];        // varlen columns of each side
  std::vector<int> var_out;          // varlen output columns
  DevBuf var_heap[2], var_ctr;       // var_ctr: heap_next[2] (u64), err (u32)
  uint64_t var_cap[2] = {0, 0}, var_upper[2] = {0, 0};
  DevBuf var_handles[RW_MAX_COLS], var_stage_off[RW_MAX_COLS], var_stage_bytes[RW_MAX_COLS];  // device staging of an input chunk
  struct VarOut { DevBuf lens, offs, bytes, tmp; size_t tmp_bytes = 0; int64_t cap = 0; uint32_t total = 0; } vout[2][J_MAX_OUT];
  int64_t noop_cap = 0;
  bool call_had_deletes = false;            // some push of the current API call saw visible Delete / UpdateDelete rows
  bool call_vis_stale = false;              // the scan-based kernel compacts its output and never writes vis bytes
  ~rwgpu_join() {
    for (auto e : ev_h2d) if (e) cudaEventDestroy(e);
    for (auto e : ev_main) if (e) cudaEventDestroy(e);
    for (auto e : pend_ev) if (e) cudaEventDestroy(e);
    if (order_ev) cudaEventDestroy(order_ev);
    if (s_h2d) cudaStreamDestroy(s_h2d);
    if (s_d2h) cudaStreamDestroy(s_d2h);
    if (stream) cudaStreamDestroy(stream);
  }
};

static int jgrid(int64_t n, int block) {
  int64_t g = (n + block - 1) / block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(g, 148 * 8));
}

static JoinSideDev side_dev(const rwgpu_join* h, int S) {
  const JoinSideHost& s = h->side[S];
  JoinSideDev d;
  d.recs = s.recs.as<uint8_t>();
  d.pools = s.pools.as<uint2>();
  d.rec_cap = s.row_cap;
  d.buckets = s.slots.as<uint8_t>();
  d.cap = s.slot_cap;
  d.stride = s.stride;
  d.bstride = s.bstride;
  return d;
}

static int join_alloc_slots(rwgpu_join* h, int S, DevBuf& buf, uint64_t cap) {
  const int bs = h->side[S].bstride;
  RW_CUDA(buf.reserve((cap + 2) * (size_t)bs));
  join_init_slots_kernel<<<jgrid((int64_t)cap + 2, 256), 256, 0, h->stream>>>(buf.as<uint8_t>(), cap, bs, h->plan.KW, h->plan.single_key);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  return RW_OK;
}

// grow the record store of side S to hold at least `rows` records (contents preserved, in place)
static int join_grow_store(rwgpu_join* h, int S, uint64_t rows) {
  JoinSideHost& s = h->side[S];
  if (h->uni) {
    if (rows >= 0x7ffffff0ull) return fail(RW_ERR_OOM, "join side exceeds 2^31 rows");
    int rc = RW_OK;
    if (rows > s.log.cap()) {
      rc = s.log.ensure(rows, h->last_st ? h->last_st : h->stream);
      s.row_cap = s.log.cap();
    }
    // less than one segment of headroom left in a log that is at least half full: have the next segment allocated in the
    // background (a fresh single-segment log of a small operator never asks for a spare)
    if (rc == RW_OK && !s.log.segs.empty() && rows + U_SEG_RECS > s.log.cap() && rows * 2 > s.log.cap()) s.log.prefetch();
    return rc;
  }
  if (rows <= s.row_cap) return RW_OK;
  if (rows >= 0x7ffffff0ull) return fail(RW_ERR_OOM, "join side exceeds 2^31 rows");
  // address space for the whole row-id range, capped at the device's memory size
  size_t free_b = 0, total_b = 0;
  cudaMemGetInfo(&free_b, &total_b);
  const size_t va_limit = std::min<size_t>((size_t)0x7ffffff0ull * (size_t)s.stride, std::max<size_t>(total_b, (size_t)1 << 30));
  RW_CUDA(cudaDeviceSynchronize());  // (growth only) pushes may be in flight on a caller's stream
  const uint64_t live_rows = std::min<uint64_t>(s.n_rows, s.row_cap);  // n_rows is an upper bound while pushes are outstanding
  cudaError_t e = s.recs.ensure((size_t)rows * (size_t)s.stride, (size_t)live_rows * (size_t)s.stride, va_limit, h->stream);
  if (e != cudaSuccess) return fail(RW_ERR_OOM, std::string("join record store: ") + cudaGetErrorString(e));
  s.row_cap = std::min<uint64_t>(s.recs.bytes() / (size_t)s.stride, 0x7ffffff0ull);
  return RW_OK;
}

static int join_grow_slots(rwgpu_join* h, int S, uint64_t need_keys) {
  JoinSideHost& s = h->side[S];
  // linear probing over 64-byte buckets: keep load <= 0.5
  if (need_keys * 2 <= s.slot_cap) return RW_OK;
  uint64_t ncap = s.slot_cap;
  while (ncap < need_keys * 4) ncap <<= 1;  // regrow to load <= 0.25
  DevBuf nb;
  int rc = join_alloc_slots(h, S, nb, ncap);
  if (rc != RW_OK) return rc;
  join_rehash_kernel<<<jgrid((int64_t)s.slot_cap + 2, 256), 256, 0, h->stream>>>(s.slots.as<uint8_t>(), s.slot_cap, nb.as<uint8_t>(), ncap,
                                                                                  s.bstride, h->plan.KW, h->plan.single_key, h->plan.n_keys);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  RW_CUDA(cudaStreamSynchronize(h->stream));
  s.slots = std::move(nb);
  s.slot_cap = ncap;
  return RW_OK;
}

static int join_ensure_scratch(rwgpu_join* h, int64_t n) {
  if (n > h->scratch_rows) {
    int64_t cap = std::max<int64_t>(n, 4096);
    RW_CUDA(h->sk.reserve((size_t)cap * 8));
    RW_CUDA(h->sk_alt.reserve((size_t)cap * 8));
    RW_CUDA(h->packed.reserve((size_t)cap * 8));
    RW_CUDA(h->offs.reserve((size_t)cap * 8));
    RW_CUDA(h->mslot.reserve((size_t)cap * 8));
    uint64_t g = 1024;
    while (g < (uint64_t)cap * 2) g <<= 1;
    RW_CUDA(h->gtable.reserve(g * 4));
    h->gcap = g;
    size_t b1 = 0, b2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, b1, (uint64_t*)nullptr, (uint64_t*)nullptr, (int)cap);
    cub::DoubleBuffer<uint64_t> db((uint64_t*)nullptr, (uint64_t*)nullptr);
    cub::DeviceRadixSort::SortKeys(nullptr, b2, db, (int)cap);
    h->cub_bytes = std::max(b1, b2) + 256;
    RW_CUDA(h->cub_tmp.reserve(h->cub_bytes));
    h->scratch_rows = cap;
  }
  return RW_OK;
}

// make room for `rows` output rows; the first `keep` rows already written are preserved
static int join_ensure_out(rwgpu_join* h, int64_t rows, cudaStream_t st, int64_t keep = 0) {
  if (rows <= h->os().out_cap) return RW_OK;
  int64_t cap = std::max<int64_t>(rows + rows / 4, 4096);
  RW_CUDA(cudaDeviceSynchronize());
  auto grow = [&](DevBuf& b, size_t elt, bool fill_one) -> int {
    DevBuf nb;
    RW_CUDA(nb.reserve((size_t)cap * elt));
    if (fill_one) RW_CUDA(cudaMemset(nb.p, 1, (size_t)cap * elt));
    if (keep > 0 && b.p) RW_CUDA(cudaMemcpy(nb.p, b.p, (size_t)keep * elt, cudaMemcpyDeviceToDevice));
    b = std::move(nb);
    return RW_OK;
  };
  int rc = grow(h->os().out_ops, 1, false);
  if (rc != RW_OK) return rc;
  rc = grow(h->os().out_vis, 1, false);
  if (rc != RW_OK) return rc;
  RW_CUDA(h->os().out_visbits.reserve((size_t)((cap + 63) / 64) * 8));
  for (size_t k = 0; k < h->out_types.size(); k++) {
    rc = grow(h->os().out_col[k], (size_t)type_width(h->out_types[k]), false);
    if (rc != RW_OK) return rc;
    rc = grow(h->os().out_valid[k], 1, true);  // invariant: valid bytes are 1 between pushes
    if (rc != RW_OK) return rc;
    RW_CUDA(h->os().out_bits[k].reserve((size_t)((cap + 63) / 64) * 8));
  }
  if (keep == 0) h->os().valid_dirty = 0;
  h->os().out_cap = cap;
  return RW_OK;
}

// restore the "valid bytes are all 1" invariant for the columns the previous push wrote NULLs to
static int join_clean_valid(rwgpu_join* h, cudaStream_t st) {
  for (size_t k = 0; k < h->out_types.size(); k++)
    if ((h->os().valid_dirty >> k) & 1) RW_CUDA(cudaMemsetAsync(h->os().out_valid[k].p, 1, (size_t)h->os().out_cap, st));
  h->os().valid_dirty = 0;
  return RW_OK;
}

static JoinOutDev out_dev(rwgpu_join* h) {
  JoinOutDev o;
  memset(&o, 0, sizeof(o));
  o.ops = h->os().out_ops.as<uint8_t>();
  o.vis = h->os().out_vis.as<uint8_t>();
  for (size_t k = 0; k < h->out_types.size(); k++) { o.col[k] = h->os().out_col[k].p; o.valid[k] = h->os().out_valid[k].as<uint8_t>(); }
  o.capacity = h->os().out_cap;
  o.heap[0] = h->var_heap[0].as<uint8_t>();
  o.heap[1] = h->var_heap[1].as<uint8_t>();
  return o;
}

// The status block is pushed to pinned host memory by a one-thread kernel (UVA: cudaMallocHost memory
// is device-addressable) instead of a cudaMemcpy: a tiny D2H copy would queue on the copy engine
// behind the megabytes of output the previous sub-batch is still draining.
__global__ void join_status_to_host_kernel(JoinStatus* src, JoinStatus* dst_host, unsigned long long tag, int reset) {
  join_status_publish(src, dst_host, tag, reset);
}
// `tag` != 0: a kernel already in the stream publishes the status itself unless it had real work
// (join_inner_delete_kernel); only then is the one-thread kernel needed.
static int join_read_status(rwgpu_join* h, cudaStream_t st, JoinStatus* out, int reset = 1, unsigned long long tag = 0) {
  JoinStatus* host = h->status_host.as<JoinStatus>();
  if (tag) {
    RW_CUDA(cudaStreamSynchronize(st));
    if (*(volatile unsigned long long*)(host + 1) == tag) {
      memcpy(out, host, sizeof(JoinStatus));
      return RW_OK;
    }
  }
  join_status_to_host_kernel<<<1, 1, 0, st>>>(h->status.as<JoinStatus>(), host, 0ull, reset);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  RW_CUDA(cudaStreamSynchronize(st));
  memcpy(out, host, sizeof(JoinStatus));
  return RW_OK;
}

static int join_check_err(rwgpu_join* h, const JoinStatus& s, cudaStream_t st) {
  if (!s.err) return RW_OK;
  unsigned int e = s.err;
  cudaMemsetAsync(&h->status.as<JoinStatus>()->err, 0, sizeof(unsigned int), st);
  if (e & JERR_DOUBLE_DELETE) return fail(RW_ERR_INCONSISTENT, "removing a join state entry but it is not in the cache");
  if (e & JERR_APPEND_ONLY_MULTI) return fail(RW_ERR_INCONSISTENT, "append-only optimisation: more than one matched row");
  if (e & JERR_STORE_CAPACITY) return fail(RW_ERR_CUDA, "internal: join record store capacity");
  if (e & JERR_BAD_COUNT) return fail(RW_ERR_INVALID, "device row count out of range");
  return fail(RW_ERR_CUDA, "internal: join output capacity");
}

// =============================================================================== unified-table path (join_uni.cuh)
static UniDev uni_dev(rwgpu_join* h) {
  UniDev t;
  t.buckets = h->uni_buckets.as<uint8_t>();
  t.cap = h->uni_cap;
  unsigned long long* ctr = h->uni_counters.as<unsigned long long>();
  for (int s = 0; s < 2; s++) {
    t.log[s] = h->side[s].log.table.as<uint8_t*>();
    t.log_cap[s] = h->side[s].log.cap();
    t.pools[s] = h->side[s].pools.as<uint2>();
    t.log_next[s] = ctr + s;
    t.n_dead[s] = ctr + 2 + s;
  }
  t.is = h->uni_is;
  return t;
}

static int uni_alloc_buckets(rwgpu_join* h, DevBuf& buf, uint64_t cap) {
  RW_CUDA(buf.reserve((cap + 2) * 64));
  uni_init_kernel<<<jgrid((int64_t)cap + 2, 256), 256, 0, h->stream>>>(buf.as<uint8_t>(), 0, cap + 2);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  return RW_OK;
}

// keep the load of the bucket array <= 0.5 (every extra probe is one more random 64-byte transaction)
static int uni_grow_table(rwgpu_join* h, uint64_t need_keys) {
  if (need_keys * 2 <= h->uni_cap) return RW_OK;
  // `need_keys` is an upper bound: every row of every outstanding push counted as a new key, and a push whose row count
  // lives on the device counted at its buffer CAPACITY (N>1: world x the rows it will really hold).  As long as the
  // keys KNOWN to exist keep the load under 0.5 and even the bound leaves a tenth of the buckets free, probing
  // terminates and nothing has to stop; the exact count arrives with the next collect.
  if (h->uni_keys_exact * 2 <= h->uni_cap && need_keys * 10 <= h->uni_cap * 9) return RW_OK;
  uint64_t ncap = h->uni_cap;
  while (ncap < need_keys * 4) ncap <<= 1;
  RW_CUDA(cudaDeviceSynchronize());  // every push in flight on any stream has finished with the old array
  DevBuf nb;
  int rc = uni_alloc_buckets(h, nb, ncap);
  if (rc != RW_OK) return rc;
  uni_rehash_kernel<<<jgrid((int64_t)h->uni_cap + 2, 256), 256, 0, h->stream>>>(h->uni_buckets.as<uint8_t>(), h->uni_cap, nb.as<uint8_t>(), ncap);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  RW_CUDA(cudaStreamSynchronize(h->stream));
  h->uni_buckets = std::move(nb);
  h->uni_cap = ncap;
  return RW_OK;
}

// barrier-time compaction of side s's log: live records only, in chain order (join_uni.cuh uni_compact_kernel)
static int uni_compact(rwgpu_join* h, int s) {
  JoinSideHost& sd = h->side[s];
  RW_CUDA(cudaDeviceSynchronize());
  SegLog fresh;
  // the live records are at most the ids handed out minus the dead ones; the pools restart empty, so leave them room
  const uint64_t live_upper = sd.n_rows > h->uni_dead[s] ? sd.n_rows - h->uni_dead[s] : 0;
  int rc = fresh.ensure(std::max<uint64_t>(live_upper, 1), h->stream);
  if (rc != RW_OK) { set_error(""); return RW_OK; }  // no room for a second log right now: keep the old one
  unsigned long long* ctr = h->uni_counters.as<unsigned long long>();
  RW_CUDA(cudaMemsetAsync(ctr + 4, 0, 8, h->stream));
  uni_compact_kernel<<<jgrid((int64_t)h->uni_cap + 2, 256), 256, 0, h->stream>>>(uni_dev(h), s, fresh.table.as<uint8_t*>(), ctr + 4);
  RW_CUDA(cudaGetLastError());
  h->launches++;
  unsigned long long live = 0;
  RW_CUDA(cudaMemcpyAsync(&live, ctr + 4, 8, cudaMemcpyDeviceToHost, h->stream));
  RW_CUDA(cudaStreamSynchronize(h->stream));
  std::swap(sd.log.segs, fresh.segs);
  {
    DevBuf t2 = std::move(sd.log.table);
    sd.log.table = std::move(fresh.table);
    fresh.table = std::move(t2);
  }
  sd.row_cap = sd.log.cap();
  sd.n_rows = live;
  h->uni_dead[s] = 0;
  const unsigned long long zero = 0;
  RW_CUDA(cudaMemcpyAsync(ctr + s, &live, 8, cudaMemcpyHostToDevice, h->stream));
  RW_CUDA(cudaMemcpyAsync(ctr + 2 + s, &zero, 8, cudaMemcpyHostToDevice, h->stream));
  RW_CUDA(cudaMemsetAsync(sd.pools.p, 0, sd.pools.bytes, h->stream));  // the warps' id pools pointed into the old log
  RW_CUDA(cudaStreamSynchronize(h->stream));
  h->compactions++;
  return RW_OK;
}

// all work of one handle forms ONE logical stream: a call on another cuda stream than the previous call's waits
// for it on the device
static int join_order(rwgpu_join* h, cudaStream_t st) {
  if (h->last_st && h->last_st != st) {
    if (!h->order_ev) RW_CUDA(cudaEventCreateWithFlags(&h->order_ev, cudaEventDisableTiming));
    RW_CUDA(cudaEventRecord(h->order_ev, h->last_st));
    RW_CUDA(cudaStreamWaitEvent(st, h->order_ev, 0));
  }
  h->last_st = st;
  return RW_OK;
}

// grid of the tail kernel: about one wave, no more than the rows need
static int uni_tail_grid(int64_t n) {
  static int max_blocks = 0;
  if (!max_blocks) {
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int a = 0, b = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, uni_tail_kernel<false>, 256, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, uni_tail_kernel<true>, 256, 0);
    per_sm = std::max(1, std::min(std::min(a, b), 3));
    max_blocks = std::max(1, sms * per_sm);
  }
  return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, max_blocks));
}

// main kernel (timed by the profiler) + the tail kernel, which ends by publishing the status block
// (tagged `tag`) into the pinned slot of the push's output set
static int uni_launch_main(rwgpu_join* h, const JoinPending& pd, bool probe_only, unsigned long long tag) {
  UniDev t = uni_dev(h);
  const JoinPlanDev* pdev = h->plan_dev.as<JoinPlanDev>();
  JoinStatus* ds = h->status.as<JoinStatus>();
  int S = pd.S;
  const bool is_row = S == h->uni_is;
  JoinOutDev od = out_dev(h);
  UniWork wk;
  wk.entry = h->uni_wk_entry.as<UniDefer>();
  wk.mask = h->uni_wk_mask.as<uint8_t>();
  W8Plan w = h->w8[S];
  h->prof.begin(pd.st);
  if (pd.plain) {
    PlainChunk pc;
    pc.ops = pd.ch.ops;
    for (int c = 0; c < 4; c++) pc.c[c] = c < w.n_u ? (const unsigned long long*)pd.ch.cols[c].data : nullptr;
    pc.key = (const unsigned long long*)pd.ch.cols[w.key_col].data;
    pc.n = pd.ch.n;
    pc.n_dev = pd.ch.n_dev;
    UniOwn own;
    own.log = t.log[S];
    own.log_cap = t.log_cap[S];
    own.pools = t.pools[S];
    own.log_next = t.log_next[S];
    PlainOut po;
    po.ops = od.ops;
    po.vis = od.vis;
    for (int c = 0; c < 4; c++) {
      po.ucol[c] = (c < w.n_u && w.u_out[c] >= 0) ? (unsigned long long*)od.col[w.u_out[c]] : nullptr;
      po.mcol[c] = (c < w.n_m && w.m_out[c] >= 0) ? (unsigned long long*)od.col[w.m_out[c]] : nullptr;
    }
    po.capacity = od.capacity;
    // resident blocks per SM (registers per thread): 4 (64) by default; RWGPU_UNI_MINB=3 / 5 / 6 for tuning runs
    static const int minb = getenv("RWGPU_UNI_MINB") ? atoi(getenv("RWGPU_UNI_MINB")) : 4;
    static const uint32_t kflags = getenv("RWGPU_UNI_FLAGS") ? (uint32_t)atoi(getenv("RWGPU_UNI_FLAGS")) : 0u;  // bit 0: L2 prefetch of the next bucket (key column two groups ahead), bit 1: deferred link store
#define UNI_LAUNCH(PO, IS, MB) uni_hot_kernel<PO, IS, MB><<<pd.grid, JF_BLOCK, 0, pd.st>>>(pc, t.buckets, t.cap, own, po, wk, ds, pd.seq_base, pd.out_base, pd.pool_chunk, kflags)
    if (probe_only) {
      if (is_row) UNI_LAUNCH(true, true, 4); else UNI_LAUNCH(true, false, 4);
    } else if (is_row) {
      UNI_LAUNCH(false, true, 4);
    } else {
      switch (minb) {
        case 3: UNI_LAUNCH(false, false, 3); break;
        case 5: UNI_LAUNCH(false, false, 5); break;
        case 6: UNI_LAUNCH(false, false, 6); break;
        default:
          if (kflags & 2u) uni_hot_kernel<false, false, 4, true><<<pd.grid, JF_BLOCK, 0, pd.st>>>(pc, t.buckets, t.cap, own, po, wk, ds, pd.seq_base, pd.out_base,
                                                                                                pd.pool_chunk, kflags);
          else UNI_LAUNCH(false, false, 4);
          break;
      }
    }
#undef UNI_LAUNCH
  } else {
    if (probe_only) uni_slow_kernel<true><<<jgrid(pd.ch.n, 256), 256, 0, pd.st>>>(pdev, w, S, pd.ch, t, od, ds, pd.seq_base, pd.out_base);
    else uni_slow_kernel<false><<<jgrid(pd.ch.n, 256), 256, 0, pd.st>>>(pdev, w, S, pd.ch, t, od, ds, pd.seq_base, pd.out_base);
  }
  h->prof.end(pd.st);
  RW_CUDA(cudaGetLastError());
  // tail: deferred rows, own-side deletes, status publication
  DevChunk chv = pd.ch;
  uint64_t seq_base = pd.seq_base;
  int64_t out_base = pd.out_base;
  JoinStatus* slot = (JoinStatus*)(h->status_host.as<uint8_t>() + 512 * pd.set);
  int reset = 3;
  unsigned int* done = (unsigned int*)(h->uni_counters.as<unsigned long long>() + 6);
  const int tg = uni_tail_grid(pd.ch.n);
  if (probe_only) uni_tail_kernel<true><<<tg, 256, 0, pd.st>>>(pdev, w, S, chv, t, od, wk, ds, seq_base, out_base, slot, tag, reset, done);
  else uni_tail_kernel<false><<<tg, 256, 0, pd.st>>>(pdev, w, S, chv, t, od, wk, ds, seq_base, out_base, slot, tag, reset, done);
  RW_CUDA(cudaGetLastError());
  h->launches += 2;
  return RW_OK;
}

// LAUNCH half of a push: main kernel + delete kernel (which publishes the status block into the output set's pinned
// slot) are enqueued on `st`; nothing is waited for.  The output goes to the CURRENT output set (h->cur).
static double uni_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static const bool uni_trace = getenv("RWGPU_TRACE") != nullptr;  // host-side timeline on stderr (debugging only)

static int uni_enqueue(rwgpu_join* h, int S, const DevChunk& ch_in, cudaStream_t st, int64_t out_base, JoinPending* pd) {
  const double tr0 = uni_trace ? uni_now_ms() : 0.0;
  DevChunk ch = ch_in;
  bool plain_cols = ch.vis_bits == nullptr;
  for (int c = 0; c < ch.n_cols && plain_cols; c++)
    plain_cols = !ch.cols[c].valid_bits && !ch.cols[c].valid_bytes && (((uintptr_t)ch.cols[c].data & 7) == 0);
  bool counted = ch.n_dev != nullptr;
  if (counted && !plain_cols) {  // only the quad-cooperative kernel reads the row count on the device
    int64_t nh = 0;
    RW_CUDA(cudaMemcpyAsync(&nh, ch.n_dev, sizeof(nh), cudaMemcpyDeviceToHost, st));
    RW_CUDA(cudaStreamSynchronize(st));
    if (nh < 0 || nh > ch.n) return fail(RW_ERR_INVALID, "device row count out of range");
    ch.n = nh;
    ch.n_dev = nullptr;
    counted = false;
  }
  const int64_t n = ch.n;  // capacity when `counted`
  JoinSideHost& own = h->side[S];
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 63) / 64, Q4_MAX_GRID));
  uint32_t pool_chunk = 32;
  while (pool_chunk < 256 && (int64_t)pool_chunk * grid * 8 < 4 * n) pool_chunk <<= 1;
  // the warps draw log ids from persistent pools in chunks: the id counter can run ahead of the rows stored by one chunk
  // per warp.  own.n_rows / uni_keys are UPPER bounds while pushes are outstanding (corrected when they are collected).
  const uint64_t id_slack = (uint64_t)grid * 8 * pool_chunk;
  int rc = join_grow_store(h, S, own.n_rows + (uint64_t)n + id_slack);
  if (rc != RW_OK) return rc;
  rc = uni_grow_table(h, h->uni_keys + (uint64_t)n);
  if (rc != RW_OK) return rc;
  rc = join_ensure_out(h, out_base + n + std::max<int64_t>(n / 2, 4096), st, out_base);
  if (rc != RW_OK) return rc;
  if (plain_cols && n > h->uni_wk_cap) {
    RW_CUDA(cudaDeviceSynchronize());  // (growth only) an outstanding push may still read the old worklist
    const int64_t cap = n + n / 4 + 64;
    RW_CUDA(h->uni_wk_entry.reserve((size_t)cap * sizeof(UniDefer)));
    RW_CUDA(h->uni_wk_mask.reserve((size_t)(cap + 7) / 8 + 16));
    h->uni_wk_cap = cap;
  }
  rc = join_order(h, st);
  if (rc != RW_OK) return rc;
  const double tr1 = uni_trace ? uni_now_ms() : 0.0;
  pd->S = S;
  pd->ch = ch;
  pd->st = st;
  pd->out_base = out_base;
  pd->set = h->cur;
  pd->plain = plain_cols;
  pd->counted = counted;
  pd->grid = grid;
  pd->pool_chunk = pool_chunk;
  pd->seq_base = h->seq;
  pd->tag = ++h->status_tag;
  pd->ids_before = own.n_rows;
  pd->keys_before = h->uni_keys;
  h->seq += (uint64_t)n;
  own.n_rows += (uint64_t)n + id_slack;  // upper bounds until the status comes back
  h->uni_keys += (uint64_t)n;
  static const bool dbg_probe_only = getenv("RWGPU_DBG_PROBE_ONLY") != nullptr;  // timing experiments only (state is not updated)
  rc = uni_launch_main(h, *pd, dbg_probe_only && S == 0, pd->tag);
  if (rc != RW_OK) return rc;
  if (!h->pend_ev[pd->set]) RW_CUDA(cudaEventCreateWithFlags(&h->pend_ev[pd->set], cudaEventDisableTiming));
  RW_CUDA(cudaEventRecord(h->pend_ev[pd->set], st));
  if (uni_trace)
    fprintf(stderr, "  [uni_enqueue S=%d n=%lld set=%d] grow/ensure %.3f ms, launch %.3f ms (log segs %zu/%zu, cap %llu keys<=%llu)\n", S, (long long)n,
            pd->set, tr1 - tr0, uni_now_ms() - tr1, h->side[0].log.segs.size(), h->side[1].log.segs.size(), (unsigned long long)h->uni_cap,
            (unsigned long long)h->uni_keys);
  return RW_OK;
}

// COLLECT half: wait for the push, read its status, redo the (state-free) emission if the extra-match area was too
// small, settle the host's bookkeeping.  h->cur must be pd.set.
static int uni_finish(rwgpu_join* h, const JoinPending& pd, int64_t* out_rows, unsigned long long* null_mask) {
  cudaStream_t st = pd.st;
  JoinStatus* ds = h->status.as<JoinStatus>();
  JoinStatus* slot = (JoinStatus*)(h->status_host.as<uint8_t>() + 512 * pd.set);
  JoinStatus hs;
  const double tr0 = uni_trace ? uni_now_ms() : 0.0;
  RW_CUDA(cudaEventSynchronize(h->pend_ev[pd.set]));
  const double tr1 = uni_trace ? uni_now_ms() : 0.0;
  int rc;
  if (*(volatile unsigned long long*)(slot + 1) != pd.tag) return fail(RW_ERR_CUDA, "join status block was not published");
  memcpy(&hs, slot, sizeof(JoinStatus));
  unsigned int err = hs.err;
  const unsigned long long first_null = hs.null_mask;
  const bool first_match = hs.pad != 0;
  const unsigned long long first_del = hs.n_del;
  const bool redone = (hs.err & JERR_OUT_CAPACITY) != 0;
  if (redone) {
    // the extra-match area overflowed: redo the probe + emit with room for every reservation.  The probe reads the
    // OTHER side's state only, which no later push of the same side has touched (pushes of different sides are never
    // outstanding together), so the redo is exact.
    const int64_t extras = (int64_t)hs.out_rows, n = pd.ch.n;
    RW_CUDA(cudaMemsetAsync(&ds->err, 0, 4, st));
    rc = join_ensure_out(h, pd.out_base + n + extras + (int64_t)pd.grid * 8 * U_XCHUNK, st, pd.out_base);
    if (rc != RW_OK) return rc;
    const unsigned long long tag2 = ++h->status_tag;
    rc = uni_launch_main(h, pd, true, tag2);
    if (rc != RW_OK) return rc;
    RW_CUDA(cudaStreamSynchronize(st));
    if (*(volatile unsigned long long*)(slot + 1) != tag2) return fail(RW_ERR_CUDA, "join status block was not published");
    memcpy(&hs, slot, sizeof(JoinStatus));
    err = (err & ~JERR_OUT_CAPACITY) | hs.err;
    hs.null_mask |= first_null & ~(1ull << 63);
    hs.pad = hs.pad || first_match;
    hs.n_del = first_del;  // (the redo is probe-only: it counts no deletes)
  }
  // bookkeeping: what the device really used, plus the upper bounds of the pushes enqueued after this one.  Those pushes
  // (still in h->pending: the caller has taken this one out) recorded the uncorrected bounds as their bases; their bases
  // move by the same amount, so that their own collect removes exactly their share (with a stale base the bounds can
  // wrap below zero, and the bucket-array growth loop never terminates)
  for (int s = 0; s < 2; s++) h->uni_dead[s] = hs.n_dead[s];
  {
    JoinSideHost& own = h->side[pd.S];
    const uint64_t n = (uint64_t)pd.ch.n, slack = (uint64_t)pd.grid * 8 * pd.pool_chunk;
    const uint64_t rows = hs.log_next[pd.S] + (own.n_rows - (pd.ids_before + n + slack));
    const uint64_t keys = hs.n_keys[0] + (h->uni_keys - (pd.keys_before + n));
    for (int i = 0; i < h->n_pending; i++) {
      if (h->pending[i].S == pd.S) h->pending[i].ids_before += rows - own.n_rows;
      h->pending[i].keys_before += keys - h->uni_keys;
    }
    own.n_rows = rows;
    h->uni_keys = keys;
    h->uni_keys_exact = hs.n_keys[0];
  }
  hs.err = err;
  rc = join_check_err(h, hs, st);
  if (rc != RW_OK) return rc;
  const int64_t n_eff = pd.counted ? (int64_t)hs.n_in : pd.ch.n;
  *out_rows = (hs.pad != 0 || hs.out_rows) ? n_eff + (int64_t)hs.out_rows : 0;
  h->call_null_mask |= hs.null_mask;
  *null_mask = h->call_null_mask;
  h->os().valid_dirty |= hs.null_mask & ((1ull << 63) - 1);
  if (hs.n_del) h->call_had_deletes = true;
  if (uni_trace)
    fprintf(stderr, "  [uni_finish S=%d set=%d] wait %.3f ms, rest %.3f ms (redo %d, extras %llu, n_del %llu, out %lld)\n", pd.S, pd.set, tr1 - tr0,
            uni_now_ms() - tr1, (int)redone, (unsigned long long)hs.out_rows,
            (unsigned long long)hs.n_del, (long long)*out_rows);
  return RW_OK;
}

static int join_push_dev_uni(rwgpu_join* h, int S, const DevChunk& ch_in, cudaStream_t st, int64_t out_base, int64_t* out_rows,
                             unsigned long long* null_mask) {
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes first");
  JoinPending pd;
  int rc = uni_enqueue(h, S, ch_in, st, out_base, &pd);
  if (rc != RW_OK) return rc;
  return uni_finish(h, pd, out_rows, null_mask);
}

// one push of a device-resident chunk; on return the output sits in the device output buffers.
// *null_mask: bit k = output column k holds NULLs, bit 63 = some rows are invisible.
// `out_base` rows of the device output buffers are already occupied by earlier sub-batches of the
// same API call (the caller zeroed status.out_rows / null_mask before the first one).
static int join_push_dev(rwgpu_join* h, int S, const DevChunk& ch_in, cudaStream_t st, int64_t out_base, int64_t* out_rows,
                         unsigned long long* null_mask) {
  *out_rows = 0;
  DevChunk ch = ch_in;
  if (ch.n <= 0) return RW_OK;
  if (ch.n >= (1ll << 31)) return fail(RW_ERR_INVALID, "chunk too large");
  if (h->uni) return join_push_dev_uni(h, S, ch_in, st, out_base, out_rows, null_mask);
  // Key64 / 8-byte-column specialisations need a chunk without bitmaps (ops == 0 still hides rows)
  bool plain_cols = ch.vis_bits == nullptr;
  for (int c = 0; c < ch.n_cols && plain_cols; c++)
    plain_cols = !ch.cols[c].valid_bits && !ch.cols[c].valid_bytes && (((uintptr_t)ch.cols[c].data & 7) == 0);
  static const bool no_q4_env = getenv("RWGPU_NO_Q4") != nullptr;
  // device-resident row count: only the quad-cooperative kernel reads it on the device; every other path
  // fetches it first (one 8-byte read-back) and proceeds with an ordinary chunk
  bool counted = ch.n_dev != nullptr;
  if (counted && !(h->fast_inner && h->q4_ok && !no_q4_env && h->w8_ok[S] && plain_cols)) {
    int64_t nh = 0;
    RW_CUDA(cudaMemcpyAsync(&nh, ch.n_dev, sizeof(nh), cudaMemcpyDeviceToHost, st));
    RW_CUDA(cudaStreamSynchronize(st));
    if (nh < 0 || nh > ch.n) return fail(RW_ERR_INVALID, "device row count out of range");
    ch.n = nh;
    ch.n_dev = nullptr;
    counted = false;
    if (nh == 0) return RW_OK;
  }
  const int64_t n = ch.n;  // capacity when `counted`
  JoinSideHost& own = h->side[S];
  static const bool trace = getenv("RWGPU_TRACE") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double tt0 = now();
  const uint64_t cap0 = own.slot_cap, rcap0 = own.row_cap;
  // quad-cooperative kernel: its warps draw overflow row ids from persistent pools in chunks, so the
  // id counter can run ahead of the rows really stored by one chunk per warp
  const bool q4 = h->fast_inner && h->q4_ok && !no_q4_env;
  const int q4_grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 63) / 64, Q4_MAX_GRID));
  uint32_t pool_chunk = 32;
  while (pool_chunk < 256 && (int64_t)pool_chunk * q4_grid * 8 < 4 * n) pool_chunk <<= 1;
  int rc = join_grow_store(h, S, own.n_rows + (uint64_t)n + (q4 ? (uint64_t)q4_grid * 8 * pool_chunk : 0));
  if (rc != RW_OK) return rc;
  rc = join_grow_slots(h, S, own.keys_upper + (uint64_t)n);
  if (rc != RW_OK) return rc;
  if (trace)
    fprintf(stderr, "  [push_dev S=%d n=%lld] grow %.3f ms (slot_cap %llu->%llu, row_cap %llu->%llu, n_rows %llu keys %llu)\n", S, (long long)n,
            now() - tt0, (unsigned long long)cap0, (unsigned long long)own.slot_cap, (unsigned long long)rcap0,
            (unsigned long long)own.row_cap, (unsigned long long)own.n_rows, (unsigned long long)own.keys_upper);
  JoinStatus* ds = h->status.as<JoinStatus>();
  const JoinPlanDev* pd = h->plan_dev.as<JoinPlanDev>();
  // n_store / n_del are zero here: every status read-back resets them (join_status_publish)
  const uint64_t seq_base = h->seq;
  h->seq += (uint64_t)n;
  JoinStatus hs;
  if (h->fast_inner) {
    // Key64 / 8-byte-column specialisation when the chunk carries no bitmaps (ops == 0 still hides rows)
    const bool use_w8 = h->w8_ok[S] && plain_cols;
    static const bool dbg_probe_only = getenv("RWGPU_DBG_PROBE_ONLY") != nullptr;  // timing experiments only (state is not updated)
    if (use_w8) {
      // positional output: n rows aligned with the input + extra matches behind them
      // (out_rows / pad: zeroed by join_begin_call and by the previous push's status read-back)
      rc = join_ensure_out(h, out_base + n + std::max<int64_t>(n / 2, 4096), st, out_base);
      if (rc != RW_OK) return rc;
      // quad-cooperative kernel when both sides fit a 64-byte bucket (<= 4 columns); else one thread per row
      const int grid = q4 ? q4_grid : jgrid(n, JF_BLOCK);
      auto launch = [&](bool probe_only, uint32_t store_base) {
        if (q4) {
          // 4 blocks of 256 threads per SM (64 registers).  Measured per 2^20 rows: 3 blocks/SM 0.262 ms, 4: 0.227,
          // 5: 0.267, 6: 0.300, 8: 0.329 -- the kernel is bound by random DRAM transactions, not by occupancy.
          if (probe_only)
            join_inner_q4_kernel<true, 4><<<grid, JF_BLOCK, 0, st>>>(pd, h->w8[S], S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h),
                                                                      ds, store_base, seq_base, out_base, pool_chunk);
          else
            join_inner_q4_kernel<false, 4><<<grid, JF_BLOCK, 0, st>>>(pd, h->w8[S], S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h),
                                                                       ds, store_base, seq_base, out_base, pool_chunk);
        } else {
          if (probe_only)
            join_inner_w8p_kernel<true><<<grid, JF_BLOCK, 0, st>>>(pd, h->w8[S], S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h), ds,
                                                                    store_base, seq_base, out_base);
          else
            join_inner_w8p_kernel<false><<<grid, JF_BLOCK, 0, st>>>(pd, h->w8[S], S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h), ds,
                                                                     store_base, seq_base, out_base);
        }
      };
      h->prof.begin(st);
      launch(dbg_probe_only && S == 0, (uint32_t)own.n_rows);
      h->prof.end(st);
      const unsigned long long tag = ++h->status_tag;
      join_inner_delete_kernel<<<jgrid(n, 256), 256, 0, st>>>(pd, S, ch, side_dev(h, S), ds, seq_base, h->status_host.as<JoinStatus>(), tag, 3);
      RW_CUDA(cudaGetLastError());
      h->launches += 2;
      rc = join_read_status(h, st, &hs, 3, tag);
      if (rc != RW_OK) return rc;
      const uint64_t stored = hs.n_store, keys = hs.n_keys[S];
      if (hs.n_del) h->call_had_deletes = true;
      unsigned int err = hs.err;
      if (hs.err & JERR_OUT_CAPACITY) {
        // the extra-match area overflowed: redo the (state-free) probe + emit with room for every row
        const int64_t extras = (int64_t)hs.out_rows;
        RW_CUDA(cudaMemsetAsync(&ds->out_rows, 0, 8, st));
        RW_CUDA(cudaMemsetAsync(&ds->err, 0, 4, st));
        RW_CUDA(cudaStreamSynchronize(st));
        rc = join_ensure_out(h, out_base + n + extras, st, out_base);
        if (rc != RW_OK) return rc;
        launch(true, 0u);
        RW_CUDA(cudaGetLastError());
        h->launches++;
        rc = join_read_status(h, st, &hs, 3);
        if (rc != RW_OK) return rc;
        err = (err & ~JERR_OUT_CAPACITY) | hs.err;
      }
      own.n_rows += stored;
      own.keys_upper = keys;
      const bool any_match = hs.pad != 0;
      hs.err = err;
      rc = join_check_err(h, hs, st);
      if (rc != RW_OK) return rc;
      const int64_t n_eff = counted ? (int64_t)hs.n_in : n;  // positional rows = rows of the input chunk
      *out_rows = (any_match || hs.out_rows) ? n_eff + (int64_t)hs.out_rows : 0;
    } else {
      rc = join_ensure_out(h, out_base + std::max<int64_t>(2 * n, 4096), st, out_base);
      if (rc != RW_OK) return rc;
      h->out_rows_cumulative = true;
      h->call_vis_stale = true;
      const int64_t tiles = (n + JF_BLOCK * JF_R - 1) / (JF_BLOCK * JF_R);
      const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, 148 * 8));
      h->prof.begin(st);
      join_inner_fused_kernel<false><<<grid, JF_BLOCK, 0, st>>>(pd, S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h), ds,
                                                                  (uint32_t)own.n_rows, seq_base);
      h->prof.end(st);
      join_inner_delete_kernel<<<jgrid(n, 256), 256, 0, st>>>(pd, S, ch, side_dev(h, S), ds, seq_base, nullptr, 0ull, 0);
      RW_CUDA(cudaGetLastError());
      h->launches += 2;
      rc = join_read_status(h, st, &hs);
      if (rc != RW_OK) return rc;
      const uint64_t stored = hs.n_store, keys = hs.n_keys[S];
      if (hs.n_del) h->call_had_deletes = true;
      unsigned int err = hs.err;
      while (hs.err & JERR_OUT_CAPACITY) {
        // the reservation overflowed: redo the (state-free) probe + emit with room for every row
        const int64_t need = (int64_t)hs.out_rows;
        const unsigned long long base_ull = (unsigned long long)out_base;
        RW_CUDA(cudaMemcpyAsync(&ds->out_rows, &base_ull, 8, cudaMemcpyHostToDevice, st));
        RW_CUDA(cudaMemsetAsync(&ds->n_store, 0, 16, st));
        RW_CUDA(cudaMemsetAsync(&ds->err, 0, 4, st));
        RW_CUDA(cudaStreamSynchronize(st));
        rc = join_ensure_out(h, need, st, out_base);
        if (rc != RW_OK) return rc;
        join_inner_fused_kernel<true><<<grid, JF_BLOCK, 0, st>>>(pd, S, ch, side_dev(h, S), side_dev(h, 1 - S), out_dev(h), ds, 0, seq_base);
        RW_CUDA(cudaGetLastError());
        h->launches++;
        rc = join_read_status(h, st, &hs);
        if (rc != RW_OK) return rc;
        err = (err & ~JERR_OUT_CAPACITY) | hs.err;
      }
      own.n_rows += stored;
      own.keys_upper = keys;
      hs.err = err;
      rc = join_check_err(h, hs, st);
      if (rc != RW_OK) return rc;
      *out_rows = (int64_t)hs.out_rows - out_base;
      // keep the cumulative convention of the scan-based kernel consistent with out_base
    }
  } else {
    rc = join_ensure_scratch(h, n);
    if (rc != RW_OK) return rc;
    JoinScratch sc;
    sc.sortkey = h->sk.as<uint64_t>();
    sc.sortkey_alt = h->sk_alt.as<uint64_t>();
    sc.packed = h->packed.as<uint64_t>();
    sc.offs = h->offs.as<uint64_t>();
    sc.match_slot = h->mslot.as<int64_t>();
    sc.gtable = h->gtable.as<int32_t>();
    uint64_t g = 1024;
    while (g < (uint64_t)n * 2) g <<= 1;
    sc.gcap = g;
    fill_i32_kernel<<<jgrid((int64_t)g, 256), 256, 0, st>>>(sc.gtable, g, -1);
    join_prepare_kernel<<<jgrid(n, 256), 256, 0, st>>>(pd, S, ch, side_dev(h, 1 - S), sc);
    RW_CUDA(cudaGetLastError());
    size_t tb = h->cub_bytes;
    cub::DeviceScan::ExclusiveSum(h->cub_tmp.p, tb, sc.packed, sc.offs, (int)n, st);
    join_totals_kernel<<<1, 1, 0, st>>>(sc.packed, sc.offs, n, ds);
    cub::DoubleBuffer<uint64_t> db(sc.sortkey, sc.sortkey_alt);
    tb = h->cub_bytes;
    cub::DeviceRadixSort::SortKeys(h->cub_tmp.p, tb, db, (int)n, 0, 64, st);
    RW_CUDA(cudaGetLastError());
    h->launches += 6;
    rc = join_read_status(h, st, &hs, 0);  // n_store (written by join_totals_kernel) must survive until the second read
    if (rc != RW_OK) return rc;
    const int64_t reserved = (int64_t)hs.out_rows;
    rc = join_ensure_out(h, out_base + reserved, st, out_base);
    if (rc != RW_OK) return rc;
    if (reserved > 0) RW_CUDA(cudaMemsetAsync(h->os().out_vis.as<uint8_t>() + out_base, 1, (size_t)reserved, st));
    h->prof.begin(st);
    join_serial_kernel<<<jgrid(n, 128), 128, 0, st>>>(pd, S, ch, side_dev(h, S), side_dev(h, 1 - S), sc, db.Current(), out_dev(h), ds,
                                                        (uint32_t)own.n_rows, (uint32_t)seq_base, out_base);
    h->prof.end(st);
    RW_CUDA(cudaGetLastError());
    h->launches++;
    rc = join_read_status(h, st, &hs);
    if (rc != RW_OK) return rc;
    own.n_rows += hs.n_store;
    own.keys_upper = hs.n_keys[S];
    rc = join_check_err(h, hs, st);
    if (rc != RW_OK) return rc;
    *out_rows = reserved;
  }
  if (!h->fast_inner) h->call_had_deletes = true;  // outer / semi / anti joins emit Delete rows for Insert inputs too
  h->call_null_mask |= hs.null_mask;  // the device copy restarts from zero after every read-back
  *null_mask = h->call_null_mask;
  h->os().valid_dirty |= hs.null_mask & ((1ull << 63) - 1);
  return RW_OK;
}

// eliminate_adjacent_noop_update over the first n rows of the current output set (device).  The positional kernels
// write vis bytes for every row; the scan-based kernel leaves them untouched, hence `vis_valid`.
static int join_eliminate_noop(rwgpu_join* h, int64_t n, bool vis_valid, cudaStream_t st, bool* hid_rows) {
  *hid_rows = false;
  if (n < 2) return RW_OK;
  if (n > h->noop_cap) {
    RW_CUDA(cudaStreamSynchronize(st));
    const int64_t cap = n + n / 4;
    RW_CUDA(h->noop_nxt.reserve((size_t)cap * 4));
    RW_CUDA(h->noop_prv.reserve((size_t)cap * 4));
    RW_CUDA(h->noop_elig.reserve((size_t)cap));
    RW_CUDA(h->noop_flag.reserve(8));
    h->noop_cap = cap;
  }
  RW_CUDA(cudaMemsetAsync(h->noop_flag.p, 0, 8, st));
  if (!vis_valid) RW_CUDA(cudaMemsetAsync(h->os().out_vis.p, 1, (size_t)n, st));
  NoopScratch sc;
  sc.nxt = h->noop_nxt.as<int32_t>();
  sc.prv = h->noop_prv.as<int32_t>();
  sc.elig = h->noop_elig.as<uint8_t>();
  const int g = jgrid(n, 256);
  unsigned int* flag = h->noop_flag.as<unsigned int>();
  const unsigned long long null_cols = h->call_null_mask & ((1ull << 63) - 1);
  noop_edges_kernel<<<g, 256, 0, st>>>(out_dev(h), h->plan_dev.as<JoinPlanDev>(), n, h->chunk_size, sc, null_cols, flag);
  noop_prev_kernel<<<g, 256, 0, st>>>(n, h->chunk_size, sc, flag);
  noop_take_kernel<<<g, 256, 0, st>>>(out_dev(h), n, sc, flag);
  noop_normalize_kernel<<<g, 256, 0, st>>>(out_dev(h), n, h->chunk_size, flag);
  RW_CUDA(cudaGetLastError());
  h->launches += 4;
  unsigned int hid = 0;  // did the pass hide anything ?
  RW_CUDA(cudaMemcpyAsync(&hid, h->noop_flag.p, 4, cudaMemcpyDeviceToHost, st));
  RW_CUDA(cudaStreamSynchronize(st));
  *hid_rows = hid != 0;
  return RW_OK;
}

// start of an API call: restore the valid-byte invariant, zero the per-call accumulators
static int join_begin_call(rwgpu_join* h, cudaStream_t st) {
  int rc = join_clean_valid(h, st);
  if (rc != RW_OK) return rc;
  JoinStatus* ds = h->status.as<JoinStatus>();
  if (h->out_rows_cumulative) RW_CUDA(cudaMemsetAsync(&ds->out_rows, 0, 8, st));  // scan-based kernel: cumulative over sub-batches
  h->out_rows_cumulative = false;
  h->call_null_mask = 0;
  h->call_had_deletes = false;
  h->call_vis_stale = false;
  return RW_OK;
}

extern "C" {

int32_t rwgpu_join_create(const rw_join_desc* d, rwgpu_join** out) {
  if (!d || !out) return fail(RW_ERR_INVALID, "null descriptor");
  int rc = rwgpu_device_check();
  if (rc != RW_OK) return rc;
  if (d->join_type < 0 || d->join_type > RW_JOIN_RIGHT_ANTI) return fail(RW_ERR_INVALID, "join type");
  if (d->n_keys < 1 || d->n_keys > RW_MAX_KEYS) return fail(RW_ERR_UNSUPPORTED, "1..4 join key columns supported");
  if (d->left.n_cols > RW_MAX_COLS || d->right.n_cols > RW_MAX_COLS) return fail(RW_ERR_UNSUPPORTED, "too many columns");
  auto h = new rwgpu_join();
  std::unique_ptr<rwgpu_join> guard(h);
  JoinPlanDev& p = h->plan;
  memset(&p, 0, sizeof(p));
  p.T = d->join_type;
  p.n_keys = d->n_keys;
  const rw_join_side_desc* sd[2] = {&d->left, &d->right};
  bool pk_in_jk[2];
  for (int s = 0; s < 2; s++) {
    JoinSideHost& hs = h->side[s];
    hs.n_cols = sd[s]->n_cols;
    hs.types.assign(sd[s]->types, sd[s]->types + sd[s]->n_cols);
    p.n_cols[s] = sd[s]->n_cols;
    int off = J_HDR;
    for (int c = 0; c < sd[s]->n_cols; c++) {
      int w = type_width(sd[s]->types[c]);
      if (!w) return fail(RW_ERR_UNSUPPORTED, "unsupported column type");
      p.col_type[s][c] = sd[s]->types[c];
      p.col_width[s][c] = w;
      off = (off + w - 1) / w * w;  // natural alignment
      p.col_off[s][c] = off;
      off += w;
    }
    p.stride[s] = (off + 15) / 16 * 16;
    hs.stride = p.stride[s];
    for (int c = 0; c < sd[s]->n_cols; c++)
      if (type_is_varlen(sd[s]->types[c])) h->var_in[s].push_back(c);
    for (int k = 0; k < d->n_keys; k++) {
      int c = sd[s]->key_indices[k];
      if (c < 0 || c >= sd[s]->n_cols) return fail(RW_ERR_INVALID, "join key index");
      if (sd[s]->types[c] == RW_T_DECIMAL) return fail(RW_ERR_UNSUPPORTED, "decimal join key");
      if (type_is_varlen(sd[s]->types[c])) return fail(RW_ERR_UNSUPPORTED, "varlen join key (KeySerialized) stays on the CPU executor");
      p.key_col[s][k] = c;
    }
    p.n_pk[s] = sd[s]->n_pk;
    for (int i = 0; i < sd[s]->n_pk; i++) {
      if (sd[s]->pk_indices[i] < 0 || sd[s]->pk_indices[i] >= sd[s]->n_cols) return fail(RW_ERR_INVALID, "pk index");
      if (type_is_varlen(sd[s]->types[sd[s]->pk_indices[i]])) return fail(RW_ERR_UNSUPPORTED, "varlen pk column");
      p.pk_col[s][i] = sd[s]->pk_indices[i];
    }
    // pk_contained_in_jk (hash_join.rs:377-378)
    pk_in_jk[s] = true;
    for (int i = 0; i < sd[s]->n_stream_key; i++) {
      bool f = false;
      for (int k = 0; k < d->n_keys; k++) f = f || (sd[s]->key_indices[k] == sd[s]->stream_key[i]);
      pk_in_jk[s] = pk_in_jk[s] && f;
    }
  }
  for (int k = 0; k < d->n_keys; k++) {
    if (d->left.types[d->left.key_indices[k]] != d->right.types[d->right.key_indices[k]])
      return fail(RW_ERR_INVALID, "join key types differ");
    p.null_safe[k] = d->null_safe ? d->null_safe[k] : 0;
  }
  const int T = p.T;
  p.append_only_optimize = d->is_append_only && pk_in_jk[0] && pk_in_jk[1];  // :381
  const bool need_l = (T == RW_JOIN_FULL_OUTER || T == RW_JOIN_LEFT_OUTER || T == RW_JOIN_LEFT_ANTI || T == RW_JOIN_LEFT_SEMI);
  const bool need_r = (T == RW_JOIN_FULL_OUTER || T == RW_JOIN_RIGHT_OUTER || T == RW_JOIN_RIGHT_ANTI || T == RW_JOIN_RIGHT_SEMI);
  p.need_degree[0] = need_l && !pk_in_jk[1];  // :397
  p.need_degree[1] = need_r && !pk_in_jk[0];  // :398
  // output schema (:337-359) and i2o mappings (builder.rs:63-80)
  int left_len = d->left.n_cols, right_len = d->right.n_cols;
  std::vector<int> nat;
  if (T == RW_JOIN_LEFT_SEMI || T == RW_JOIN_LEFT_ANTI) { nat.assign(d->left.types, d->left.types + left_len); right_len = 0; }
  else if (T == RW_JOIN_RIGHT_SEMI || T == RW_JOIN_RIGHT_ANTI) { nat.assign(d->right.types, d->right.types + right_len); left_len = 0; }
  else { nat.assign(d->left.types, d->left.types + left_len); nat.insert(nat.end(), d->right.types, d->right.types + right_len); }
  (void)right_len;
  if (d->n_output < 0 || d->n_output > J_MAX_OUT) return fail(RW_ERR_UNSUPPORTED, "too many output columns");
  p.n_out = d->n_output;
  for (int oi = 0; oi < d->n_output; oi++) {
    int idx = d->output_indices[oi];
    if (idx < 0 || idx >= (int)nat.size()) return fail(RW_ERR_INVALID, "output_indices out of bound");
    p.out_type[oi] = nat[idx];
    p.out_width[oi] = type_width(nat[idx]);
    h->out_types.push_back(nat[idx]);
    if (type_is_varlen(nat[idx])) h->var_out.push_back(oi);
    int s = idx < left_len ? 0 : 1;
    int local = idx < left_len ? idx : idx - left_len;
    p.map_in[s][p.n_map[s]] = local;
    p.map_out[s][p.n_map[s]] = oi;
    p.n_map[s]++;
  }
  p.cond_cmp = d->cond.cmp;
  p.cond_lhs = d->cond.lhs;
  p.cond_rhs = d->cond.rhs;
  if (p.cond_cmp != RW_CMP_NONE) {
    int tot = d->left.n_cols + d->right.n_cols;
    if (p.cond_cmp < 0 || p.cond_cmp > RW_CMP_NE || p.cond_lhs < 0 || p.cond_lhs >= tot || p.cond_rhs < 0 || p.cond_rhs >= tot)
      return fail(RW_ERR_INVALID, "join condition");
    for (int idx : {p.cond_lhs, p.cond_rhs}) {
      int t = idx < d->left.n_cols ? d->left.types[idx] : d->right.types[idx - d->left.n_cols];
      if (type_is_float(t) || t == RW_T_DECIMAL || type_is_varlen(t)) return fail(RW_ERR_UNSUPPORTED, "non-integer join condition stays on the CPU executor");
    }
  }
  p.single_key = (p.n_keys == 1);
  p.KW = p.single_key ? 1 : 1 + p.n_keys;
  p.SW = p.KW + 1;
  p.bhdr = ((p.KW + 1) * 8 + 15) / 16 * 16;  // the inline record starts 16-byte aligned (its header is written with one 16-byte store)
  for (int s2 = 0; s2 < 2; s2++) {
    p.bstride[s2] = (p.bhdr + p.stride[s2] + 15) / 16 * 16;
    h->side[s2].bstride = p.bstride[s2];
  }
  p.strict = d->strict_consistency;
  h->chunk_size = std::max(d->chunk_size > 0 ? d->chunk_size : 1024, 2);  // builder.rs:44-47
  h->fast_inner = (T == RW_JOIN_INNER) && !p.append_only_optimize;
  // W8 specialisation: one 8-byte non-float key, <= 8 columns per side, all 8 bytes wide, no
  // condition, every input column projected to at most one output column
  for (int s2 = 0; s2 < 2 && h->fast_inner; s2++) {
    W8Plan& w = h->w8[s2];
    memset(&w, 0, sizeof(w));
    bool ok = p.single_key && p.cond_cmp == RW_CMP_NONE && p.n_cols[0] <= W8_MAXC && p.n_cols[1] <= W8_MAXC;
    for (int side = 0; side < 2 && ok; side++)
      for (int c = 0; c < p.n_cols[side]; c++) ok = ok && p.col_width[side][c] == 8 && p.col_off[side][c] == J_HDR + 8 * c;
    ok = ok && !type_is_float(p.col_type[s2][p.key_col[s2][0]]);
    w.n_u = p.n_cols[s2];
    w.n_m = p.n_cols[1 - s2];
    w.key_col = p.key_col[s2][0];
    for (int c = 0; c < W8_MAXC; c++) { w.u_out[c] = -1; w.m_out[c] = -1; }
    for (int i = 0; i < p.n_map[s2] && ok; i++) {
      if (w.u_out[p.map_in[s2][i]] >= 0) ok = false;
      w.u_out[p.map_in[s2][i]] = (int8_t)p.map_out[s2][i];
    }
    for (int i = 0; i < p.n_map[1 - s2] && ok; i++) {
      if (w.m_out[p.map_in[1 - s2][i]] >= 0) ok = false;
      w.m_out[p.map_in[1 - s2][i]] = (int8_t)p.map_out[1 - s2][i];
    }
    h->w8_ok[s2] = ok;
  }
  h->q4_ok = h->w8_ok[0] && h->w8_ok[1] && p.bhdr == 16 && p.stride[0] == 48 && p.stride[1] == 48 && p.bstride[0] == 64 &&
             p.bstride[1] == 64 && p.n_cols[0] <= 4 && p.n_cols[1] <= 4;

  // unified table: one bucket array for both sides (join_uni.cuh).  RWGPU_NO_UNI=1 keeps the two-table kernels.
  h->uni = h->fast_inner && h->w8_ok[0] && h->w8_ok[1] && p.n_cols[0] <= 4 && p.n_cols[1] <= 4 && getenv("RWGPU_NO_UNI") == nullptr;
  h->uni_is = pk_in_jk[1] ? 1 : (pk_in_jk[0] ? 0 : 1);

  RW_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  RW_CUDA(h->var_ctr.reserve(32));
  RW_CUDA(cudaMemsetAsync(h->var_ctr.p, 0, 32, h->stream));
  RW_CUDA(h->plan_dev.reserve(sizeof(JoinPlanDev)));
  RW_CUDA(cudaMemcpyAsync(h->plan_dev.p, &p, sizeof(p), cudaMemcpyHostToDevice, h->stream));
  RW_CUDA(h->status.reserve(sizeof(JoinStatus)));
  RW_CUDA(cudaMemsetAsync(h->status.p, 0, sizeof(JoinStatus), h->stream));
  RW_CUDA(h->status_host.reserve(1024));
  if (h->uni) {
    const uint64_t hint = std::max(d->left.row_capacity_hint, d->right.row_capacity_hint);
    uint64_t cap = 1024;
    while (cap * 4 < hint * 10) cap <<= 1;  // load <= 0.4 at `hint` keys
    h->uni_cap = cap;
    rc = uni_alloc_buckets(h, h->uni_buckets, cap);
    if (rc != RW_OK) return rc;
    RW_CUDA(h->uni_counters.reserve(8 * sizeof(unsigned long long)));
    RW_CUDA(cudaMemsetAsync(h->uni_counters.p, 0, 8 * sizeof(unsigned long long), h->stream));
    for (int s = 0; s < 2; s++) {
      h->side[s].stride = 48;
      h->last_st = h->stream;
      // chained side: every row lives in its log; inline side: only the 2nd, 3rd ... row of a key
      uint64_t rows = s == h->uni_is ? std::max<uint64_t>(4096, sd[s]->row_capacity_hint / 4) : std::max<uint64_t>(4096, 2 * sd[s]->row_capacity_hint);
      if (sd[s]->stored_rows_hint && s != h->uni_is) rows = std::max<uint64_t>(4096, sd[s]->stored_rows_hint);
      rc = join_grow_store(h, s, std::min<uint64_t>(rows, 0x40000000ull));
      if (rc != RW_OK) return rc;
      RW_CUDA(h->side[s].pools.reserve((size_t)Q4_MAX_GRID * (JF_BLOCK / 32) * sizeof(uint2)));
      RW_CUDA(cudaMemsetAsync(h->side[s].pools.p, 0, h->side[s].pools.bytes, h->stream));
    }
  }
  for (int s = 0; s < 2 && !h->uni; s++) {
    uint64_t hint = sd[s]->row_capacity_hint;
    uint64_t cap = 1024;
    while (cap * 4 < hint * 10) cap <<= 1;  // load <= 0.4 at `hint` keys (every extra probe is a 64 B HBM access)
    h->side[s].slot_cap = cap;
    rc = join_alloc_slots(h, s, h->side[s].slots, cap);
    if (rc != RW_OK) return rc;
    // overflow rows only; sized from the planner's cardinality hint (2 rows per expected key) so that a
    // stream of the expected size never pays a doubling (allocate + copy + free) in its data path
    rc = join_grow_store(h, s, std::max<uint64_t>(1024, std::min<uint64_t>(2 * hint, 0x40000000ull)));
    if (rc != RW_OK) return rc;
    RW_CUDA(h->side[s].pools.reserve((size_t)Q4_MAX_GRID * (JF_BLOCK / 32) * sizeof(uint2)));
    RW_CUDA(cudaMemsetAsync(h->side[s].pools.p, 0, h->side[s].pools.bytes, h->stream));
    if (rc != RW_OK) return rc;
  }
  RW_CUDA(cudaStreamSynchronize(h->stream));
  *out = guard.release();
  return RW_OK;
}

void rwgpu_join_destroy(rwgpu_join* h) {
  if (!h) return;
  cudaDeviceSynchronize();  // pushes may be outstanding on the handle's or a caller's stream
  for (int i = 0; i < 2; i++) {
    delete h->hpend[i].out;
    if (h->s_out[i]) cudaStreamDestroy(h->s_out[i]);
  }
  delete h;
}

int32_t rwgpu_join_push_device(rwgpu_join* h, int32_t side, const rw_chunk* c, rw_chunk* view, void* cuda_stream) {
  return rwgpu_join_push_device_counted(h, side, c, nullptr, view, cuda_stream);
}

// ---- varlen payload: heaps, interning, materialisation (see varlen_intern_kernel)
static int var_ensure_heap(rwgpu_join* h, int S, uint64_t bytes) {
  if (h->var_upper[S] + bytes <= h->var_cap[S]) return RW_OK;
  RW_CUDA(cudaDeviceSynchronize());
  unsigned long long used = 0;
  RW_CUDA(cudaMemcpy(&used, h->var_ctr.as<unsigned long long>() + S, 8, cudaMemcpyDeviceToHost));
  h->var_upper[S] = used;
  if (used + bytes <= h->var_cap[S]) return RW_OK;
  const uint64_t ncap = std::max<uint64_t>(std::max<uint64_t>(h->var_cap[S] * 2, (used + bytes) + (used + bytes) / 2), 1 << 20);
  if (ncap >= (1ull << 40)) return fail(RW_ERR_OOM, "varlen heap exceeds 1 TiB");
  DevBuf nb;
  RW_CUDA(nb.reserve((size_t)ncap));
  if (used) RW_CUDA(cudaMemcpy(nb.p, h->var_heap[S].p, (size_t)used, cudaMemcpyDeviceToDevice));
  h->var_heap[S] = std::move(nb);
  h->var_cap[S] = ncap;
  return RW_OK;
}

// intern rows [0, m) of one varlen column (device pointers; value r = bytes_base[offs[r] .. offs[r+1])) -> handles[m]
static int var_intern(rwgpu_join* h, int S, const uint8_t* bytes_base, const uint32_t* offs, const uint8_t* ops, const uint64_t* vis_bits,
                      const uint64_t* valid_bits, int64_t m, uint64_t* handles, cudaStream_t st) {
  if (m <= 0) return RW_OK;
  varlen_intern_kernel<<<jgrid(m, 256), 256, 0, st>>>(bytes_base, offs, ops, vis_bits, valid_bits, m, h->var_heap[S].as<uint8_t>(),
                                                       h->var_ctr.as<unsigned long long>() + S, h->var_cap[S], S + 1, handles,
                                                       (unsigned int*)(h->var_ctr.as<unsigned long long>() + 2));
  RW_CUDA(cudaGetLastError());
  h->launches++;
  return RW_OK;
}

static int var_check_err(rwgpu_join* h, cudaStream_t st) {
  unsigned int e = 0;
  RW_CUDA(cudaMemcpyAsync(&e, h->var_ctr.as<unsigned long long>() + 2, 4, cudaMemcpyDeviceToHost, st));
  RW_CUDA(cudaStreamSynchronize(st));
  if (!e) return RW_OK;
  RW_CUDA(cudaMemsetAsync(h->var_ctr.as<unsigned long long>() + 2, 0, 4, st));
  if (e & 1u) return fail(RW_ERR_UNSUPPORTED, "a varlen value of 4 MiB or more");
  return fail(RW_ERR_CUDA, "internal: varlen heap capacity");
}

// handles[n] (device) -> vo.offs[n + 1] + vo.bytes on the device; vo.total = bytes.  vis / valid: byte arrays or nullptr.
static int var_materialize(rwgpu_join* h, rwgpu_join::VarOut& vo, const uint64_t* handles, const uint8_t* vis, const uint8_t* valid, int64_t n,
                           cudaStream_t st) {
  if (n + 1 > vo.cap) {
    RW_CUDA(cudaStreamSynchronize(st));
    const int64_t cap = n + n / 4 + 64;
    RW_CUDA(vo.lens.reserve((size_t)cap * 4));
    RW_CUDA(vo.offs.reserve((size_t)cap * 4));
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)cap);
    RW_CUDA(vo.tmp.reserve(tb + 256));
    vo.tmp_bytes = tb + 256;
    vo.cap = cap;
  }
  vo.total = 0;
  if (n == 0) { RW_CUDA(cudaMemsetAsync(vo.offs.p, 0, 4, st)); return RW_OK; }
  varlen_lens_kernel<<<jgrid(n, 256), 256, 0, st>>>(handles, vis, valid, n, vo.lens.as<uint32_t>());
  size_t tb = vo.tmp_bytes;
  cub::DeviceScan::ExclusiveSum(vo.tmp.p, tb, vo.lens.as<uint32_t>(), vo.offs.as<uint32_t>(), (int)n, st);
  varlen_total_kernel<<<1, 1, 0, st>>>(vo.lens.as<uint32_t>(), vo.offs.as<uint32_t>(), n);
  RW_CUDA(cudaGetLastError());
  uint32_t total = 0;
  RW_CUDA(cudaMemcpyAsync(&total, vo.offs.as<uint32_t>() + n, 4, cudaMemcpyDeviceToHost, st));
  RW_CUDA(cudaStreamSynchronize(st));
  vo.total = total;
  RW_CUDA(vo.bytes.reserve((size_t)total + 16));
  if (total) {
    varlen_gather_kernel<<<jgrid(n, 256), 256, 0, st>>>(handles, vo.offs.as<uint32_t>(), n, h->var_heap[0].as<uint8_t>(), h->var_heap[1].as<uint8_t>(),
                                                         vo.bytes.as<uint8_t>());
    RW_CUDA(cudaGetLastError());
  }
  h->launches += 4;
  return RW_OK;
}

// device chunk with varlen columns (rw_chunk pointers are DEVICE pointers): intern them, point the DevChunk at the handles
static int var_intern_device_chunk(rwgpu_join* h, int side, const rw_chunk* c, DevChunk* ch, cudaStream_t st) {
  if (h->var_in[side].empty()) return RW_OK;
  if (ch->n_dev) return fail(RW_ERR_UNSUPPORTED, "a device-resident row count with varlen columns");
  const int64_t n = c->n_rows;
  for (int k : h->var_in[side]) {
    if (n && !c->columns[k].offsets) return fail(RW_ERR_INVALID, "varlen column without offsets");
    uint32_t o0 = 0, o1 = 0;
    if (n) {
      RW_CUDA(cudaMemcpyAsync(&o0, c->columns[k].offsets, 4, cudaMemcpyDeviceToHost, st));
      RW_CUDA(cudaMemcpyAsync(&o1, c->columns[k].offsets + n, 4, cudaMemcpyDeviceToHost, st));
      RW_CUDA(cudaStreamSynchronize(st));
    }
    int rc = var_ensure_heap(h, side, (uint64_t)(o1 - o0) + 8ull * (uint64_t)n);
    if (rc != RW_OK) return rc;
    h->var_upper[side] += (uint64_t)(o1 - o0) + 8ull * (uint64_t)n;
    RW_CUDA(h->var_handles[k].reserve((size_t)std::max<int64_t>(n, 1) * 8));
    rc = var_intern(h, side, (const uint8_t*)c->columns[k].data, c->columns[k].offsets, c->ops, c->visibility, c->columns[k].validity, n,
                    h->var_handles[k].as<uint64_t>(), st);
    if (rc != RW_OK) return rc;
    ch->cols[k].data = h->var_handles[k].p;
  }
  return var_check_err(h, st);
}

// JoinChunkBuilder::post_process (join/builder.rs:166-168): eliminate_adjacent_noop_update on what the call emitted.
// Only a call that saw Delete rows can have emitted a Delete / Insert pair.
static int join_post_process(rwgpu_join* h, int64_t n, unsigned long long* nullm, cudaStream_t st) {
  if (!h->call_had_deletes || n < 2) return RW_OK;
  bool hid = false;
  int rc = join_eliminate_noop(h, n, !h->call_vis_stale, st, &hid);
  if (rc != RW_OK) return rc;
  if (hid) *nullm |= 1ull << 63;
  return RW_OK;
}

// device view of the current output set's first n rows (bitmaps are packed on `st` where NULLs / holes exist)
static int join_fill_view(rwgpu_join* h, int64_t n, unsigned long long nullm, rw_chunk* view, cudaStream_t st) {
  std::vector<rw_column>& cols = h->dev_view_cols[h->cur];
  cols.resize(h->out_types.size());
  for (size_t k = 0; k < h->out_types.size(); k++) {
    rw_column& col = cols[k];
    col.type = h->out_types[k];
    col.reserved = 0;
    col.data = h->os().out_col[k].p;
    col.validity = nullptr;
    col.offsets = nullptr;
    if (type_is_varlen(h->out_types[k])) {  // handles -> offsets + bytes (device)
      rwgpu_join::VarOut& vo = h->vout[h->cur][k];
      int rc = var_materialize(h, vo, h->os().out_col[k].as<uint64_t>(), (nullm >> 63) ? h->os().out_vis.as<uint8_t>() : nullptr,
                               ((nullm >> k) & 1) ? h->os().out_valid[k].as<uint8_t>() : nullptr, n, st);
      if (rc != RW_OK) return rc;
      col.data = vo.bytes.p;
      col.offsets = vo.offs.as<uint32_t>();
    }
    if (((nullm >> k) & 1) && n > 0) {
      pack_bytes_to_bits_kernel<<<jgrid((n + 63) / 64, 256), 256, 0, st>>>(h->os().out_valid[k].as<uint8_t>(), h->os().out_bits[k].as<uint64_t>(), n);
      RW_CUDA(cudaGetLastError());
      col.validity = h->os().out_bits[k].as<uint64_t>();
    }
  }
  view->n_rows = n;
  view->n_cols = (int32_t)h->out_types.size();
  view->reserved = 0;
  view->ops = h->os().out_ops.as<uint8_t>();
  view->visibility = nullptr;
  if ((nullm >> 63) && n > 0) {
    pack_bytes_to_bits_kernel<<<jgrid((n + 63) / 64, 256), 256, 0, st>>>(h->os().out_vis.as<uint8_t>(), h->os().out_visbits.as<uint64_t>(), n);
    RW_CUDA(cudaGetLastError());
    view->visibility = h->os().out_visbits.as<uint64_t>();
  }
  view->columns = cols.data();
  return RW_OK;
}

int32_t rwgpu_join_push_device_counted(rwgpu_join* h, int32_t side, const rw_chunk* c, const int64_t* n_rows_dev, rw_chunk* view,
                                       void* cuda_stream) {
  if (!h || !c || !view) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (c->n_cols != h->side[side].n_cols) return fail(RW_ERR_INVALID, "chunk schema mismatch");
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes first");
  DevChunk ch;
  int rc = devchunk_from_abi(c, &ch);
  if (rc != RW_OK) return rc;
  ch.n_dev = n_rows_dev;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
  int64_t n = 0;
  unsigned long long nullm = 0;
  rc = join_begin_call(h, st);
  if (rc != RW_OK) return rc;
  rc = var_intern_device_chunk(h, side, c, &ch, st);
  if (rc != RW_OK) return rc;
  rc = join_push_dev(h, side, ch, st, 0, &n, &nullm);
  if (rc != RW_OK) return rc;
  rc = join_post_process(h, n, &nullm, st);
  if (rc != RW_OK) return rc;
  return join_fill_view(h, n, nullm, view, st);
}

// LAUNCH half (see rwgpu.h).  Unified-table handles really only enqueue; other plan shapes run the push to
// completion here and hand the result over at collect time, so callers need not care which kind they hold.
int32_t rwgpu_join_push_device_async(rwgpu_join* h, int32_t side, const rw_chunk* c, const int64_t* n_rows_dev, void* cuda_stream) {
  if (!h || !c) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (c->n_cols != h->side[side].n_cols) return fail(RW_ERR_INVALID, "chunk schema mismatch");
  if (h->n_pending >= 2) return fail(RW_ERR_INVALID, "two pushes are already outstanding: collect one first");
  if (h->n_pending && h->pending[0].S != side)
    return fail(RW_ERR_INVALID, "pushes of different sides cannot be outstanding together: collect first");
  DevChunk ch;
  int rc = devchunk_from_abi(c, &ch);
  if (rc != RW_OK) return rc;
  ch.n_dev = n_rows_dev;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
  h->cur = h->n_pending ? 1 - h->pending[h->n_pending - 1].set : h->cur;
  rc = join_begin_call(h, st);
  if (rc != RW_OK) return rc;
  JoinPending pd;
  rc = var_intern_device_chunk(h, side, c, &ch, st);
  if (rc != RW_OK) return rc;
  if (h->uni && ch.n > 0 && ch.n < (1ll << 31) && h->var_in[side].empty()) {
    rc = uni_enqueue(h, side, ch, st, 0, &pd);
    if (rc != RW_OK) return rc;
  } else {
    pd.S = side;
    pd.set = h->cur;
    pd.st = st;
    pd.sync_done = true;
    rc = join_push_dev(h, side, ch, st, 0, &pd.rows, &pd.nullm);
    if (rc != RW_OK) return rc;
    rc = join_post_process(h, pd.rows, &pd.nullm, st);
    if (rc != RW_OK) return rc;
  }
  h->pending[h->n_pending++] = pd;
  return RW_OK;
}

int32_t rwgpu_join_collect(rwgpu_join* h, rw_chunk* view, void* cuda_stream) {
  if (!h || !view) return fail(RW_ERR_INVALID, "null");
  if (h->n_pending == 0) return fail(RW_ERR_INVALID, "no push outstanding");
  const JoinPending pd = h->pending[0];
  if (h->hpend[pd.set].active) return fail(RW_ERR_INVALID, "the oldest outstanding push was launched with a host chunk: use rwgpu_join_collect_out");
  h->pending[0] = h->pending[1];
  h->n_pending--;
  h->cur = pd.set;
  int64_t n = pd.rows;
  unsigned long long nullm = pd.nullm;
  if (!pd.sync_done) {
    h->call_null_mask = 0;
    h->call_had_deletes = false;
    int rc = uni_finish(h, pd, &n, &nullm);
    if (rc != RW_OK) return rc;
    const double tp0 = uni_trace ? uni_now_ms() : 0.0;
    rc = join_post_process(h, n, &nullm, pd.st);
    if (rc != RW_OK) return rc;
    if (uni_trace) fprintf(stderr, "  [collect] post-process (no-op elimination: %d) %.3f ms\n", (int)h->call_had_deletes, uni_now_ms() - tp0);
  }
  int rc = join_fill_view(h, n, nullm, view, cuda_stream ? (cudaStream_t)cuda_stream : pd.st);
  // the next synchronous push must not land in the set a still-outstanding push writes to
  if (h->n_pending) h->cur = h->pending[h->n_pending - 1].set;
  return rc;
}

// HOST chunk.  Large chunks are cut into sub-batches (multiples of 64 rows, so bitmap words split
// cleanly) that flow through three streams: H2D of sub-batch j+1 overlaps the kernels of j and the
// D2H of j-1.  Sub-batches are ordinary consecutive pushes, so the operator semantics are unchanged;
// their outputs land back to back in one device buffer and one pinned host block.
int32_t rwgpu_join_push(rwgpu_join* h, int32_t side, const rw_chunk* c, rwgpu_out** out) {
  if (!h || !c || !out) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (c->n_cols != h->side[side].n_cols) return fail(RW_ERR_INVALID, "chunk schema mismatch");
  for (int k = 0; k < c->n_cols; k++)
    if (c->columns[k].type != h->side[side].types[k]) return fail(RW_ERR_INVALID, "chunk column type mismatch");
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes first");
  const int64_t n = c->n_rows;
  static const bool trace = getenv("RWGPU_TRACE") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  if (!h->s_h2d) {
    RW_CUDA(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    RW_CUDA(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) {
      RW_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
      RW_CUDA(cudaEventCreateWithFlags(&h->ev_main[i], cudaEventDisableTiming));
    }
  }
  // each sub-batch costs one status read-back (~40 us): keep them >= 32K rows
  const int J = n >= (1 << 19) ? 8 : (n >= (1 << 17) ? 4 : (n >= (1 << 16) ? 2 : 1));
  int64_t sub = (n + J - 1) / J;
  sub = (sub + 63) / 64 * 64;
  // device staging: [ops | vis words | per column: data, valid words], regions sized for the whole chunk
  const size_t nw = (size_t)((n + 63) / 64) * 8;
  size_t off = 0;
  auto region = [&](size_t bytes) { size_t o = align_up_j(off, 256); off = o + bytes; return o; };
  const size_t o_ops = region((size_t)n), o_vis = region(nw);
  size_t o_data[RW_MAX_COLS], o_valid[RW_MAX_COLS], o_voff[RW_MAX_COLS], o_vbytes[RW_MAX_COLS];
  uint64_t var_bytes_in = 0;  // bytes of the chunk's varlen columns (interned into the side's heap below)
  for (int k = 0; k < c->n_cols; k++) {
    o_data[k] = region((size_t)n * type_width(c->columns[k].type));  // (varlen: the 8-byte handles)
    o_valid[k] = region(nw);
    o_voff[k] = o_vbytes[k] = 0;
    if (type_is_varlen(c->columns[k].type)) {
      if (n && !c->columns[k].offsets) return fail(RW_ERR_INVALID, "varlen column without offsets");
      const size_t vb = n ? (size_t)(c->columns[k].offsets[n] - c->columns[k].offsets[0]) : 0;
      o_voff[k] = region((size_t)(n + 1) * 4);
      o_vbytes[k] = region(vb + 16);
      var_bytes_in += vb + 8ull * (uint64_t)n;
    }
  }
  if (var_bytes_in) {
    int rcv = var_ensure_heap(h, side, var_bytes_in);
    if (rcv != RW_OK) return rcv;
    h->var_upper[side] += var_bytes_in;
  }
  RW_CUDA(h->up.reserve(off + 256));
  RW_CUDA(h->up_host.reserve(off + 256));
  uint8_t* hp = h->up_host.as<uint8_t>();
  uint8_t* dp = h->up.as<uint8_t>();
  // a caller buffer that is already pinned is copied straight from user memory; pageable small
  // pieces go through the pinned staging block (one memcpy), pageable large ones directly
  auto is_pinned = [](const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
  };
  auto h2d = [&](size_t dst_off, const void* src, size_t bytes, bool pinned) {
    if (!bytes) return;
    if (pinned || bytes >= (1u << 20)) cudaMemcpyAsync(dp + dst_off, src, bytes, cudaMemcpyHostToDevice, h->s_h2d);
    else { memcpy(hp + dst_off, src, bytes); cudaMemcpyAsync(dp + dst_off, hp + dst_off, bytes, cudaMemcpyHostToDevice, h->s_h2d); }
  };
  RW_CUDA(cudaStreamSynchronize(h->s_d2h));  // previous call's copies are long done; cheap guard for buffer reuse
  bool pin_ops = n ? is_pinned(c->ops) : false, pin_col[RW_MAX_COLS];
  for (int k = 0; k < c->n_cols; k++) pin_col[k] = n ? is_pinned(c->columns[k].data) : false;
  // enqueue every sub-batch's H2D up front
  int n_sub = 0;
  for (int64_t lo = 0; lo < n; lo += sub, n_sub++) {
    const int64_t m = std::min<int64_t>(sub, n - lo);
    const size_t wlo = (size_t)(lo / 64) * 8, wn = (size_t)((m + 63) / 64) * 8;
    h2d(o_ops + (size_t)lo, c->ops + lo, (size_t)m, pin_ops);
    if (c->visibility) h2d(o_vis + wlo, (const uint8_t*)c->visibility + wlo, wn, false);
    for (int k = 0; k < c->n_cols; k++) {
      const int w = type_width(c->columns[k].type);
      if (type_is_varlen(c->columns[k].type)) {  // offsets lo .. lo+m and the bytes they span
        const uint32_t* of = c->columns[k].offsets;
        h2d(o_voff[k] + (size_t)lo * 4, of + lo, (size_t)(m + 1) * 4, false);
        h2d(o_vbytes[k] + (size_t)(of[lo] - of[0]), (const uint8_t*)c->columns[k].data + of[lo], (size_t)(of[lo + m] - of[lo]), pin_col[k]);
      } else {
        h2d(o_data[k] + (size_t)lo * w, (const uint8_t*)c->columns[k].data + (size_t)lo * w, (size_t)m * w, pin_col[k]);
      }
      if (c->columns[k].validity) h2d(o_valid[k] + wlo, (const uint8_t*)c->columns[k].validity + wlo, wn, false);
    }
    RW_CUDA(cudaEventRecord(h->ev_h2d[n_sub], h->s_h2d));
  }
  RW_CUDA(cudaGetLastError());
  const double t1 = now();
  int rc = join_begin_call(h, h->stream);
  if (rc != RW_OK) return rc;
  auto o = new rwgpu_out();
  std::unique_ptr<rwgpu_out> guard(o);
  o->chunk_size = h->chunk_size;
  // pinned host block laid out for `host_cap` rows; re-laid (host copy of the prefix) if outputs exceed it
  int64_t host_cap = std::max<int64_t>(2 * n, 1024);
  if (!o->layout(host_cap, h->out_types, ~0ull >> 1, true, h->pool)) return fail(RW_ERR_OOM, "pinned output block");
  // Positional inner-join output (row r of the output = input row r): the update side's output columns are
  // byte-for-byte the caller's input columns, which already sit in host memory -- they are not copied back
  // over PCIe; the output chunk views alias the input buffers instead (contract in rwgpu.h).
  static const bool no_alias = getenv("RWGPU_NO_ALIAS") != nullptr;
  bool alias_ok = !no_alias && h->fast_inner && h->w8_ok[side] && !c->visibility && n > 0;
  for (int k = 0; k < c->n_cols && alias_ok; k++) alias_ok = c->columns[k].validity == nullptr;
  std::vector<int> alias_src(h->out_types.size(), -1);
  if (alias_ok)
    for (int k = 0; k < c->n_cols; k++)
      if (h->w8[side].u_out[k] >= 0 && !type_is_varlen(c->columns[k].type)) alias_src[(size_t)h->w8[side].u_out[k]] = k;
  bool aligned = true;  // every sub-batch produced exactly its positional rows (no extras, no empty result)
  int64_t total = 0;
  unsigned long long nullm = 0;
  int js = 0;
  const double t2 = now();
  for (int64_t lo = 0; lo < n; lo += sub, js++) {
    const int64_t m = std::min<int64_t>(sub, n - lo);
    DevChunk ch;
    memset(&ch, 0, sizeof(ch));
    ch.n = m;
    ch.n_cols = c->n_cols;
    ch.ops = dp + o_ops + lo;
    ch.vis_bits = c->visibility ? (const uint64_t*)(dp + o_vis + (size_t)(lo / 64) * 8) : nullptr;
    for (int k = 0; k < c->n_cols; k++) {
      const int w = type_width(c->columns[k].type);
      ch.cols[k].type = c->columns[k].type;
      ch.cols[k].width = w;
      ch.cols[k].data = dp + o_data[k] + (size_t)lo * w;
      ch.cols[k].valid_bits = c->columns[k].validity ? (const uint64_t*)(dp + o_valid[k] + (size_t)(lo / 64) * 8) : nullptr;
    }
    double ta = 0, tb = 0;
    if (trace) { ta = now(); cudaEventSynchronize(h->ev_h2d[js]); tb = now(); }
    RW_CUDA(cudaStreamWaitEvent(h->stream, h->ev_h2d[js], 0));
    for (int k : h->var_in[side]) {  // bytes -> the side's heap, the column becomes a column of handles
      rc = var_intern(h, side, dp + o_vbytes[k] - c->columns[k].offsets[0], (const uint32_t*)(dp + o_voff[k]) + lo, ch.ops, ch.vis_bits,
                      ch.cols[k].valid_bits, m, (uint64_t*)(dp + o_data[k]) + lo, h->stream);
      if (rc != RW_OK) { cudaStreamSynchronize(h->s_d2h); return rc; }
    }
    int64_t rows = 0;
    rc = join_push_dev(h, side, ch, h->stream, total, &rows, &nullm);
    if (trace) fprintf(stderr, "   sub %d: wait-h2d %.3f  push_dev %.3f ms\n", js, tb - ta, now() - tb);
    if (rc != RW_OK) { cudaStreamSynchronize(h->s_d2h); return rc; }
    aligned = aligned && rows == m;
    if (total + rows > host_cap) {  // rare: amplification above 2x -- grow the host block, keep the copied prefix
      RW_CUDA(cudaStreamSynchronize(h->s_d2h));
      auto o2 = new rwgpu_out();
      o2->chunk_size = h->chunk_size;
      const int64_t ncap = (total + rows) * 2;
      if (!o2->layout(ncap, h->out_types, ~0ull >> 1, true, h->pool)) { delete o2; return fail(RW_ERR_OOM, "pinned output block"); }
      if (total > 0) {
        memcpy(o2->ops, o->ops, (size_t)total);
        for (size_t k = 0; k < h->out_types.size(); k++)
          if (!type_is_varlen(h->out_types[k])) memcpy(o2->data[k], o->data[k], (size_t)total * type_width(h->out_types[k]));
      }
      guard.reset(o2);
      o = o2;
      host_cap = ncap;
    }
    if (rows > 0) {
      RW_CUDA(cudaEventRecord(h->ev_main[js], h->stream));
      RW_CUDA(cudaStreamWaitEvent(h->s_d2h, h->ev_main[js], 0));
      cudaMemcpyAsync(o->ops + total, h->os().out_ops.as<uint8_t>() + total, (size_t)rows, cudaMemcpyDeviceToHost, h->s_d2h);
      for (size_t k = 0; k < h->out_types.size(); k++) {
        if (alias_src[k] >= 0) continue;  // decided after the last sub-batch
        if (type_is_varlen(h->out_types[k])) continue;  // materialised after the last sub-batch
        const size_t w = type_width(h->out_types[k]);
        cudaMemcpyAsync(o->data[k] + (size_t)total * w, h->os().out_col[k].as<uint8_t>() + (size_t)total * w, (size_t)rows * w,
                        cudaMemcpyDeviceToHost, h->s_d2h);
      }
    }
    total += rows;
  }
  rc = join_post_process(h, total, &nullm, h->stream);
  if (rc != RW_OK) { cudaStreamSynchronize(h->s_d2h); return rc; }
  if (!h->var_in[side].empty()) {
    rc = var_check_err(h, h->stream);
    if (rc != RW_OK) { cudaStreamSynchronize(h->s_d2h); return rc; }
  }
  for (int k : h->var_out) {  // handles -> offsets + bytes, then to the host
    rwgpu_join::VarOut& vo = h->vout[h->cur][k];
    rc = var_materialize(h, vo, h->os().out_col[k].as<uint64_t>(), (nullm >> 63) ? h->os().out_vis.as<uint8_t>() : nullptr,
                         ((nullm >> k) & 1) ? h->os().out_valid[k].as<uint8_t>() : nullptr, total, h->stream);
    if (rc != RW_OK) { cudaStreamSynchronize(h->s_d2h); return rc; }
    uint8_t* hb = o->var_bytes((size_t)k, vo.total);
    if (!hb) { cudaStreamSynchronize(h->s_d2h); return fail(RW_ERR_OOM, "pinned varlen output"); }
    RW_CUDA(cudaMemcpyAsync(o->offsets[k], vo.offs.p, (size_t)(total + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
    if (vo.total) RW_CUDA(cudaMemcpyAsync(hb, vo.bytes.p, vo.total, cudaMemcpyDeviceToHost, h->stream));
  }
  for (size_t k = 0; k < h->out_types.size(); k++) {
    if (alias_src[k] < 0) continue;
    if (aligned && total == n) {
      o->data[k] = (uint8_t*)const_cast<void*>(c->columns[alias_src[k]].data);  // zero-copy: the caller's input column
    } else if (total > 0) {  // extra matches or an empty sub-batch broke the row alignment: ordinary copy
      // (every sub-batch's kernels have completed: join_push_dev synchronises on its status read-back)
      cudaMemcpyAsync(o->data[k], h->os().out_col[k].p, (size_t)total * type_width(h->out_types[k]), cudaMemcpyDeviceToHost, h->s_d2h);
    }
  }
  // NULL / visibility bytes only for the columns that need them (known once all sub-batches ran)
  if (total > 0) {
    if (nullm >> 63) cudaMemcpyAsync(o->vis_bytes, h->os().out_vis.p, (size_t)total, cudaMemcpyDeviceToHost, h->s_d2h);
    for (size_t k = 0; k < h->out_types.size(); k++)
      if ((nullm >> k) & 1) cudaMemcpyAsync(o->valid_bytes[k], h->os().out_valid[k].p, (size_t)total, cudaMemcpyDeviceToHost, h->s_d2h);
  }
  const double t3 = now();
  RW_CUDA(cudaStreamSynchronize(h->stream));
  RW_CUDA(cudaStreamSynchronize(h->s_d2h));
  RW_CUDA(cudaStreamSynchronize(h->s_h2d));
  const double t4 = now();
  o->n_rows = total;
  if (!(nullm >> 63)) o->vis_bytes = nullptr;
  for (size_t k = 0; k < h->out_types.size(); k++)
    if (!((nullm >> k) & 1)) o->valid_bytes[k] = nullptr;
  o->finalize();
  if (trace)
    fprintf(stderr, "[rwgpu_join_push] n=%lld out=%lld J=%d  h2d-enqueue %.3f  layout %.3f  sub-batches %.3f  drain %.3f  finalize %.3f  total %.3f ms\n",
            (long long)n, (long long)total, n_sub, t1 - t0, t2 - t1, t3 - t2, t4 - t3, now() - t4, now() - t0);
  *out = guard.release();
  return RW_OK;
}

// ---- launch / collect split for HOST chunks.  rwgpu_join_push handles one chunk per call and returns when its output
// sits in host memory: H2D, kernels and D2H of ONE call overlap (sub-batches), consecutive calls do not.  Here the call
// only ENQUEUES: input H2D on the copy-in stream, the push on the main stream, and -- the common case being one output
// row per input row -- the D2H of the positional rows on the copy-out stream.  While the caller launches chunk s+1
// (its H2D uses the other PCIe direction), chunk s's output streams back; collect waits, copies what the status block
// says is still missing (extra matches, NULL / visibility bytes) and cuts the chunk views.
int32_t rwgpu_join_push_async(rwgpu_join* h, int32_t side, const rw_chunk* c) {
  if (!h || !c) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (c->n_cols != h->side[side].n_cols) return fail(RW_ERR_INVALID, "chunk schema mismatch");
  for (int k = 0; k < c->n_cols; k++)
    if (c->columns[k].type != h->side[side].types[k]) return fail(RW_ERR_INVALID, "chunk column type mismatch");
  if (h->n_pending >= 2) return fail(RW_ERR_INVALID, "two pushes are already outstanding: collect one first");
  if (h->n_pending && h->pending[0].S != side)
    return fail(RW_ERR_INVALID, "pushes of different sides cannot be outstanding together: collect first");
  const int64_t n = c->n_rows;
  const int set = h->n_pending ? 1 - h->pending[h->n_pending - 1].set : h->cur;
  rwgpu_join::HostPending& hp = h->hpend[set];
  if (hp.active) return fail(RW_ERR_INVALID, "output set still holds an uncollected host push");
  hp = rwgpu_join::HostPending();
  hp.active = true;
  hp.n = n;
  hp.in = *c;
  hp.in_cols.assign(c->columns, c->columns + c->n_cols);
  hp.in.columns = hp.in_cols.data();
  JoinPending pd;
  pd.S = side;
  pd.set = set;
  pd.st = h->stream;
  bool simple = h->uni && n > 0 && n < (1ll << 31) && h->var_in[side].empty() && h->var_out.empty();
  if (!simple) {
    // other plan shapes / varlen payload / empty chunks: run the synchronous call now, hand the result over at collect
    if (h->n_pending) return fail(RW_ERR_INVALID, "this join shape runs its pushes synchronously: collect the outstanding push first");
    hp.active = false;
    rwgpu_out* o = nullptr;
    int rc = rwgpu_join_push(h, side, c, &o);
    if (rc != RW_OK) return rc;
    hp.active = true;
    hp.sync_done = true;
    hp.out = o;
    pd.sync_done = true;  // (nothing is outstanding: `set` is the current set)
    h->pending[h->n_pending++] = pd;
    return RW_OK;
  }
  if (!h->s_h2d) {
    RW_CUDA(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    RW_CUDA(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) {
      RW_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
      RW_CUDA(cudaEventCreateWithFlags(&h->ev_main[i], cudaEventDisableTiming));
    }
  }
  if (!h->ev_up2[set]) RW_CUDA(cudaEventCreateWithFlags(&h->ev_up2[set], cudaEventDisableTiming));
  if (!h->s_out[set]) RW_CUDA(cudaStreamCreateWithFlags(&h->s_out[set], cudaStreamNonBlocking));
  cudaStream_t sd = h->s_out[set];
  // ---- input: device staging of this set
  const size_t nw = (size_t)((n + 63) / 64) * 8;
  size_t off = 0;
  auto region = [&](size_t bytes) { size_t o = align_up_j(off, 256); off = o + bytes; return o; };
  const size_t o_ops = region((size_t)n), o_vis = region(nw);
  size_t o_data[RW_MAX_COLS], o_valid[RW_MAX_COLS];
  for (int k = 0; k < c->n_cols; k++) {
    o_data[k] = region((size_t)n * type_width(c->columns[k].type));
    o_valid[k] = region(nw);
  }
  if (off + 256 > h->up2[set].bytes) {
    RW_CUDA(cudaDeviceSynchronize());  // (growth only)
    RW_CUDA(h->up2[set].reserve(off + off / 4 + 256));
    RW_CUDA(h->up2_host[set].reserve(off + off / 4 + 256));
  }
  uint8_t* hs = h->up2_host[set].as<uint8_t>();
  uint8_t* dp = h->up2[set].as<uint8_t>();
  auto is_pinned = [](const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
  };
  // (the copy-in stream is ordered behind the kernels that read this staging two pushes ago: that push was collected)
  auto h2d = [&](size_t dst_off, const void* src, size_t bytes, bool pinned) {
    if (!bytes) return;
    if (pinned || bytes >= (1u << 20)) cudaMemcpyAsync(dp + dst_off, src, bytes, cudaMemcpyHostToDevice, h->s_h2d);
    else { memcpy(hs + dst_off, src, bytes); cudaMemcpyAsync(dp + dst_off, hs + dst_off, bytes, cudaMemcpyHostToDevice, h->s_h2d); }
  };
  h2d(o_ops, c->ops, (size_t)n, is_pinned(c->ops));
  if (c->visibility) h2d(o_vis, c->visibility, nw, false);
  for (int k = 0; k < c->n_cols; k++) {
    h2d(o_data[k], c->columns[k].data, (size_t)n * type_width(c->columns[k].type), is_pinned(c->columns[k].data));
    if (c->columns[k].validity) h2d(o_valid[k], c->columns[k].validity, nw, false);
  }
  RW_CUDA(cudaEventRecord(h->ev_up2[set], h->s_h2d));
  RW_CUDA(cudaGetLastError());
  DevChunk ch;
  memset(&ch, 0, sizeof(ch));
  ch.n = n;
  ch.n_cols = c->n_cols;
  ch.ops = dp + o_ops;
  ch.vis_bits = c->visibility ? (const uint64_t*)(dp + o_vis) : nullptr;
  for (int k = 0; k < c->n_cols; k++) {
    ch.cols[k].type = c->columns[k].type;
    ch.cols[k].width = type_width(c->columns[k].type);
    ch.cols[k].data = dp + o_data[k];
    ch.cols[k].valid_bits = c->columns[k].validity ? (const uint64_t*)(dp + o_valid[k]) : nullptr;
  }
  // ---- the push
  h->cur = set;
  int rc = join_begin_call(h, h->stream);
  if (rc != RW_OK) { hp.active = false; return rc; }
  RW_CUDA(cudaStreamWaitEvent(h->stream, h->ev_up2[set], 0));
  rc = uni_enqueue(h, side, ch, h->stream, 0, &pd);
  if (rc != RW_OK) { hp.active = false; return rc; }
  // ---- output block + the copy-out of the positional rows
  auto o = new rwgpu_out();
  o->chunk_size = h->chunk_size;
  hp.host_cap = std::max<int64_t>(2 * n, 1024);
  if (!o->layout(hp.host_cap, h->out_types, ~0ull >> 1, true, h->pool)) { delete o; hp.active = false; return fail(RW_ERR_OOM, "pinned output block"); }
  hp.out = o;
  static const bool no_alias = getenv("RWGPU_NO_ALIAS") != nullptr;
  hp.alias_ok = !no_alias && h->w8_ok[side] && !c->visibility;
  for (int k = 0; k < c->n_cols && hp.alias_ok; k++) hp.alias_ok = c->columns[k].validity == nullptr;
  hp.alias_src.assign(h->out_types.size(), -1);
  if (hp.alias_ok)
    for (int k = 0; k < c->n_cols; k++)
      if (h->w8[side].u_out[k] >= 0) hp.alias_src[(size_t)h->w8[side].u_out[k]] = k;
  RW_CUDA(cudaStreamWaitEvent(sd, h->pend_ev[set], 0));
  cudaMemcpyAsync(o->ops, h->os().out_ops.p, (size_t)n, cudaMemcpyDeviceToHost, sd);
  for (size_t k = 0; k < h->out_types.size(); k++) {
    if (hp.alias_src[k] >= 0) continue;
    const size_t w = type_width(h->out_types[k]);
    cudaMemcpyAsync(o->data[k], h->os().out_col[k].p, (size_t)n * w, cudaMemcpyDeviceToHost, sd);
  }
  RW_CUDA(cudaGetLastError());
  h->pending[h->n_pending++] = pd;
  return RW_OK;
}

int32_t rwgpu_join_collect_out(rwgpu_join* h, rwgpu_out** out) {
  if (!h || !out) return fail(RW_ERR_INVALID, "null");
  if (h->n_pending == 0) return fail(RW_ERR_INVALID, "no push outstanding");
  const JoinPending pd = h->pending[0];
  rwgpu_join::HostPending& hp = h->hpend[pd.set];
  if (!hp.active) return fail(RW_ERR_INVALID, "the oldest outstanding push was launched with a device chunk: use rwgpu_join_collect");
  h->pending[0] = h->pending[1];
  h->n_pending--;
  hp.active = false;
  if (hp.sync_done) {
    *out = hp.out;
    hp.out = nullptr;
    return RW_OK;
  }
  std::unique_ptr<rwgpu_out> guard(hp.out);
  hp.out = nullptr;
  rwgpu_out* o = guard.get();
  cudaStream_t sd = h->s_out[pd.set];
  h->cur = pd.set;
  h->call_null_mask = 0;
  h->call_had_deletes = false;
  int64_t total = 0;
  unsigned long long nullm = 0;
  const uint8_t* ops_before = h->os().out_ops.as<uint8_t>();
  auto bail = [&](int rc) { cudaStreamSynchronize(sd); if (h->n_pending) h->cur = h->pending[h->n_pending - 1].set; return rc; };
  int rc = uni_finish(h, pd, &total, &nullm);
  if (rc != RW_OK) return bail(rc);
  rc = join_post_process(h, total, &nullm, pd.st);
  if (rc != RW_OK) return bail(rc);
  const int64_t n = hp.n;
  // what the launch already copied is good unless the emission was redone into re-allocated buffers
  bool pre_ok = h->os().out_ops.as<uint8_t>() == ops_before && total >= n;
  if (total > hp.host_cap) {  // rare: amplification above 2x -- a larger host block, everything is copied again
    RW_CUDA(cudaStreamSynchronize(sd));
    auto o2 = new rwgpu_out();
    o2->chunk_size = h->chunk_size;
    if (!o2->layout(total + total / 4, h->out_types, ~0ull >> 1, true, h->pool)) { delete o2; return bail(fail(RW_ERR_OOM, "pinned output block")); }
    guard.reset(o2);
    o = o2;
    pre_ok = false;
  }
  const bool aligned = total == n;  // exactly the positional rows: the update side's columns ARE the caller's input columns
  if (total > 0) {
    const int64_t from = pre_ok ? n : 0;  // rows [0, n) of the non-aliased columns are already on their way
    const int64_t ops_from = h->call_had_deletes ? 0 : from;  // (the no-op elimination pass may have rewritten ops)
    if (total > ops_from)
      cudaMemcpyAsync(o->ops + ops_from, h->os().out_ops.as<uint8_t>() + ops_from, (size_t)(total - ops_from), cudaMemcpyDeviceToHost, sd);
    for (size_t k = 0; k < h->out_types.size(); k++) {
      const size_t w = type_width(h->out_types[k]);
      if (hp.alias_src[k] >= 0) {
        if (aligned) o->data[k] = (uint8_t*)const_cast<void*>(hp.in_cols[(size_t)hp.alias_src[k]].data);  // zero-copy
        else cudaMemcpyAsync(o->data[k], h->os().out_col[k].p, (size_t)total * w, cudaMemcpyDeviceToHost, sd);
      } else if (total > from) {
        cudaMemcpyAsync(o->data[k] + (size_t)from * w, h->os().out_col[k].as<uint8_t>() + (size_t)from * w, (size_t)(total - from) * w,
                        cudaMemcpyDeviceToHost, sd);
      }
    }
    if (nullm >> 63) cudaMemcpyAsync(o->vis_bytes, h->os().out_vis.p, (size_t)total, cudaMemcpyDeviceToHost, sd);
    for (size_t k = 0; k < h->out_types.size(); k++)
      if ((nullm >> k) & 1) cudaMemcpyAsync(o->valid_bytes[k], h->os().out_valid[k].p, (size_t)total, cudaMemcpyDeviceToHost, sd);
  }
  RW_CUDA(cudaStreamSynchronize(sd));
  o->n_rows = total;
  if (!(nullm >> 63)) o->vis_bytes = nullptr;
  for (size_t k = 0; k < h->out_types.size(); k++)
    if (!((nullm >> k) & 1)) o->valid_bytes[k] = nullptr;
  o->finalize();
  if (h->n_pending) h->cur = h->pending[h->n_pending - 1].set;
  *out = guard.release();
  return RW_OK;
}

int32_t rwgpu_join_barrier(rwgpu_join* h, uint64_t /*epoch*/) {
  if (!h) return fail(RW_ERR_INVALID, "null");
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes before the barrier");
  // state lives in HBM (StateStore stubbed to memory, north_star): a barrier is an ordering point
  RW_CUDA(cudaStreamSynchronize(h->stream));
  if (h->last_st && h->last_st != h->stream) RW_CUDA(cudaStreamSynchronize(h->last_st));
  // watermark-driven state cleaning (hash_join.rs:791-891 -> JoinHashMap::update_watermark; the state table drops the
  // range below the watermark when the epoch commits)
  for (int s = 0; s < 2; s++) {
    if (!h->wm_pending[s]) continue;
    h->wm_pending[s] = false;
    if (h->uni) uni_clean_kernel<<<jgrid((int64_t)h->uni_cap + 2, 256), 256, 0, h->stream>>>(uni_dev(h), s, (long long)h->wm_value[s]);
    else join_clean_kernel<<<jgrid((int64_t)h->side[s].slot_cap + 2, 256), 256, 0, h->stream>>>(h->plan_dev.as<JoinPlanDev>(), side_dev(h, s),
                                                                                                   h->wm_key_pos[s], (long long)h->wm_value[s]);
    RW_CUDA(cudaGetLastError());
    h->launches++;
    h->wm_cleanings++;
    if (h->uni) {  // the dead count decides about compaction below
      unsigned long long nd = 0;
      RW_CUDA(cudaMemcpyAsync(&nd, h->uni_counters.as<unsigned long long>() + 2 + s, 8, cudaMemcpyDeviceToHost, h->stream));
      RW_CUDA(cudaStreamSynchronize(h->stream));
      h->uni_dead[s] = nd;
    }
  }
  RW_CUDA(cudaStreamSynchronize(h->stream));
  // ... and the point where deleted rows are reclaimed (the reference's delete frees the entry at once,
  // join/hash_join.rs:659-681): a log that is more than half dead is rebuilt from its live records
  if (h->uni)
    for (int s = 0; s < 2; s++)
      if (h->uni_dead[s] >= 4096 && h->uni_dead[s] * 2 >= h->side[s].n_rows) {
        int rc = uni_compact(h, s);
        if (rc != RW_OK) return rc;
      }
  return RW_OK;
}

int32_t rwgpu_join_update_watermark(rwgpu_join* h, int32_t side, int32_t key_pos, int64_t value) {
  if (!h) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (key_pos < 0 || key_pos >= h->plan.n_keys) return fail(RW_ERR_INVALID, "join key position");
  const int t = h->plan.col_type[side][h->plan.key_col[side][key_pos]];
  if (type_is_float(t) || t == RW_T_BOOL) return fail(RW_ERR_UNSUPPORTED, "watermarks on this key type keep the state (CPU semantics unchanged)");
  if (h->uni && key_pos != 0) return fail(RW_ERR_INVALID, "join key position");
  // a later watermark on the same side only moves up
  if (!h->wm_pending[side] || value > h->wm_value[side] || key_pos != h->wm_key_pos[side]) {
    h->wm_pending[side] = true;
    h->wm_key_pos[side] = key_pos;
    h->wm_value[side] = value;
  }
  return RW_OK;
}

// ---- state persistence: see the comment above uni_snapshot_kernel
int32_t rwgpu_join_snapshot(rwgpu_join* h, int32_t side, rwgpu_out** out) {
  if (!h || !out) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes first");
  RW_CUDA(cudaDeviceSynchronize());
  const JoinSideHost& sd = h->side[side];
  const int n_cols = sd.n_cols;
  // upper bound of the live rows: every log / store record ever handed out + one inline record per key
  const uint64_t keys = h->uni ? h->uni_keys + 2 : sd.keys_upper + 2;
  int64_t cap = (int64_t)std::min<uint64_t>(sd.n_rows + keys, (uint64_t)1 << 40);
  DevBuf counters;
  RW_CUDA(counters.reserve(256));
  std::vector<DevBuf> col(n_cols), val(n_cols);
  SnapOut o;
  int64_t n = 0;
  unsigned int has_null[RW_MAX_COLS];
  for (int attempt = 0; attempt < 2; attempt++) {
    memset(&o, 0, sizeof(o));
    RW_CUDA(cudaMemset(counters.p, 0, 256));
    o.n_rows = counters.as<unsigned long long>();
    o.has_null = (unsigned int*)(o.n_rows + 1);
    o.capacity = cap;
    for (int k = 0; k < n_cols; k++) {
      RW_CUDA(col[k].reserve((size_t)std::max<int64_t>(cap, 1) * type_width(sd.types[k])));
      RW_CUDA(val[k].reserve((size_t)std::max<int64_t>(cap, 1)));
      o.col[k] = col[k].p;
      o.valid[k] = val[k].as<uint8_t>();
    }
    if (h->uni) uni_snapshot_kernel<<<jgrid((int64_t)h->uni_cap + 2, 256), 256, 0, h->stream>>>(uni_dev(h), side, n_cols, o);
    else join_snapshot_kernel<<<jgrid((int64_t)sd.slot_cap + 2, 256), 256, 0, h->stream>>>(h->plan_dev.as<JoinPlanDev>(), side, side_dev(h, side), o);
    RW_CUDA(cudaGetLastError());
    h->launches++;
    unsigned long long cnt = 0;
    RW_CUDA(cudaMemcpyAsync(&cnt, counters.p, 8, cudaMemcpyDeviceToHost, h->stream));
    RW_CUDA(cudaMemcpyAsync(has_null, o.has_null, sizeof(unsigned int) * RW_MAX_COLS, cudaMemcpyDeviceToHost, h->stream));
    RW_CUDA(cudaStreamSynchronize(h->stream));
    n = (int64_t)cnt;
    if (n <= cap) break;
    cap = n;  // (the bound was too small: once more with the exact size)
  }
  auto ro = new rwgpu_out();
  ro->chunk_size = h->chunk_size;
  unsigned long long nullm = 0;
  for (int k = 0; k < n_cols; k++) if (has_null[k]) nullm |= 1ull << k;
  if (!ro->layout(n, sd.types, nullm, false, h->pool)) { delete ro; return fail(RW_ERR_OOM, "pinned output block"); }
  if (n > 0) {
    memset(ro->ops, RW_OP_INSERT, (size_t)n);
    for (int k = 0; k < n_cols; k++) {
      if (type_is_varlen(sd.types[k])) {  // handles -> offsets + bytes
        rwgpu_join::VarOut vo;
        int rcv = var_materialize(h, vo, col[k].as<uint64_t>(), nullptr, has_null[k] ? val[k].as<uint8_t>() : nullptr, n, h->stream);
        if (rcv != RW_OK) { delete ro; return rcv; }
        uint8_t* hb = ro->var_bytes((size_t)k, vo.total);
        if (!hb) { delete ro; return fail(RW_ERR_OOM, "pinned varlen output"); }
        cudaMemcpyAsync(ro->offsets[k], vo.offs.p, (size_t)(n + 1) * 4, cudaMemcpyDeviceToHost, h->stream);
        if (vo.total) cudaMemcpyAsync(hb, vo.bytes.p, vo.total, cudaMemcpyDeviceToHost, h->stream);
        cudaStreamSynchronize(h->stream);  // (vo's device buffers die at the end of this iteration)
      } else {
        cudaMemcpyAsync(ro->data[k], col[k].p, (size_t)n * type_width(sd.types[k]), cudaMemcpyDeviceToHost, h->stream);
      }
      if (ro->valid_bytes[k]) cudaMemcpyAsync(ro->valid_bytes[k], val[k].p, (size_t)n, cudaMemcpyDeviceToHost, h->stream);
    }
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { delete ro; return fail(RW_ERR_CUDA, cudaGetErrorString(e)); }
  }
  ro->finalize();
  *out = ro;
  return RW_OK;
}

int32_t rwgpu_join_push(rwgpu_join* h, int32_t side, const rw_chunk* c, rwgpu_out** out);

int32_t rwgpu_join_restore(rwgpu_join* h, int32_t side, const rw_chunk* rows) {
  if (!h || !rows) return fail(RW_ERR_INVALID, "null");
  if (side != 0 && side != 1) return fail(RW_ERR_INVALID, "side");
  if (rows->n_cols != h->side[side].n_cols) return fail(RW_ERR_INVALID, "chunk schema mismatch");
  if (h->n_pending) return fail(RW_ERR_INVALID, "collect the outstanding asynchronous pushes first");
  // replay as inserts through the ordinary push, a slice (a multiple of 64 rows: bitmap words split cleanly) at a time;
  // the output is discarded
  const int64_t slice = 1 << 20;
  for (int64_t lo = 0; lo < rows->n_rows; lo += slice) {
    const int64_t m = std::min<int64_t>(slice, rows->n_rows - lo);
    std::vector<rw_column> cols(rows->n_cols);
    for (int k = 0; k < rows->n_cols; k++) {
      cols[k] = rows->columns[k];
      if (type_is_varlen(rows->columns[k].type)) {
        cols[k].offsets = rows->columns[k].offsets + lo;  // (offsets[0] need not be 0: `data` stays the column's base)
      } else {
        cols[k].data = (const uint8_t*)rows->columns[k].data + (size_t)lo * type_width(rows->columns[k].type);
      }
      if (rows->columns[k].validity) cols[k].validity = rows->columns[k].validity + lo / 64;
    }
    rw_chunk part = *rows;
    part.n_rows = m;
    part.ops = rows->ops + lo;
    part.visibility = rows->visibility ? rows->visibility + lo / 64 : nullptr;
    part.columns = cols.data();
    rwgpu_out* out = nullptr;
    int rc = rwgpu_join_push(h, side, &part, &out);
    if (rc != RW_OK) return rc;
    rwgpu_out_release(out);
  }
  return RW_OK;
}

uint64_t rwgpu_join_compactions(rwgpu_join* h) { return h ? h->compactions : 0; }

int32_t rwgpu_join_debug_set_seq(rwgpu_join* h, uint64_t seq) {
  if (!h) return fail(RW_ERR_INVALID, "null");
  h->seq = seq;
  return RW_OK;
}

int32_t rwgpu_join_profile(rwgpu_join* h, int32_t enable, double* ms, uint64_t* launches) {
  if (!h) return fail(RW_ERR_INVALID, "null");
  RW_CUDA(cudaDeviceSynchronize());
  h->prof.collect();
  if (ms) *ms = h->prof.ms;
  if (launches) *launches = h->prof.n;
  h->prof.ms = 0;
  h->prof.n = 0;
  h->prof.on = enable != 0;
  return RW_OK;
}

int32_t rwgpu_join_stats(rwgpu_join* h, uint64_t* left_rows, uint64_t* right_rows, uint64_t* launches) {
  if (!h) return fail(RW_ERR_INVALID, "null");
  RW_CUDA(cudaStreamSynchronize(h->stream));
  if (left_rows) *left_rows = h->side[0].n_rows;
  if (right_rows) *right_rows = h->side[1].n_rows;
  if (launches) *launches = h->launches;
  return RW_OK;
}

}  // extern "C"
