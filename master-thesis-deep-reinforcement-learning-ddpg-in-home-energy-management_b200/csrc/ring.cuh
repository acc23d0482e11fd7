// ring.cuh — the replay ring's record format and sampling rule: everything that knows where a field of a slot lives, how a compact
// record names its series row and which slot a minibatch draw lands on.
//
// Layout: 23 fields per slot, tiled so that one slot's fields sit at fixed 128-byte strides:
// element (slot, k) lives at ((slot >> 5) * 23 + k) * 32 + (slot & 31).
// A warp writing 32 consecutive slots stores one full 128-byte line per field, with the field offset an
// immediate (no per-field address arithmetic in the rollout kernel).
//
// A slot holds one of two record forms, told apart by field RING_SRC:
//   RING_SRC == 0 (all bits): a FULL record, fields 0..21 = s[9] a[2] r s'[9] done.  cudaMemset at creation makes every slot full.
//   RING_SRC != 0: a COMPACT record written by a rollout whose state rows come from an env series: only s[0..1] (Soc_b, Soc_ev),
//     a[0..1], r and s'[0..1] are stored; s[2..8] is series row `row` (1-based) and s'[2..8] row `row + 1` of the ring's copy of
//     that series (entry `entry` of the ring's series table), done = 0.  RING_SRC holds the bits of ring_tag(entry, row).
// The series table is reachable from the ring pointer alone: RING_HEADER_FLOATS floats in front of slot 0 hold RING_MAX_SERIES
// device pointers to the ring's copies of the series (32-byte rows, as ShemsEnv::series).
//
// Logical index i (0 = oldest) of a ring holding len records lives in physical slot (head - len + i) mod cap.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include "philox.cuh"

#define RING_FIELDS 23
#define RING_S 0      // s[0..8]
#define RING_A 9      // a[0..1]
#define RING_R 11     // r
#define RING_S2 12    // s'[0..8]
#define RING_DONE 21  // done
#define RING_SRC 22   // 0: full record; else the bits of ring_tag(entry, row) of a compact record
#define RING_TRANSITION_FIELDS 22  // the logical transition s a r s' done
__host__ __device__ __forceinline__ size_t ring_base(long long slot) { return ((size_t)(slot >> 5) * RING_FIELDS) * 32 + (size_t)(slot & 31); }

#define RING_MAX_SERIES 16
#define RING_HEADER_FLOATS 32   // 128 bytes: RING_MAX_SERIES pointers; keeps slot 0 on a 128-byte line
#define RING_TAG_ROW_BITS 24    // row < 2^24, entry < RING_MAX_SERIES; the row is >= 1, so a tag is never 0
#define RING_TAG_ROW_MASK ((1u << RING_TAG_ROW_BITS) - 1u)
#define RING_TAG_MAX_ROW ((int32_t)RING_TAG_ROW_MASK)  // the largest series row a compact record can name
static_assert(RING_MAX_SERIES * sizeof(float*) <= RING_HEADER_FLOATS * sizeof(float), "the series table fits the header");

// floats to allocate for a ring of cap slots, header included; the ring proper starts at ring_in_alloc(alloc)
__host__ __device__ __forceinline__ size_t ring_alloc_floats(long long cap) {
  return RING_HEADER_FLOATS + RING_FIELDS * 32 * (((size_t)cap + 31) / 32);
}
__host__ __device__ __forceinline__ float* ring_in_alloc(float* alloc) { return alloc + RING_HEADER_FLOATS; }
// the series table in the header: entry i is the device pointer to the ring's copy of series i
__host__ __device__ __forceinline__ const float* const* ring_table(const float* ring) {
  return reinterpret_cast<const float* const*>(ring - RING_HEADER_FLOATS);
}

__host__ __device__ __forceinline__ uint32_t ring_tag(int entry, int row1) { return ((uint32_t)entry << RING_TAG_ROW_BITS) | (uint32_t)row1; }
// the 8 floats of the series row a record at q names, (soc_ev, h_countdown, electkwh, PV_generation | p_buy, hour_cos, hour_sin,
// season), or NULL for a full record.  table: ring_table(ring) on the device, host copies of the same series on the host.
__host__ __device__ __forceinline__ const float* ring_row(const float* const* table, const float* q) {
#ifdef __CUDA_ARCH__
  const uint32_t tag = __float_as_uint(q[RING_SRC * 32]);
#else
  uint32_t tag;
  memcpy(&tag, q + RING_SRC * 32, sizeof(tag));
#endif
  return tag ? table[tag >> RING_TAG_ROW_BITS] + 8 * (size_t)((tag & RING_TAG_ROW_MASK) - 1u) : nullptr;
}
// logical field f in [0, RING_TRANSITION_FIELDS) of the record at q with series row `row` (ring_row): state field k = 2..8 is
// column k - 1 of the row, s' follows at +8
__host__ __device__ __forceinline__ float ring_field(const float* q, const float* row, int f) {
  if (row) {
    if (f >= RING_S + 2 && f < RING_A) return row[f - RING_S - 1];
    if (f >= RING_S2 + 2 && f < RING_DONE) return row[8 + f - RING_S2 - 1];
    if (f == RING_DONE) return 0.0f;
  }
  return q[f * 32];
}

// physical slot of logical index li of a ring of len records whose next push goes to slot head
__host__ __device__ __forceinline__ long long ring_slot(long long li, long long head, long long len, long long cap) {
  long long slot = head - len + li;
  if (slot < 0) slot += cap;
  return slot;
}
// slot of transition i of a push that starts at slot head
__host__ __device__ __forceinline__ long long ring_push_slot(long long head, long long i, long long cap) {
  const long long slot = head + i;
  return slot - (slot / cap) * cap;
}

// The record addresses a writer visits at slots s, s + N, s + 2N, ... (mod cap) when N and cap are multiples of 32: slot + N keeps
// the lane (slot & 31) and moves N / 32 tiles, so the address advances by a constant stride and wraps with one compare.
struct RingWalk {
  float* q;            // record of the current slot
  const float* last;   // from here on the next slot wraps
  ptrdiff_t stride, back;  // N / 32 tiles, and the same less the ring's cap / 32 tiles
};
__host__ __device__ __forceinline__ RingWalk ring_walk(float* ring, long long slot, long long N, long long cap) {
  RingWalk w;
  w.q = ring + ring_base(slot);
  w.stride = (ptrdiff_t)(N >> 5) * RING_FIELDS * 32;
  w.back = w.stride - (ptrdiff_t)(cap >> 5) * RING_FIELDS * 32;
  w.last = ring - w.back;  // N <= cap: at most one wrap
  return w;
}
__host__ __device__ __forceinline__ void ring_walk_next(RingWalk& w) { w.q += (w.q >= w.last) ? w.back : w.stride; }

// minibatch row j of update `update`: Philox(seed, id = j, ctr = update, stream SAMPLE) -> logical index floor(u * len)
__host__ __device__ __forceinline__ long long ring_draw(uint64_t seed, uint64_t j, uint32_t update, long long len) {
  uint32_t w[4];
  philox4x32_10(seed, j, update, STREAM_SAMPLE, w);
  long long li = (long long)(u53(w[0], w[1]) * (double)len);
  if (li >= len) li = len - 1;
  return li;
}

// ---- proportional prioritized replay (replay_enable_priorities; Schaul et al., 2016)
// A memory with priorities keeps a sum tree beside the ring: P2 = the next power of two >= cap, nodes 0 .. 2 P2 - 1 (node 0 unused),
// node 1 the root, node i the parent of 2i and 2i+1, the leaf of slot s node P2 + s.  Every internal node is RN32(left + right),
// always recomputed from its children (never updated by deltas), so the tree's bits are a function of its leaves alone.  Unfilled
// slots and the padding past cap are 0.  PRIO_HEADER_FLOATS floats in front of node 0 hold p_max and the arrival counter of
// replay_prio_refresh_kernel.
#define PRIO_HEADER_FLOATS 32
#define PRIO_PMAX 0      // header float: the largest priority ever written (starts at 1)
#define PRIO_ARRIVED 1   // header word: blocks of the running refresh launch that are done
__host__ __device__ __forceinline__ long long prio_p2(long long cap) {
  long long p = 1;
  while (p < cap) p <<= 1;
  return p;
}
__host__ __device__ __forceinline__ size_t prio_alloc_floats(long long cap) { return PRIO_HEADER_FLOATS + 2 * (size_t)prio_p2(cap); }
__host__ __device__ __forceinline__ float* prio_header(float* tree) { return tree - PRIO_HEADER_FLOATS; }

// prioritized minibatch row j of B of update `update`: U = u53(Philox(seed, id = j, ctr = update, stream PER)), x = RN32((j + U) root / B)
// (stratified: one draw per B-th of the mass), then down from the root: left if x < L or R == 0, else x = RN32(x - L) and right.  A
// subtree without mass is never entered, so the draw lands on a slot of positive priority even when x rounds up to the root.  Returns
// the physical slot; *leaf = its priority.
__host__ __device__ __forceinline__ long long ring_draw_prioritized(const float* tree, long long p2, uint64_t seed, uint64_t j, uint32_t update,
                                                                   int B, float* leaf) {
  uint32_t w[4];
  philox4x32_10(seed, j, update, STREAM_PER, w);
  float x = (float)(((double)j + u53(w[0], w[1])) * (double)tree[1] / (double)B);
  long long n = 1;
  while (n < p2) {
    const float L = tree[2 * n], R = tree[2 * n + 1];
    if (x < L || R == 0.0f) n = 2 * n;
    else { x = x - L; n = 2 * n + 1; }
  }
  *leaf = tree[n];
  return n - p2;
}
// logical index (0 = oldest) of physical slot `slot` of a ring of len records whose next push goes to slot head
__host__ __device__ __forceinline__ long long ring_logical(long long slot, long long head, long long len, long long cap) {
  long long li = (slot - head + len) % cap;
  if (li < 0) li += cap;
  return li;
}
// importance weight before the normalisation by the minibatch's largest: (leaf len / root)^-beta in Float64
__host__ __device__ __forceinline__ double ring_is_weight(float leaf, long long len, float root, float beta) {
  return pow((double)leaf * (double)len / (double)root, -(double)beta);
}
// priority of a row after its TD target: RN32((|RN32(y - q)| + eps)^alpha)
__host__ __device__ __forceinline__ float ring_priority(float y, float q, float alpha, float eps) {
  const float d = y - q;
  return (float)pow((double)fabsf(d) + (double)eps, (double)alpha);
}

// the words both record forms store; a compact record adds its tag, a full one the other 14 fields
__device__ __forceinline__ void ring_store_own(float* q, float sb, float sev, float a0, float a1, float r, float sb2, float sev2) {
  q[(RING_S + 0) * 32] = sb; q[(RING_S + 1) * 32] = sev;
  q[(RING_A + 0) * 32] = a0; q[(RING_A + 1) * 32] = a1;
  q[RING_R * 32] = r;
  q[(RING_S2 + 0) * 32] = sb2; q[(RING_S2 + 1) * 32] = sev2;
}
__device__ __forceinline__ void ring_store_full(float* q, const float* s, float a0, float a1, float r, const float* s2, float done) {
  ring_store_own(q, s[0], s[1], a0, a1, r, s2[0], s2[1]);
#pragma unroll
  for (int k = 2; k < 9; ++k) q[(RING_S + k) * 32] = s[k];
#pragma unroll
  for (int k = 2; k < 9; ++k) q[(RING_S2 + k) * 32] = s2[k];
  q[RING_DONE * 32] = done;
  q[RING_SRC * 32] = 0.0f;
}
// series_tag = ring_tag(entry, 0) of the ring's copy of the series: s[2..8] is its row `row`, s'[2..8] row `row + 1`, done = 0
__device__ __forceinline__ void ring_store_compact(float* q, float sb, float sev, float a0, float a1, float r, float sb2, float sev2,
                                                   uint32_t series_tag, int row) {
  ring_store_own(q, sb, sev, a0, a1, r, sb2, sev2);
  q[RING_SRC * 32] = __uint_as_float(series_tag | (uint32_t)row);
}
// ring_store_compact for two records of the same series row in slots s and s + 1, s even (so both sit in one tile): q is slot s's
// record, element i of each argument belongs to slot s + i, and each field of both is one 8-byte store
__device__ __forceinline__ void ring_store_compact_pair(float* q, const float sb[2], const float sev[2], const float a0[2], const float a1[2],
                                                        const float r[2], const float sb2[2], const float sev2[2], uint32_t series_tag, int row) {
  auto st2 = [q](int f, float x, float y) { *reinterpret_cast<float2*>(q + f * 32) = make_float2(x, y); };
  st2(RING_S + 0, sb[0], sb[1]); st2(RING_S + 1, sev[0], sev[1]);
  st2(RING_A + 0, a0[0], a0[1]); st2(RING_A + 1, a1[0], a1[1]);
  st2(RING_R, r[0], r[1]);
  st2(RING_S2 + 0, sb2[0], sb2[1]); st2(RING_S2 + 1, sev2[0], sev2[1]);
  const float tag = __uint_as_float(series_tag | (uint32_t)row);
  st2(RING_SRC, tag, tag);
}
