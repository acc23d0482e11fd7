// ddpg_fused_dev.cuh — device building blocks of the cluster-fused kernels (csrc/ddpg_fused.cu, csrc/actor_rollout.cu): the shared-memory
// plan of a CTA, W2 staging, the per-layer forward / backward pieces and the distributed-shared-memory exchanges.  See ddpg_fused.cu
// for the design.  Every product is written with explicit fmaf(): the functions give the same bits in a translation unit built with
// -fmad=false (actor_rollout.cu, which also holds Julia-exact environment arithmetic) as in one built with contraction on.
#pragma once
#include <cooperative_groups.h>
#include <string.h>

#include "common.h"
#include "ddpg_fused.h"
#include "philox.cuh"
#include "act_epilogue.cuh"

namespace cg = cooperative_groups;

#ifndef FUSED_THREADS
#define FUSED_THREADS 256
#endif
#define FT FUSED_THREADS          // threads per CTA: 256 (8 warps) or 512 (16 warps: two threads per layer-1 unit, 16 k-groups)
static_assert(FT == 256 || FT == 512, "FUSED_THREADS must be 256 or 512");
constexpr int NW = FT / 32;       // warps = k-groups of the layer-2 products
constexpr int HALVES = FT / 256;  // threads per layer-1 unit
#define WP 68    // pitch (floats) of a staged W2 slice: rows start on 16-byte boundaries (16-byte copies); a warp reading one row, or 32
                 // rows as float4 (quarter-warp phases of 8 rows x 16 bytes, 272 bytes apart), is free of bank conflicts

struct FusedSmem {
  float W[2][FUSED_MAX_L1 * WP];   // two staged W2 slices [k][col]
  float h1T[2][FUSED_MAX_L1 * 8];  // layer-1 activations of the cluster's 8 rows, unit-major [k][row] (one 32-byte broadcast per k)
  float red[NW * 8 * 64];          // [warp][row][col] partial sums of the layer-2 product
  float h2s[2][8 * 64];            // this CTA's slice of the layer-2 activations [row][col]
  float dzT[64 * 8];               // gradient at this CTA's layer-2 slice, unit-major [col][row]
  float x[2][8 * 12];              // network inputs [row][11] (pitch 12)
  float xch[3][8 * 8 * 2];         // all-gather buffers [source CTA][row][j], filled by the peers
  float rs[8 * HALVES * 32 * 8];   // reduce-scatter buffer [source CTA x column half][unit of my layer-1 slice][row], filled by the peers
  float dz1s[8 * 32];              // gradient at this CTA's layer-1 slice [row][unit]
  float dout[8 * 2];               // gradient at the net's output [row][j]
  float qv[8], rr[8], dd[8];
  unsigned long long src_row[8];   // where the cluster's 8 sampled transitions live (ring offset or column of the caller's arrays)
  const float* src_ser[8];         // a compact ring record's series row (ring.cuh ring_row), else NULL
  unsigned long long ns_row[8];    // n-step rows: ring offset of the walk's last record (s' comes from there) ...
  const float* ns_ser[8];          // ... its series row ...
  float ns_r[8], ns_d[8];          // ... and the walk's r and done
};

__device__ __forceinline__ void cp_async4z(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 4 : 0;  // src-size 0: zero fill
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc));
}

// stage W2[0..l1)[n0 .. n0+nv) of a net into Ws[k][col], one commit group per slice.  vec: rows are 16-byte aligned on both sides and
// nv % 4 == 0 -> 16-byte cp.async (16 per thread and slice at 250/500; columns >= nv are never read as weights).  Otherwise 4-byte
// cp.async with columns >= nv zero-filled.
// (One bulk async copy per row, completing on an mbarrier, was measured first: issuing the 250 small copies of a slice costs the CTA
//  1.0 µs — the TMA unit takes one 256-byte copy every ~8 cycles — against ~0.1 µs for these.)
__device__ __forceinline__ void stage_w2(float* Ws, const float* __restrict__ W2, int l1, int l2, int n0, int nv, bool vec, int tid) {
  if (vec) {
    const int ch = tid & 15;   // a thread keeps its 16-byte column chunk and walks the rows tid/16, tid/16 + 16, ...
    if (ch * 4 < nv) {
      float* dst = Ws + (tid >> 4) * WP + ch * 4;
      const float* src = W2 + (long long)(tid >> 4) * l2 + n0 + ch * 4;
      for (int k = tid >> 4; k < l1; k += FT / 16, dst += (FT / 16) * WP, src += (long long)(FT / 16) * l2) cp_async16(dst, src);
    }
  } else {
    for (int e = tid; e < l1 * 64; e += FT) {
      const int k = e >> 6, col = e & 63;
      const bool ok = col < nv;
      cp_async4z(Ws + k * WP + col, ok ? W2 + (long long)k * l2 + n0 + col : W2, ok);
    }
  }
  cp_commit();
}

// Everything small a CTA reads from a net — its W1 column and b1 (thread = layer-1 unit), its slice of b2 and W3 (lane = columns
// lane, lane+32) — is loaded into registers when the kernel starts: the global-memory latency is paid once, under the W2 staging,
// instead of once per dependent step of the chain.
struct L1Regs { float w[11]; float b; };
__device__ __forceinline__ L1Regs load_l1(const float* __restrict__ W1, const float* __restrict__ b1, int K, int l1, int tid) {
  L1Regs R;
  const int k = tid & 255;   // FT = 512: threads k and k + 256 share unit k
  const bool ok = k < l1;
#pragma unroll
  for (int i = 0; i < 11; ++i) R.w[i] = (ok && i < K) ? __ldg(W1 + i * l1 + k) : 0.0f;
  R.b = ok ? __ldg(b1 + k) : 0.0f;
  return R;
}
struct TailRegs { float b2[2]; float w3[2][2]; };
__device__ __forceinline__ TailRegs load_tail(const float* __restrict__ b2s, const float* __restrict__ W3s, int J, int nv, int lane) {
  TailRegs T;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int c = lane + 32 * h;
    const bool ok = c < nv;
    T.b2[h] = ok ? __ldg(b2s + c) : 0.0f;
    T.w3[h][0] = ok ? __ldg(W3s + c * J) : 0.0f;
    T.w3[h][1] = (ok && J == 2) ? __ldg(W3s + c * J + 1) : 0.0f;
  }
  return T;
}

// layer 1, all l1 units, the cluster's 8 rows: h1T[k][r] = relu(b1[k] + sum_i W1[i][k] x[r][i])      (Dense(in, L1, relu))
__device__ __forceinline__ void f1(const L1Regs& R, int K, int l1, const float* x, float* h1T, int tid) {
  constexpr int RPT = 8 / HALVES;              // rows per thread
  const int k = tid & 255, r0 = (tid >> 8) * RPT;
  if (k < l1) {
    float acc[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) acc[r] = 0.0f;
#pragma unroll
    for (int i = 0; i < 11; ++i) {
      if (i < K) {
#pragma unroll
        for (int r = 0; r < RPT; ++r) acc[r] = fmaf(x[(r0 + r) * 12 + i], R.w[i], acc[r]);
      }
    }
    float o[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) { const float v = acc[r] + R.b; o[r] = v > 0.0f ? v : 0.0f; }
#pragma unroll
    for (int q = 0; q < RPT / 4; ++q)
      *reinterpret_cast<float4*>(h1T + k * 8 + r0 + 4 * q) = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
  }
}

// layer 2, this CTA's slice: h2s[r][col] = relu(b2[col] + sum_k h1[r][k] Ws[k][col]).  Warp w takes k = w, w+NW, ...; lane the columns
// lane and lane+32; the warps' partial sums meet in shared memory in warp order.  Ends with a barrier (h2s visible, Ws/red free).
__device__ __forceinline__ void f2(const float* Ws, const TailRegs& T, int l1, int nv, const float* h1T, float* red, float* h2s, int tid) {
  const int w = tid >> 5, lane = tid & 31;
  float a0[8], a1[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) { a0[r] = 0.0f; a1[r] = 0.0f; }
#pragma unroll 8
  for (int k = w; k < l1; k += NW) {
    const float w0 = Ws[k * WP + lane], w1 = Ws[k * WP + lane + 32];
    const float4 ha = *reinterpret_cast<const float4*>(h1T + k * 8), hb = *reinterpret_cast<const float4*>(h1T + k * 8 + 4);
    a0[0] = fmaf(ha.x, w0, a0[0]); a1[0] = fmaf(ha.x, w1, a1[0]);
    a0[1] = fmaf(ha.y, w0, a0[1]); a1[1] = fmaf(ha.y, w1, a1[1]);
    a0[2] = fmaf(ha.z, w0, a0[2]); a1[2] = fmaf(ha.z, w1, a1[2]);
    a0[3] = fmaf(ha.w, w0, a0[3]); a1[3] = fmaf(ha.w, w1, a1[3]);
    a0[4] = fmaf(hb.x, w0, a0[4]); a1[4] = fmaf(hb.x, w1, a1[4]);
    a0[5] = fmaf(hb.y, w0, a0[5]); a1[5] = fmaf(hb.y, w1, a1[5]);
    a0[6] = fmaf(hb.z, w0, a0[6]); a1[6] = fmaf(hb.z, w1, a1[6]);
    a0[7] = fmaf(hb.w, w0, a0[7]); a1[7] = fmaf(hb.w, w1, a1[7]);
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) { red[(w * 8 + r) * 64 + lane] = a0[r]; red[(w * 8 + r) * 64 + lane + 32] = a1[r]; }
  __syncthreads();
  const int c = tid & 63;                       // (c & 31) == lane: T.b2[c >> 5] is this column's bias
  const float bias = (tid & 32) ? T.b2[1] : T.b2[0];
#pragma unroll
  for (int o = 0; o < 512 / FT; ++o) {          // output (row, column c)
    const int row = (tid >> 6) + o * (FT / 64);
    float v = red[row * 64 + c];
#pragma unroll
    for (int g = 1; g < NW; ++g) v += red[(g * 8 + row) * 64 + c];
    float out = 0.0f;
    if (c < nv) { v += bias; out = v > 0.0f ? v : 0.0f; }
    h2s[row * 64 + c] = out;
  }
  __syncthreads();
}

// output layer (J = 1 or 2 units): this CTA's share of the dot product over its layer-2 slice, row = warp, handed to every CTA of
// the cluster (slot [my rank][row][j] of their all-gather buffer `buf`)
__device__ __forceinline__ void f3_partial(const TailRegs& T, const float* h2s, FusedSmem* S, int buf, cg::cluster_group& cluster, int rank, int tid) {
  const int w = tid >> 5, lane = tid & 31;
  if (w >= 8) return;                                                   // row = warp: warps 8.. (FT = 512) have no row
  const float h0 = h2s[w * 64 + lane], h1 = h2s[w * 64 + lane + 32];   // zero beyond the slice, like the weights
  float p0 = fmaf(h1, T.w3[1][0], h0 * T.w3[0][0]);
  float p1 = fmaf(h1, T.w3[1][1], h0 * T.w3[0][1]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { p0 += __shfl_xor_sync(0xffffffffu, p0, o); p1 += __shfl_xor_sync(0xffffffffu, p1, o); }
  if (lane < FUSED_CLUSTER) {
    FusedSmem* peer = cluster.map_shared_rank(S, lane);
    peer->xch[buf][(rank * 8 + w) * 2 + 0] = p0;
    peer->xch[buf][(rank * 8 + w) * 2 + 1] = p1;
  }
}
__device__ __forceinline__ float xch_sum(const FusedSmem* S, int buf, int r, int j) {  // the 8 CTAs' shares in rank order
  float v = S->xch[buf][r * 2 + j];
#pragma unroll
  for (int s = 1; s < FUSED_CLUSTER; ++s) v += S->xch[buf][(s * 8 + r) * 2 + j];
  return v;
}

// back through the output layer: the gradient at this CTA's layer-2 slice dzT[col][r] = (sum_j W3[col][j] dout[r][j]) * [h2 > 0];
// w3c0/1 = W3[col = tid & 63][0/1] (preloaded)
__device__ __forceinline__ void b3_dz(float w3c0, float w3c1, int J, int nv, const float* h2s, const float* dout, float* dzT, int tid) {
  const int col = tid & 63;
#pragma unroll
  for (int q = 0; q < 512 / FT; ++q) {
    const int r = (tid >> 6) + q * (FT / 64);
    float v = 0.0f;
    if (col < nv) {
      v = w3c0 * dout[r * 2];
      if (J == 2) v = fmaf(w3c1, dout[r * 2 + 1], v);
      v = (h2s[r * 64 + col] > 0.0f) ? v : 0.0f;
    }
    dzT[col * 8 + r] = v;
  }
}
// dW3 (and db3 on rank 0) of these 8 rows into the cluster's partial-gradient copy
__device__ __forceinline__ void b3_grads(int J, int nv, const float* h2s, const float* dout, float* part_w3s, float* part_b3, int tid) {
  if (tid < nv * J) {
    const int col = tid / J, j = tid - col * J;
    float v = 0.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) v = fmaf(h2s[r * 64 + col], dout[r * 2 + j], v);
    part_w3s[col * J + j] = v;
  }
  if (part_b3 && tid >= 128 && tid < 128 + J) {
    const int j = tid - 128;
    float v = 0.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) v += dout[r * 2 + j];
    part_b3[j] = v;
  }
}

// dW2 of these 8 rows, this CTA's columns: part[k][col] = sum_r h1[r][k] dz[r][col]; db2[col] = sum_r dz[r][col]
__device__ __forceinline__ void bw2(const float* h1T, const float* dzT, int l1, int l2, int nv, float* part_w2s, float* part_b2s, int tid) {
  const int w = tid >> 5, lane = tid & 31;
  const float4 d0a = *reinterpret_cast<const float4*>(dzT + lane * 8), d0b = *reinterpret_cast<const float4*>(dzT + lane * 8 + 4);
  const float4 d1a = *reinterpret_cast<const float4*>(dzT + (lane + 32) * 8), d1b = *reinterpret_cast<const float4*>(dzT + (lane + 32) * 8 + 4);
  const bool ok0 = lane < nv, ok1 = lane + 32 < nv;
#pragma unroll 8
  for (int k = w; k < l1; k += NW) {
    const float4 ha = *reinterpret_cast<const float4*>(h1T + k * 8), hb = *reinterpret_cast<const float4*>(h1T + k * 8 + 4);
    float o0 = ha.x * d0a.x, o1 = ha.x * d1a.x;
    o0 = fmaf(ha.y, d0a.y, o0); o1 = fmaf(ha.y, d1a.y, o1);
    o0 = fmaf(ha.z, d0a.z, o0); o1 = fmaf(ha.z, d1a.z, o1);
    o0 = fmaf(ha.w, d0a.w, o0); o1 = fmaf(ha.w, d1a.w, o1);
    o0 = fmaf(hb.x, d0b.x, o0); o1 = fmaf(hb.x, d1b.x, o1);
    o0 = fmaf(hb.y, d0b.y, o0); o1 = fmaf(hb.y, d1b.y, o1);
    o0 = fmaf(hb.z, d0b.z, o0); o1 = fmaf(hb.z, d1b.z, o1);
    o0 = fmaf(hb.w, d0b.w, o0); o1 = fmaf(hb.w, d1b.w, o1);
    float* row = part_w2s + (long long)k * l2;
    if (ok0) row[lane] = o0;
    if (ok1) row[lane + 32] = o1;
  }
  if (tid < nv) {
    float v = 0.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) v += dzT[tid * 8 + r];
    part_b2s[tid] = v;
  }
}

// back through layer 2: this CTA's share (its columns) of dX[r][k] = sum_col W2[k][col] dz[r][col], thread = k (FT = 512: two
// threads per k, 32 columns each), scattered to the CTA that owns layer-1 unit k (slot [my rank x half][k - its first unit][row] of its
// reduce-scatter buffer)
__device__ __forceinline__ void bx2(const float* Ws, const float* dzT, int l1, int nv, int n1s, bool vec, FusedSmem* S, cg::cluster_group& cluster,
                                    int rank, int tid) {
  const int k = tid & 255, half = tid >> 8;
  if (k < l1) {
    float acc[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = 0.0f;
    const float* wr = Ws + k * WP;
    int c = half * (64 / HALVES);
    const int c_end = min(nv, c + 64 / HALVES);
    if (vec) {  // nv % 4 == 0: four columns per shared-memory read of the row
#pragma unroll 2
      for (; c + 4 <= c_end; c += 4) {
        const float4 w4 = *reinterpret_cast<const float4*>(wr + c);
        const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 da = *reinterpret_cast<const float4*>(dzT + (c + u) * 8), db = *reinterpret_cast<const float4*>(dzT + (c + u) * 8 + 4);
          acc[0] = fmaf(wv[u], da.x, acc[0]); acc[1] = fmaf(wv[u], da.y, acc[1]); acc[2] = fmaf(wv[u], da.z, acc[2]); acc[3] = fmaf(wv[u], da.w, acc[3]);
          acc[4] = fmaf(wv[u], db.x, acc[4]); acc[5] = fmaf(wv[u], db.y, acc[5]); acc[6] = fmaf(wv[u], db.z, acc[6]); acc[7] = fmaf(wv[u], db.w, acc[7]);
        }
      }
    }
    for (; c < c_end; ++c) {
      const float wv = wr[c];
      const float4 da = *reinterpret_cast<const float4*>(dzT + c * 8), db = *reinterpret_cast<const float4*>(dzT + c * 8 + 4);
      acc[0] = fmaf(wv, da.x, acc[0]); acc[1] = fmaf(wv, da.y, acc[1]); acc[2] = fmaf(wv, da.z, acc[2]); acc[3] = fmaf(wv, da.w, acc[3]);
      acc[4] = fmaf(wv, db.x, acc[4]); acc[5] = fmaf(wv, db.y, acc[5]); acc[6] = fmaf(wv, db.z, acc[6]); acc[7] = fmaf(wv, db.w, acc[7]);
    }
    const int owner = k / n1s, kk = k - owner * n1s;
    FusedSmem* peer = cluster.map_shared_rank(S, owner);
    float4* dst = reinterpret_cast<float4*>(peer->rs + ((rank * HALVES + half) * 32 + kk) * 8);   // two 16-byte stores into the owner's shared memory
    dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
}
// after the cluster barrier: add the shares in source order and apply layer 1's ReLU mask -> dz1s[r][kk] (this CTA's layer-1 units)
__device__ __forceinline__ void rs_finish(FusedSmem* S, const float* h1T, int k0, int n1v, int tid) {
  if (tid >= 256) return;
  const int r = tid >> 5, kk = tid & 31;
  float v = 0.0f;
  if (kk < n1v) {
    v = S->rs[kk * 8 + r];
#pragma unroll
    for (int s = 1; s < FUSED_CLUSTER * HALVES; ++s) v += S->rs[(s * 32 + kk) * 8 + r];
    v = (h1T[(k0 + kk) * 8 + r] > 0.0f) ? v : 0.0f;
  }
  S->dz1s[r * 32 + kk] = v;
}

// dW1 / db1 of these 8 rows for this CTA's layer-1 units: part[i][k] = sum_r x[r][i] dz1[r][k]
__device__ __forceinline__ void bw1(const float* x, int K1, const float* dz1s, int l1, int n1v, float* part_w1s, float* part_b1s, int tid) {
  for (int e = tid; e < K1 * 32; e += FT) {
    const int i = e >> 5, kk = e & 31;
    if (kk < n1v) {
      float v = 0.0f;
#pragma unroll
      for (int r = 0; r < 8; ++r) v = fmaf(x[r * 12 + i], dz1s[r * 32 + kk], v);
      part_w1s[i * l1 + kk] = v;
    }
  }
  if (tid < n1v) {
    float v = 0.0f;
#pragma unroll
    for (int r = 0; r < 8; ++r) v += dz1s[r * 32 + tid];
    part_b1s[tid] = v;
  }
}

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); }

// -DFUSED_TRACE (tools/trace_fused.py builds that variant): thread 0 of CTA 0 stamps clock64() at the marked points
#ifdef FUSED_TRACE
__device__ long long fused_trace[2][32];
#define STAMP(k, i) do { if (blockIdx.x == 0 && threadIdx.x == 0) fused_trace[k][i] = clock64(); } while (0)
extern "C" __attribute__((visibility("default"))) int ddpg_fused_trace_read(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, fused_trace, sizeof(fused_trace));
}
#else
#define STAMP(k, i) do { } while (0)
#endif

// programmatic dependent launch: the kernel may start while its predecessor in the stream still runs; everything the predecessor
// writes is read only after grid_dependency_wait()
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

struct Geo { int rank, row0, n0, nv, k0, n1v, n1s; };
__device__ __forceinline__ Geo make_geo(int l1, int l2, int vec16, cg::cluster_group& cluster) {
  Geo g;
  g.rank = (int)cluster.block_rank();
  g.row0 = (int)(blockIdx.x / FUSED_CLUSTER) * FUSED_ROWS;
  int n2s = (l2 + FUSED_CLUSTER - 1) / FUSED_CLUSTER;
  if (vec16) n2s = (n2s + 3) & ~3;   // slices start on 16-byte boundaries of the W2 rows
  g.n1s = (l1 + FUSED_CLUSTER - 1) / FUSED_CLUSTER;
  g.n0 = min(g.rank * n2s, l2); g.nv = min(n2s, l2 - g.n0);
  g.k0 = min(g.rank * g.n1s, l1); g.n1v = min(g.n1s, l1 - g.k0);
  return g;
}

