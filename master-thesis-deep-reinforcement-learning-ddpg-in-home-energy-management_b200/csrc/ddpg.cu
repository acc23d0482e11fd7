// ddpg.cu — the DDPG minibatch update of RL-SHEMS/algorithms/DDPG.jl (replay :121-145, act :148-176,
// soft_update! :99-103, update_model! :105-108, losses :114-119) on one GPU.
//
// Design (B200):
//  * All four nets live in flat fp32 buffers  [W1|b1|W2|b2|W3|b3]; a layer weight is stored exactly
//    as Flux stores it (out×in column-major == Wt[in][out] row-major, `out` contiguous), so
//    get/set_layer are plain copies and every GEMM reads weights coalesced along `out`.
//  * Activations are sample-major [B][width].
//  * One generic tiled SGEMM kernel (32×32×32 tiles, 128 threads, 2×4 register blocking, register
//    double buffering) runs every contraction; a launch carries up to 4 independent problems
//    (blockIdx.z) so that e.g. actor_target-L1, critic-L1 and actor-L1 share one dependent phase.
//    Bias/ReLU/tanh, ReLU-mask, tanh-grad, TD-target and the bias-gradient column sums are fused
//    into its epilogue.  At B=120 the update is launch/latency bound (308 MFLOP ≈ 4 µs of fp32
//    SIMT peak) so the whole sequence (21 dependent phases) is captured once in a CUDA graph.
//  * Adam (+ Polyak for both targets) is one fused elementwise kernel over the flat buffers, with
//    the Float64 element math Flux.ADAM performs when β, ϵ are Float64.
//  * Minibatch sampling is on the device: Philox indices -> gather from the replay ring ->
//    normalize() fused, so no host round trip per update (the reference does 5 H2D copies).
#include <new>
#include <vector>
#include <string.h>
#include <stdlib.h>
#include <stddef.h>
#include <math.h>
#include <unistd.h>

#include "common.h"
#include "philox.cuh"
#include "tc_gemm.h"
#include "ddpg_fused.h"
#include "act_epilogue.cuh"

// ----------------------------------------------------------------------------- GEMM
enum { EPI_NONE = 0, EPI_BIAS_RELU, EPI_BIAS_TANH, EPI_BIAS_ID, EPI_RELU_MASK, EPI_TD_TARGET, EPI_TANH_GRAD, EPI_SCALE_MASK };

struct GemmProblem {
  const float* A; long long sAm, sAk;  // A(m,k) = A[m*sAm + k*sAk]
  const float* B; long long sBk, sBn;  // B(k,n) = B[k*sBk + n*sBn]
  float* C; long long ldc;             // C(m,n) = C[m*ldc + n]
  int M, N, K;
  int epi;
  const float* bias;   // [N]                         (BIAS_*, TD_TARGET)
  const float* aux;    // RELU_MASK/SCALE_MASK: H(m,n) with ld auxld; TANH_GRAD: Y(m,n); TD_TARGET: r[m]
  long long auxld;
  const float* aux2;   // TD_TARGET: done[m]
  const float* aux3;   // TD_TARGET: q[m] (critic output on (s,a))
  float* out2;         // TD_TARGET: dq[m] = 2 (q - y) / B
  float* dbias;        // column sums of B(k,n) over k (bias gradient), written by the m-tile 0 CTAs
  float alpha;         // SCALE_MASK: scale
  const DdpgCtrl* ctrl;  // TD_TARGET: learner 0's control block; γ = ctrl[learner].hp.gamma
  float inv_batch;     // TD_TARGET: 1/B
};
struct GemmBatch {
  GemmProblem p[4]; int count;
  // split-K (count == 1, dW-type problems with K = batch >= 1024): blockIdx.z is the K-split; split s writes its partial
  // [M*N | N] (tile sums | bias-gradient column sums) at C + s*split_stride; splitk_reduce_kernel adds them in a fixed order
  int ksplit; long long split_stride;
  // population of independent learners (ksplit == 1): blockIdx.z = learner * count + problem; learner l reads its weights
  // (B, bias) ls_w floats and everything else (A, C, aux*, out2, dbias) ls_x floats behind learner 0's pointers
  int pop; long long ls_w, ls_x;
};
__device__ __forceinline__ void gemm_shift(GemmProblem& p, int learner, long long ow, long long ox) {
  p.A += ox; p.B += ow; p.C += ox;
  if (p.ctrl) p.ctrl += learner;
  if (p.bias) p.bias += ow;
  if (p.aux) p.aux += ox;
  if (p.aux2) p.aux2 += ox;
  if (p.aux3) p.aux3 += ox;
  if (p.out2) p.out2 += ox;
  if (p.dbias) p.dbias += ox;
}

#define BK 32
#define GEMM_KGROUPS 4                       // intra-CTA split-K: each k-group owns BK/4 of every k-tile
#define GEMM_STAGES 3

// 4-byte cp.async (LDGSTS) with zero fill when `valid` is false: the tile loads bypass registers and stay in flight
// across GEMM_STAGES tiles.
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// the fused epilogues (see the EPI_* enum)
__device__ __forceinline__ float gemm_epilogue(const GemmProblem& p, int m, int n, float v) {
  switch (p.epi) {
    case EPI_BIAS_RELU: v += p.bias[n]; v = v > 0.0f ? v : 0.0f; break;
    case EPI_BIAS_TANH: v += p.bias[n]; v = tanhf(v); break;
    case EPI_BIAS_ID: v += p.bias[n]; break;
    case EPI_RELU_MASK: v = (p.aux[m * p.auxld + n] > 0.0f) ? v : 0.0f; break;
    case EPI_SCALE_MASK: v = (p.aux[m * p.auxld + n] > 0.0f) ? v * p.alpha : 0.0f; break;
    case EPI_TANH_GRAD: { const float y = p.aux[m * p.auxld + n]; v = v * (1.0f - y * y); } break;
    case EPI_TD_TARGET: {  // y = r + γ(1-done) q'   (DDPG.jl:133);  dq = 2 (q - y) / B  (d mse / d q)
      const float q2 = v + p.bias[n];
      const float y = p.aux[m] + (p.ctrl->hp.gamma * (1.0f - p.aux2[m])) * q2;
      v = y;
      p.out2[m] = 2.0f * (p.aux3[m] - y) * p.inv_batch;
    } break;
    default: break;
  }
  return v;
}

// C = epilogue(A · B) for up to 4 independent problems (blockIdx.z).  TBM×TBN output tile per CTA, k-tiles of 32 in a
// 3-stage cp.async ring.  These problems are small (B = 120 rows): the kernel is built for latency, not for peak
// FLOPs — 4 k-groups × the classic 2×4 register tiling keep the schedulers busy, partial sums meet in shared memory
// in a fixed order (deterministic), and all threads run the fused epilogue and the coalesced store.  The 16×16
// variant quadruples the CTA count for launches that would otherwise occupy a fraction of the 148 SMs.
template <int TBM, int TBN>
__global__ void __launch_bounds__(TBM * TBN / 2)
gemm_batch_kernel(const GemmBatch gb) {
  constexpr int THREADS = TBM * TBN / 2;          // 4 k-groups x (TBM/2 x TBN/4) threads
  constexpr int GROUP = THREADS / GEMM_KGROUPS;
  constexpr int TXN = TBN / 4;                    // threads along n inside a k-group
  constexpr int AS_LD = TBM + 2, BS_LD = TBN + 4, RED_LD = TBN + 1;
  constexpr int EA = TBM * BK / THREADS, EB = BK * TBN / THREADS;
  const bool splitk = gb.ksplit > 1;
  const int learner = splitk ? 0 : blockIdx.z / gb.count;
  GemmProblem p = gb.p[splitk ? 0 : blockIdx.z - learner * gb.count];
  if (learner) gemm_shift(p, learner, learner * gb.ls_w, learner * gb.ls_x);
  const int split = splitk ? blockIdx.z : 0;
  const int m0 = blockIdx.x * TBM, n0 = blockIdx.y * TBN;  // M tiles on grid.x (no 65535 limit for large batches)
  if (m0 >= p.M || n0 >= p.N) return;
  __shared__ __align__(16) float As[GEMM_STAGES][BK][AS_LD];
  __shared__ __align__(16) float Bs[GEMM_STAGES][BK][BS_LD];
  __shared__ float red[GEMM_KGROUPS][TBM][RED_LD];
  __shared__ float colred[GEMM_KGROUPS][TBN];
  const int tid = threadIdx.x;
  const int kg = tid / GROUP, t = tid % GROUP;
  const int tx = t % TXN, ty = t / TXN;  // thread tile inside the k-group: rows ty*2..+1, cols tx*4..+3
  // global->smem mapping, walking the contiguous dimension of each operand
  const bool a_kfast = (p.sAk == 1);
  const bool b_nfast = (p.sBn == 1);
  const float* a_ptr[EA]; const float* b_ptr[EB];
  float* a_dst[EA]; float* b_dst[EB];
  int a_k[EA], b_k[EB]; bool a_ok[EA], b_ok[EB];
#pragma unroll
  for (int j = 0; j < EA; ++j) {
    const int e = tid + j * THREADS;
    const int kk_a = a_kfast ? (e & 31) : (e / TBM), mm = a_kfast ? (e >> 5) : (e % TBM);
    a_k[j] = kk_a; a_ok[j] = (m0 + mm) < p.M;
    a_ptr[j] = p.A + (long long)(m0 + mm) * p.sAm + (long long)kk_a * p.sAk;
    a_dst[j] = &As[0][kk_a][mm];
  }
#pragma unroll
  for (int j = 0; j < EB; ++j) {
    const int e = tid + j * THREADS;
    const int kk_b = b_nfast ? (e / TBN) : (e & 31), nn = b_nfast ? (e % TBN) : (e >> 5);
    b_k[j] = kk_b; b_ok[j] = (n0 + nn) < p.N;
    b_ptr[j] = p.B + (long long)kk_b * p.sBk + (long long)(n0 + nn) * p.sBn;
    b_dst[j] = &Bs[0][kk_b][nn];
  }
  const long long a_step = (long long)BK * p.sAk, b_step = (long long)BK * p.sBk;
  auto issue_tile = [&](int tile, int buf) {
    const int k0 = tile * BK;
#pragma unroll
    for (int j = 0; j < EA; ++j) {
      const bool va = a_ok[j] && (k0 + a_k[j] < p.K);
      cp_async4(a_dst[j] + buf * (BK * AS_LD), va ? a_ptr[j] + tile * a_step : p.A, va);
    }
#pragma unroll
    for (int j = 0; j < EB; ++j) {
      const bool vb = b_ok[j] && (k0 + b_k[j] < p.K);
      cp_async4(b_dst[j] + buf * (BK * BS_LD), vb ? b_ptr[j] + tile * b_step : p.B, vb);
    }
  };
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float colsum = 0.0f;
  const bool want_dbias = (p.dbias != nullptr) && (blockIdx.x == 0);
  const bool col_thread = want_dbias && (tid < GEMM_KGROUPS * TBN);  // thread (col = tid % TBN, k-quarter = tid / TBN)
  const int ntiles_all = (p.K + BK - 1) / BK;
  const int tiles_per = splitk ? (ntiles_all + gb.ksplit - 1) / gb.ksplit : ntiles_all;
  const int t_begin = split * tiles_per;
  const int ntiles = max(0, min(ntiles_all, t_begin + tiles_per) - t_begin);  // this CTA's k-tiles: t_begin .. t_begin+ntiles-1
#pragma unroll
  for (int s = 0; s < GEMM_STAGES - 1; ++s) {
    if (s < ntiles) issue_tile(t_begin + s, s);
    cp_async_commit();
  }
  constexpr int KSUB = BK / GEMM_KGROUPS;
  for (int tile = 0; tile < ntiles; ++tile) {
    cp_async_wait<GEMM_STAGES - 2>();  // tile `tile` has landed (this thread's copies) ...
    __syncthreads();                   // ... and everyone's; everyone is also done with tile-1, whose buffer is refilled next
    {
      const int tn = tile + GEMM_STAGES - 1;
      if (tn < ntiles) issue_tile(t_begin + tn, tn % GEMM_STAGES);
      cp_async_commit();
    }
    const int buf = tile % GEMM_STAGES;
#pragma unroll
    for (int kq = 0; kq < KSUB; ++kq) {
      const int kk = kg * KSUB + kq;
      const float2 a = *reinterpret_cast<const float2*>(&As[buf][kk][ty * 2]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      acc[0][0] = fmaf(a.x, b.x, acc[0][0]); acc[0][1] = fmaf(a.x, b.y, acc[0][1]);
      acc[0][2] = fmaf(a.x, b.z, acc[0][2]); acc[0][3] = fmaf(a.x, b.w, acc[0][3]);
      acc[1][0] = fmaf(a.y, b.x, acc[1][0]); acc[1][1] = fmaf(a.y, b.y, acc[1][1]);
      acc[1][2] = fmaf(a.y, b.z, acc[1][2]); acc[1][3] = fmaf(a.y, b.w, acc[1][3]);
    }
    if (col_thread) {
#pragma unroll
      for (int kq = 0; kq < KSUB; ++kq) colsum += Bs[buf][(tid / TBN) * KSUB + kq][tid % TBN];
    }
  }
  // meet the k-groups' partial sums in shared memory (fixed order: deterministic)
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[kg][ty * 2 + i][tx * 4 + j] = acc[i][j];
  if (col_thread) colred[tid / TBN][tid % TBN] = colsum;
  __syncthreads();
  const long long soff = (long long)split * gb.split_stride;
  if (want_dbias && tid < TBN && n0 + tid < p.N)
    p.dbias[soff + n0 + tid] = ((colred[0][tid] + colred[1][tid]) + colred[2][tid]) + colred[3][tid];
#pragma unroll
  for (int o = 0; o < (TBM * TBN) / THREADS; ++o) {
    const int e = tid + o * THREADS;
    const int mm = e / TBN, nn = e % TBN;
    const int m = m0 + mm, n = n0 + nn;
    if (m >= p.M || n >= p.N) continue;
    const float v = ((red[0][mm][nn] + red[1][mm][nn]) + red[2][mm][nn]) + red[3][mm][nn];
    p.C[soff + m * p.ldc + n] = splitk ? v : gemm_epilogue(p, m, n, v);
  }
}

// Skinny problems (N <= 2: the output layers and the back-prop into the two action inputs): one warp per output row,
// lanes stride over k, all loads of the row issued before the first use, warp-shuffle reduction.  A must be k-contiguous.
__global__ void __launch_bounds__(256)
gemm_skinny_kernel(const GemmBatch gb) {
  GemmProblem p = gb.p[blockIdx.y];
  if (blockIdx.z) gemm_shift(p, blockIdx.z, blockIdx.z * gb.ls_w, blockIdx.z * gb.ls_x);
  // the one or two weight columns are shared by the block's 8 rows: staged once in shared memory (K <= SKINNY_MAX_K)
  constexpr int SKINNY_MAX_K = 1024;
  __shared__ float bsm[2][SKINNY_MAX_K];
  const bool two = p.N > 1, staged = p.K <= SKINNY_MAX_K;
  if (staged) {
    for (int k = threadIdx.x; k < p.K; k += 256) {
      bsm[0][k] = __ldg(p.B + (long long)k * p.sBk);
      bsm[1][k] = two ? __ldg(p.B + (long long)k * p.sBk + p.sBn) : 0.0f;
    }
    __syncthreads();
  }
  const int m = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (m >= p.M) return;
  float a0 = 0.0f, a1 = 0.0f;
  const float* arow = p.A + (long long)m * p.sAm;
  for (int kb = 0; kb < p.K; kb += 512) {  // 16 k-values per lane and pass: all loads of the row are issued before the first FMA
    float av[16], b0[16], b1[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int k = kb + i * 32 + lane;
      av[i] = (k < p.K) ? __ldg(arow + k) : 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int k = kb + i * 32 + lane;
      const bool ok = k < p.K;
      if (staged) { b0[i] = ok ? bsm[0][k] : 0.0f; b1[i] = ok ? bsm[1][k] : 0.0f; }
      else {
        b0[i] = ok ? __ldg(p.B + (long long)k * p.sBk) : 0.0f;
        b1[i] = (ok && two) ? __ldg(p.B + (long long)k * p.sBk + p.sBn) : 0.0f;
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) { a0 = fmaf(av[i], b0[i], a0); a1 = fmaf(av[i], b1[i], a1); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
  if (lane == 0) {
    p.C[m * p.ldc] = gemm_epilogue(p, m, 0, a0);
    if (two) p.C[m * p.ldc + 1] = gemm_epilogue(p, m, 1, a1);
  }
}

// second pass of every split-K product: out[i] = sum_s ws[s*stride + i], fixed order (deterministic, unlike atomics)
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ ws, long long stride, int splits, float* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = ws[i];
  for (int s = 1; s < splits; ++s) acc += ws[(long long)s * stride + i];
  out[i] = acc;
}
// ---- large-batch helpers (B >= SPLITK_MIN_BATCH): the thin products around the 250x500 contractions are streaming
// passes over [B][width] activations, so they get streaming kernels instead of tiled GEMMs.

// Weighted column sums over a slab of rows: J == 0: ws[slab][n] = sum_b Z[b][n]          (bias gradient beside a tensor-core dW)
//                                           J >= 1: ws[slab][n*J + j] = sum_b Z[b][n] w[b][j]   (dW of an output layer, Flux layout
//                                                   [in][out=J]) followed by ws[slab][N*J + j] = sum_b w[b][j] (its bias gradient)
// Block = 32 columns x 8 row lanes; the row lanes meet in shared memory in a fixed order.
template <int J>
__global__ void __launch_bounds__(256)
wcolsum_partial_kernel(const float* __restrict__ Z, long long ld, int B, int N, const float* __restrict__ w, int rows_per, long long stride,
                       float* __restrict__ ws, long long pop_stride, float* __restrict__ out_final, unsigned* __restrict__ counters) {
  constexpr int JJ = J > 0 ? J : 1;
  constexpr int CHUNK = 256;  // rows whose weights are staged in shared memory at a time
  Z += (long long)blockIdx.z * pop_stride; ws += (long long)blockIdx.z * pop_stride;  // learner of a population (one slab: writes the gradient itself)
  if (J > 0) w += (long long)blockIdx.z * pop_stride;
  __shared__ float red[8][32][JJ];
  __shared__ float wsm[CHUNK * JJ];
  __shared__ int is_last;
  const int c = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + c;
  const int r0 = blockIdx.y * rows_per, r1 = min(B, r0 + rows_per);
  float acc[JJ], bsum = 0.0f;
#pragma unroll
  for (int j = 0; j < JJ; ++j) acc[j] = 0.0f;
  for (int cb = r0; cb < r1; cb += CHUNK) {
    const int ce = min(r1, cb + CHUNK);
    if (J > 0) {
      __syncthreads();
      for (int e = threadIdx.x; e < (ce - cb) * J; e += 256) wsm[e] = w[(long long)cb * J + e];
      __syncthreads();
      if (blockIdx.x == 0 && c < J) for (int r = cb + rl; r < ce; r += 8) bsum += wsm[(r - cb) * J + c];  // bias gradient: sum_b w[b][j]
    }
    if (n < N) {
#pragma unroll 8
      for (int r = cb + rl; r < ce; r += 8) {
        const float z = Z[(long long)r * ld + n];
        if (J == 0) acc[0] += z;
        else {
#pragma unroll
          for (int j = 0; j < JJ; ++j) acc[j] = fmaf(z, wsm[(r - cb) * J + j], acc[j]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < JJ; ++j) red[rl][c][j] = acc[j];
  __syncthreads();
  float* out = ws + (long long)blockIdx.y * stride;
  if (rl == 0 && n < N) {
#pragma unroll
    for (int j = 0; j < JJ; ++j) {
      float t = red[0][c][j];
#pragma unroll
      for (int q = 1; q < 8; ++q) t += red[q][c][j];
      out[(long long)n * JJ + j] = t;
    }
  }
  if (J > 0 && blockIdx.x == 0) {
    __syncthreads();
    red[rl][c][0] = bsum;
    __syncthreads();
    if (rl == 0 && c < J) {
      float u = red[0][c][0];
#pragma unroll
      for (int q = 1; q < 8; ++q) u += red[q][c][0];
      out[(long long)N * J + c] = u;
    }
  }
  if (gridDim.y == 1) return;  // a single slab wrote the result itself
  // several slabs: the last block of this column group to finish adds the slabs' partial sums in slab order (deterministic)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned old = atomicAdd(&counters[blockIdx.x], 1u);
    is_last = (old == gridDim.y - 1);
    if (is_last) counters[blockIdx.x] = 0u;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int e = threadIdx.x; e < 32 * JJ; e += 256) {
    const int cc = e / JJ, j = e - cc * JJ, nn = blockIdx.x * 32 + cc;
    if (nn >= N) continue;
    float t = 0.0f;
    for (unsigned sl = 0; sl < gridDim.y; ++sl) t += __ldcg(ws + (long long)sl * stride + (long long)nn * JJ + j);
    out_final[(long long)nn * JJ + j] = t;
  }
  if (J > 0 && blockIdx.x == 0 && threadIdx.x < J) {
    float t = 0.0f;
    for (unsigned sl = 0; sl < gridDim.y; ++sl) t += __ldcg(ws + (long long)sl * stride + (long long)N * J + threadIdx.x);
    out_final[(long long)N * J + threadIdx.x] = t;
  }
}

// First layer for many rows (K = 9 or 11 inputs): Y[m][n] = relu(b[n] + sum_k X[m][k] W[k][n]), up to 3 problems per launch.
// A thread keeps its 4 weight columns in registers and walks 8 rows; stores are 16-byte, coalesced along n.
struct L1Batch { const float* X[3]; const float* W[3]; const float* bias[3]; float* Y[3]; int K[3]; int M, N, ldx, ldy, count; long long ls_w, ls_x; };
__global__ void __launch_bounds__(256)
l1_fwd_kernel(const L1Batch a) {
  const int learner = blockIdx.z / a.count, z = blockIdx.z - learner * a.count, K = a.K[z];  // grid.z = learner * count + problem
  const float* __restrict__ X = a.X[z] + learner * a.ls_x; const float* __restrict__ W = a.W[z] + learner * a.ls_w;
  const float* __restrict__ bias = a.bias[z] + learner * a.ls_w;
  float* __restrict__ Y = a.Y[z] + learner * a.ls_x;
  __shared__ float xs[32][12];
  const int m0 = blockIdx.x * 32;
  for (int e = threadIdx.x; e < 32 * 12; e += 256) {
    const int r = e / 12, k = e - r * 12;
    xs[r][k] = (m0 + r < a.M && k < K) ? X[(long long)(m0 + r) * a.ldx + k] : 0.0f;
  }
  const int n = (blockIdx.y * 64 + (threadIdx.x & 63)) * 4, rg = threadIdx.x >> 6;
  float w[12][4], bv[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    bv[u] = (n + u < a.N) ? bias[n + u] : 0.0f;
#pragma unroll
    for (int k = 0; k < 12; ++k) w[k][u] = (k < K && n + u < a.N) ? W[(long long)k * a.N + n + u] : 0.0f;
  }
  __syncthreads();
  if (n >= a.N) return;
#pragma unroll 4
  for (int i = 0; i < 8; ++i) {
    const int r = rg * 8 + i, m = m0 + r;
    if (m >= a.M) break;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 12; ++k) {
      const float x = xs[r][k];
#pragma unroll
      for (int u = 0; u < 4; ++u) o[u] = fmaf(x, w[k][u], o[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) { o[u] += bv[u]; o[u] = o[u] > 0.0f ? o[u] : 0.0f; }
    float* y = Y + (long long)m * a.ldy + n;
    if (n + 3 < a.N) *reinterpret_cast<float4*>(y) = make_float4(o[0], o[1], o[2], o[3]);
    else {
#pragma unroll
      for (int u = 0; u < 4; ++u) if (n + u < a.N) y[u] = o[u];
    }
  }
}

// Back-propagation through an output layer with J <= 2 outputs: dX[b][n] = relu'(H[b][n]) * sum_j dZ[b][j] W[n][j]
// (Flux weight Wt[in=n][out=j]).  One thread per 4 columns; H and dX share the leading dimension ld (multiple of 4).
template <int J>
__global__ void __launch_bounds__(256)
outer_mask_kernel(const float* __restrict__ dZ, const float* __restrict__ W, const float* __restrict__ H, long long ld, int B, int N,
                  float* __restrict__ dX, long long pop_stride) {
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");   // the dX product after it sets itself up under this kernel (tc_gemm.cu)
  {  // blockIdx.y = learner of a population
    const long long lo = (long long)blockIdx.y * pop_stride;
    dZ += lo; W += lo; H += lo; dX += lo;
  }
  const unsigned n4 = (unsigned)(N + 3) / 4u;
  const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;   // B * n4 < 2^31 (checked by the launcher): 32-bit division
  if (e >= (unsigned)B * n4) return;
  const int b = (int)(e / n4), n = (int)(e - (unsigned)b * n4) * 4;
  float dz[J];
#pragma unroll
  for (int j = 0; j < J; ++j) dz[j] = dZ[(long long)b * J + j];
  float o[4], hv[4];
  const float* hrow = H + (long long)b * ld + n;
  if (n + 3 < N) { const float4 t = *reinterpret_cast<const float4*>(hrow); hv[0] = t.x; hv[1] = t.y; hv[2] = t.z; hv[3] = t.w; }
  else {
#pragma unroll
    for (int u = 0; u < 4; ++u) hv[u] = (n + u < N) ? hrow[u] : 0.0f;
  }
  float wv[4 * J];  // W[n..n+3][0..J-1] is contiguous: J 16-byte loads when aligned
  if (n + 3 < N && (reinterpret_cast<uintptr_t>(W) & 15) == 0) {
#pragma unroll
    for (int q = 0; q < J; ++q) {
      const float4 t = *reinterpret_cast<const float4*>(W + (long long)n * J + q * 4);
      wv[q * 4 + 0] = t.x; wv[q * 4 + 1] = t.y; wv[q * 4 + 2] = t.z; wv[q * 4 + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 4 * J; ++e) wv[e] = (n + e / J < N) ? W[(long long)n * J + e] : 0.0f;
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    float v = 0.0f;
#pragma unroll
    for (int j = 0; j < J; ++j) v = fmaf(dz[j], wv[u * J + j], v);
    o[u] = hv[u] > 0.0f ? v : 0.0f;
  }
  float* x = dX + (long long)b * ld + n;
  if (n + 3 < N) *reinterpret_cast<float4*>(x) = make_float4(o[0], o[1], o[2], o[3]);
  else {
#pragma unroll
    for (int u = 0; u < 4; ++u) if (n + u < N) x[u] = o[u];
  }
}

// ----------------------------------------------------------------------------- learner state
struct LayerDims { int in, out; long long w_off, b_off; };
struct NetDims { LayerDims l[3]; long long n_params; };

// struct DdpgCtrl: ddpg_fused.h (the fused critic pass samples the minibatch itself)
#define DP_MAX_WORLD 16
#define DP_TIMEOUT_NS 4000000000ull
// peers of a data-parallel learner: rank r's flat gradient buffer and flag array, mapped into this process (CUDA IPC over NVLink)
// box[r]: rank r's exchange box = DP_BOX_FLAG_WORDS flag words (one per source rank), then [DP_MAX_WORLD][in_stride] inbound gradient sums
struct DpPeers { unsigned* box[DP_MAX_WORLD]; long long in_stride; unsigned long long timeout_ns; int world, rank; };
#define DP_BOX_FLAG_WORDS 64ll

struct Ddpg {
  int device;
  cudaStream_t stream;
  DdpgParams p;
  NetDims dims[2];       // 0 actor-shaped, 1 critic-shaped
  float* net[4];         // flat params
  float* grad[2];        // flat grads (actor, critic) — contiguous: grad[1] then grad[0] in gradbuf
  float* gradbuf;
  float* adam_m[2]; float* adam_v[2];
  double beta_pow[2][2];
  long long n_updates;
  float* norm;           // [18] s_min | s_max
  // minibatch + activations (B rows)
  float *xs, *xs2, *xspi, *r, *done;
  float *t_h1, *t_h2, *c_h1, *c_h2, *a_h1, *a_h2, *tc_h1, *tc_h2, *p_h1, *p_h2;
  float *q, *y, *dq, *qpi;
  float *dz2, *dz1, *dzp2, *dzp1, *dza3, *dza2, *dza1;
  float* loss_scratch;   // [2]
  DdpgCtrl* ctrl;
  int32_t* idx_dev; long long idx_cap;
  // act() scratch (n rows)
  float *act_x, *act_h1, *act_h2, *act_y; long long act_cap;
  cudaGraph_t graph; cudaGraphExec_t graph_exec; 
  float* dqpi;     // [B] constant -1/B: d(-mean q)/dq
  bool ctrl_init;
  int ld1, ld2;    // leading dimensions of the [B][l1] / [B][l2] activation buffers (l1, l2 rounded up to 32 floats = 128 bytes)
  bool tc;         // layer-2 contractions on TF32 tensor cores (use_tensor_cores, batch >= 256, operands 16-byte aligned)
  bool chain;      // one learner in tensor-core mode at widths l1 <= 256, l2 <= 512: a net's whole forward pass is ONE kernel (tc_fwd_chain)
  unsigned* counters;  // [WS_COUNTERS] arrival counters of the fused slab reductions (zero between kernels)
  float* ws;       // split-K workspace (tensor-core dW, SIMT dW with K = batch >= 1024, bias-gradient partial sums)
  long long ws_floats;
  // Large batches / populations: the weight-gradient products of a backward pass (dW3, dW2, their bias sums) are off the dX critical
  // path; they run on a side stream (a parallel branch of the update's graph) with their own workspace and arrival counters.
  cudaStream_t side; cudaEvent_t ev_fork, ev_mid, ev_join; float* ws_side; unsigned* counters_side;
  // population: `pop` independent learners in one handle.  Every float buffer above lives in one slab per learner
  // (learner l's copy is l*pop_stride floats behind learner 0's), so a launch covers all learners through blockIdx.
  int pop, sel;            // sel: the learner get/set/init/losses address (ddpg_select_learner)
  long long pop_stride;
  float* slab;
  const float** rings_dev; // [pop] replay ring of every learner (device array)
  long long idx_stride;    // ints between consecutive learners' host-supplied minibatch indices
  long long act_stride;    // floats between consecutive learners' act() scratch blocks
  // data-parallel learner over NVLink peer memory (ddpg_dp_export / ddpg_dp_connect / ddpg_update_dp)
  DpPeers dp;
  bool dp_on;
  unsigned* dp_box;        // this rank's exchange box (allocated by ddpg_dp_export; written by the peers)
  void* dp_opened[2 * DP_MAX_WORLD]; int dp_n_opened;
  cudaGraph_t graph_dp; cudaGraphExec_t graph_dp_exec;
  // ddpg_episode scratch: a, scaled [2][N], s_prev [9][N], r [N]
  float *ep_a, *ep_scaled, *ep_sprev, *ep_r; double* ep_r64; long long ep_cap;
  // cluster-fused small-batch update (csrc/ddpg_fused.cu): per-cluster partial gradients [batch/8][n_params] of actor / critic
  bool fused; float* parts[2];
  bool rollout_ok;   // widths within the shared-memory plan of the persistent cluster kernel (ddpg_rollout: one learner; ddpg_evaluate: any)
  // best actor of every learner (run_episodes' best_run, DDPG.jl:282-289): its own allocation outside the slabs, learner l's copy
  // best_stride floats behind learner 0's; best_score [P] Float64 (start -100000, the reference's), best_run [P]
  float* best; long long best_stride; double* best_score; int32_t* best_run;
  int noise_kind; float ou_theta, ou_mu, ou_dt;   // ddpg_set_noise
  DdpgHparams* hp;   // [pop] host copy of every learner's ctrl->hp (ddpg_get_hparams; σ_eff of the one-learner cluster kernels)
  bool hp_stale;     // ddpg_exploit rewrote ctrl->hp on the device: ddpg_get_hparams reloads hp before it answers
  float* ou_x; long long ou_cap;                   // OUNoise.X of every instance of ddpg_episode's environment ([2][N])
  // prioritized replay (ddpg_set_prioritized): the updates draw from every learner's sum tree (trees_dev, staged beside rings_dev),
  // weigh the critic's dq and write the rows' priorities back.  per_knobs: α, β, ε on the device (handle-wide, written in stream order);
  // per_slot / per_leaf [pop][B]: the slot each row of the current update drew and its priority at the draw
  bool per; float per_host[3]; float* per_knobs; float** trees_dev; int32_t* per_slot; float* per_leaf;
  // n-step returns (ddpg_set_nstep): nstep > 1 gathers every row by walking its memory's successor links (links_dev, staged beside
  // rings_dev); nstep_knob: n on the device (handle-wide, written in stream order), so only a switch between 1 and > 1 re-captures
  int nstep; int* nstep_knob; const int32_t** links_dev;
};
static inline int round_ld(int x) { return (x + 31) & ~31; }  // activation rows start on 128-byte lines: one L2 request per TMA box row
#ifndef TC_MIN_ROWS
#define TC_MIN_ROWS 256
#endif
#define SPLITK_MIN_BATCH 1024
#define CHAIN_MIN_BATCH 2048
#define SPLITK_MAX 32
#define WS_COUNTERS 1024

static void make_dims(NetDims& d, int in, int l1, int l2, int out) {
  const int ins[3] = {in, l1, l2}, outs[3] = {l1, l2, out};
  long long off = 0;
  for (int k = 0; k < 3; ++k) {
    d.l[k].in = ins[k]; d.l[k].out = outs[k];
    d.l[k].w_off = off; off += (long long)ins[k] * outs[k];
    d.l[k].b_off = off; off += outs[k];
  }
  d.n_params = off;
}
static inline const NetDims& dims_of(const Ddpg* h, int net) { return h->dims[(net == DDPG_NET_CRITIC || net == DDPG_NET_CRITIC_TARGET) ? 1 : 0]; }
// every slab buffer starts on a 256-byte boundary: W2 rows are 16-byte aligned iff l2 and both W2 offsets are multiples of 4 floats
static inline bool w2_vec16(const Ddpg* h) { return h->p.l2 % 4 == 0 && h->dims[0].l[1].w_off % 4 == 0 && h->dims[1].l[1].w_off % 4 == 0; }

extern "C" int32_t ddpg_default_params(DdpgParams* p) {
  REQUIRE(p, SHEMS_ERR_INVALID, "ddpg_default_params: NULL");
  memset(p, 0, sizeof(*p));
  p->state_size = 9; p->action_size = 2; p->l1 = 250; p->l2 = 500; p->batch = 120;  // README.md:68-86
  p->gamma = 0.99f; p->tau = 1e-3f; p->lr_actor = 1e-4f; p->lr_critic = 1e-3f;
  p->adam_beta1 = 0.9; p->adam_beta2 = 0.999; p->adam_eps = 1e-8;
  p->act_lo[0] = p->act_lo[1] = 0.0f; p->act_hi[0] = p->act_hi[1] = 1.0f;
  p->use_tensor_cores = 0;
  return SHEMS_OK;
}

#define DMALLOC(ptr, count)                                                                         \
  do {                                                                                              \
    cudaError_t _e = cudaMalloc((void**)&(ptr), sizeof(*(ptr)) * (size_t)(count));                  \
    if (_e == cudaSuccess) _e = cudaMemset((ptr), 0, sizeof(*(ptr)) * (size_t)(count));             \
    if (_e != cudaSuccess) { shems_set_error("ddpg: cudaMalloc(%s) -> %s", #ptr, cudaGetErrorString(_e)); ddpg_destroy(h); return SHEMS_ERR_CUDA; } \
  } while (0)

extern "C" int32_t ddpg_create(const DdpgParams* p, int32_t device, Ddpg** out) {
  REQUIRE(p && out, SHEMS_ERR_INVALID, "ddpg_create: NULL argument");
  REQUIRE(p->state_size == 9 && p->action_size == 2, SHEMS_ERR_INVALID, "ddpg_create: STATE_SIZE/ACTION_SIZE must be 9/2 (shems_LU1)");
  REQUIRE(p->l1 >= 1 && p->l2 >= 1 && p->batch >= 1, SHEMS_ERR_INVALID, "ddpg_create: l1=%d l2=%d batch=%d", p->l1, p->l2, p->batch);
  REQUIRE(p->population >= 0 && p->population <= 4096, SHEMS_ERR_INVALID, "ddpg_create: population=%d", p->population);
  const int pop = p->population > 1 ? p->population : 1;
  REQUIRE(pop == 1 || p->batch < SPLITK_MIN_BATCH, SHEMS_ERR_INVALID,
          "ddpg_create: a population of learners runs the small-batch path (batch < %d)", SPLITK_MIN_BATCH);
  REQUIRE(shems_device_count() > 0, SHEMS_ERR_CUDA, "ddpg_create: no CUDA device (this library has no CPU fallback)");
  GUARD(device);
  Ddpg* h = new (std::nothrow) Ddpg();
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_create: out of host memory");
  memset(h, 0, sizeof(*h));
  h->device = device; h->p = *p; h->pop = pop; h->p.population = pop;
  const int S = p->state_size, A = p->action_size, B = p->batch, C = S + A;
  make_dims(h->dims[0], S, p->l1, p->l2, A);
  make_dims(h->dims[1], C, p->l1, p->l2, 1);
  h->ld1 = round_ld(p->l1); h->ld2 = round_ld(p->l2);
  const int l1 = h->ld1, l2 = h->ld2;  // allocation strides
  // W2 of both nets must start on a 16-byte boundary and have 16-byte rows for the TMA descriptors
  h->tc = p->use_tensor_cores && w2_vec16(h);
  h->ws_floats = (long long)SPLITK_MAX * ((long long)p->l1 * p->l2 + p->l2 + (long long)C * p->l1 + p->l1 + (long long)p->l2 * A + A);
  DMALLOC(h->ws, h->ws_floats);
  DMALLOC(h->counters, WS_COUNTERS);
  DMALLOC(h->ws_side, h->ws_floats);
  DMALLOC(h->counters_side, WS_COUNTERS);
  {
    cudaError_t e_ = cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking);
    if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&h->ev_mid, cudaEventDisableTiming);
    if (e_ == cudaSuccess) e_ = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    if (e_ != cudaSuccess) { shems_set_error("ddpg_create: side stream/events -> %s", cudaGetErrorString(e_)); ddpg_destroy(h); return SHEMS_ERR_CUDA; }
  }
  if (h->tc) { int s_ = tc_gemm_prepare(); if (s_) { ddpg_destroy(h); return s_; } }
  {
    const char* ev = getenv("SHEMS_TC_CHAIN");
    // measured (tools/time_ddpg_large.py): 196 vs 249 us per update at B = 8192, 291 vs 407 at 16384, 153 vs 171 at 4096 and 130 vs 141 at 2048, but 120 vs 116 at 1024 (few
    // tiles per net leave the per-tile latency of the chain kernels exposed) — on from CHAIN_MIN_BATCH rows; SHEMS_TC_CHAIN=0 / 1 forces it off / on
    // a population (grid.y = learner): the same rule on the rows of all learners together
    h->chain = h->tc && p->l1 <= 256 && p->l2 <= 512 && p->l2 % 4 == 0 &&
               (ev ? ev[0] != '0' : (long long)p->batch * pop >= (pop > 1 ? CHAIN_MIN_BATCH / 2 : CHAIN_MIN_BATCH));   // populations: 10 x 120 rows already win (132 vs 135 us)
  }
  // one slab per learner: every buffer is carved at a 256-byte boundary (TMA operands, float4 accesses)
  const long long na = h->dims[0].n_params, nc = h->dims[1].n_params;
  struct Carve { float** ptr; long long count; };
  const Carve plan[] = {
      {&h->net[0], na}, {&h->net[1], nc}, {&h->net[2], na}, {&h->net[3], nc}, {&h->gradbuf, ((nc + 63) & ~63ll) + na},
      {&h->adam_m[0], na}, {&h->adam_v[0], na}, {&h->adam_m[1], nc}, {&h->adam_v[1], nc}, {&h->norm, 18},
      {&h->xs, (long long)B * C}, {&h->xs2, (long long)B * C}, {&h->xspi, (long long)B * C}, {&h->r, B}, {&h->done, B},
      {&h->t_h1, (long long)B * l1}, {&h->t_h2, (long long)B * l2}, {&h->c_h1, (long long)B * l1}, {&h->c_h2, (long long)B * l2},
      {&h->a_h1, (long long)B * l1}, {&h->a_h2, (long long)B * l2}, {&h->tc_h1, (long long)B * l1}, {&h->tc_h2, (long long)B * l2},
      {&h->p_h1, (long long)B * l1}, {&h->p_h2, (long long)B * l2}, {&h->q, B}, {&h->y, B}, {&h->dq, B}, {&h->qpi, B},
      {&h->dz2, (long long)B * l2}, {&h->dz1, (long long)B * l1}, {&h->dzp2, (long long)B * l2}, {&h->dzp1, (long long)B * l1},
      {&h->dza3, (long long)B * A}, {&h->dza2, (long long)B * l2}, {&h->dza1, (long long)B * l1}, {&h->loss_scratch, 2}, {&h->dqpi, B}};
  long long off = 0;
  for (const Carve& c : plan) off += (c.count + 63) & ~63ll;
  h->pop_stride = off;
  DMALLOC(h->slab, off * pop);
  off = 0;
  for (const Carve& c : plan) { *c.ptr = h->slab + off; off += (c.count + 63) & ~63ll; }
  h->grad[1] = h->gradbuf; h->grad[0] = h->gradbuf + ((nc + 63) & ~63ll);  // the actor part starts on a 256-byte boundary (TMA stores of dW)
  // one learner at a small batch (the reference's B = 120): the update runs as two cluster kernels (SHEMS_DDPG_FUSED=0 opts out)
  if (pop == 1 && !h->tc && ddpg_fused_shape_ok(B, p->l1, p->l2)) {
    const char* ev = getenv("SHEMS_DDPG_FUSED");
    int s_ = ddpg_fused_prepare();
    if (s_) { ddpg_destroy(h); return s_; }
    DMALLOC(h->parts[0], (long long)(B / FUSED_ROWS) * na);
    DMALLOC(h->parts[1], (long long)(B / FUSED_ROWS) * nc);
    h->fused = !(ev && ev[0] == '0');
  }
  if (ddpg_fused_shape_ok(FUSED_ROWS, p->l1, p->l2)) {
    int s_ = actor_rollout_prepare();
    if (s_) { ddpg_destroy(h); return s_; }
    h->rollout_ok = true;
  }
  DMALLOC(h->ctrl, pop);
  DMALLOC(h->rings_dev, pop);
  DMALLOC(h->trees_dev, pop);
  DMALLOC(h->per_knobs, 3);
  DMALLOC(h->links_dev, pop);
  DMALLOC(h->nstep_knob, 1);
  DMALLOC(h->per_slot, (long long)pop * B);
  DMALLOC(h->per_leaf, (long long)pop * B);
  h->best_stride = (na + 63) & ~63ll;   // every copy starts on a 256-byte boundary (float4 copies)
  DMALLOC(h->best, h->best_stride * pop);
  DMALLOC(h->best_score, pop);
  DMALLOC(h->best_run, pop);
  {
    std::vector<double> bs((size_t)pop, -100000.0);   // best_score = -100000 (DDPG_reinforce_charger_v1.jl), best_run = 0, zero weights
    const cudaError_t e_ = cudaMemcpy(h->best_score, bs.data(), sizeof(double) * (size_t)pop, cudaMemcpyHostToDevice);
    if (e_ != cudaSuccess) { shems_set_error("ddpg_create: best_score -> %s", cudaGetErrorString(e_)); ddpg_destroy(h); return SHEMS_ERR_CUDA; }
  }
  h->hp = (DdpgHparams*)malloc(sizeof(DdpgHparams) * (size_t)pop);
  if (!h->hp) { shems_set_error("ddpg_create: out of host memory"); ddpg_destroy(h); return SHEMS_ERR_INVALID; }
  {
    std::vector<float> c((size_t)B, -1.0f / (float)B);
    float nm[18];
    for (int k = 0; k < 9; ++k) { nm[k] = 0.0f; nm[9 + k] = 1.0f; }
    std::vector<DdpgCtrl> ctl((size_t)pop);
    memset(ctl.data(), 0, sizeof(DdpgCtrl) * (size_t)pop);
    for (int l = 0; l < pop; ++l) {
      cudaMemcpy(h->dqpi + l * h->pop_stride, c.data(), sizeof(float) * (size_t)B, cudaMemcpyHostToDevice);
      cudaMemcpy(h->norm + l * h->pop_stride, nm, sizeof(nm), cudaMemcpyHostToDevice);
      for (int n = 0; n < 2; ++n) {
        ctl[l].bp[n][0] = p->adam_beta1; ctl[l].bp[n][1] = p->adam_beta2;
        ctl[l].rc[n][0] = 1.0 / (1.0 - p->adam_beta1); ctl[l].rc[n][1] = 1.0 / (1.0 - p->adam_beta2);
      }
      h->hp[l] = DdpgHparams{{p->lr_critic, p->lr_actor}, p->gamma, p->tau, 1.0f};
      ctl[l].hp = h->hp[l];
    }
    cudaMemcpy(h->ctrl, ctl.data(), sizeof(DdpgCtrl) * (size_t)pop, cudaMemcpyHostToDevice);
  }
  for (int n = 0; n < 2; ++n) { h->beta_pow[n][0] = p->adam_beta1; h->beta_pow[n][1] = p->adam_beta2; }
  h->nstep = 1;
  {
    const cudaError_t e_ = cudaMemcpy(h->nstep_knob, &h->nstep, sizeof(int), cudaMemcpyHostToDevice);
    if (e_ != cudaSuccess) { shems_set_error("ddpg_create: nstep -> %s", cudaGetErrorString(e_)); ddpg_destroy(h); return SHEMS_ERR_CUDA; }
  }
  *out = h;
  return SHEMS_OK;
}

extern "C" int32_t ddpg_destroy(Ddpg* h) {
  if (!h) return SHEMS_OK;
  GUARD(h->device);
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->graph) cudaGraphDestroy(h->graph);
  cudaFree(h->slab);
  cudaFree(h->parts[0]); cudaFree(h->parts[1]);
  cudaFree(h->act_x);  // act() scratch: one allocation (x | h1 | h2 | y per learner)
  cudaFree(h->ep_a);   // episode scratch: one allocation
  cudaFree(h->ou_x);
  if (h->graph_dp_exec) cudaGraphExecDestroy(h->graph_dp_exec);
  if (h->graph_dp) cudaGraphDestroy(h->graph_dp);
  for (int i = 0; i < h->dp_n_opened; ++i) cudaIpcCloseMemHandle(h->dp_opened[i]);
  cudaFree(h->best); cudaFree(h->best_score); cudaFree(h->best_run);
  cudaFree(h->ctrl); cudaFree(h->idx_dev); cudaFree(h->ws); cudaFree((void*)h->rings_dev); cudaFree(h->trees_dev); cudaFree(h->dp_box); cudaFree(h->counters);
  cudaFree(h->ws_side); cudaFree(h->counters_side);
  cudaFree(h->per_knobs); cudaFree(h->per_slot); cudaFree(h->per_leaf);
  cudaFree(h->nstep_knob); cudaFree((void*)h->links_dev);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_mid) cudaEventDestroy(h->ev_mid);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->side) cudaStreamDestroy(h->side);
  free(h->hp);
  delete h;
  return SHEMS_OK;
}

// get/set/init-style calls address one learner of a population (default 0)
extern "C" int32_t ddpg_select_learner(Ddpg* h, int32_t learner) {
  REQUIRE(h && learner >= 0 && learner < h->pop, SHEMS_ERR_INVALID, "ddpg_select_learner: learner=%d outside 0..%d", learner, h ? h->pop - 1 : -1);
  h->sel = learner;
  return SHEMS_OK;
}
extern "C" int32_t ddpg_population(const Ddpg* h) { return h ? h->pop : 0; }
static inline long long sel_off(const Ddpg* h) { return (long long)h->sel * h->pop_stride; }

// η_actor, η_critic, γ, τ and the exploration-noise scale of the selected learner.  The write is enqueued on the handle's stream:
// updates and act() calls enqueued before it use the old values, everything enqueued after it the new ones.  Captured update graphs
// read the values from the control block, so nothing is re-captured.
extern "C" int32_t ddpg_set_hparams(Ddpg* h, float lr_actor, float lr_critic, float gamma, float tau, float noise_scale) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_set_hparams: NULL handle");
  REQUIRE(isfinite(lr_actor) && isfinite(lr_critic) && isfinite(gamma) && isfinite(tau) && isfinite(noise_scale), SHEMS_ERR_INVALID,
          "ddpg_set_hparams: values must be finite (lr_actor=%g lr_critic=%g gamma=%g tau=%g noise_scale=%g)", (double)lr_actor, (double)lr_critic,
          (double)gamma, (double)tau, (double)noise_scale);
  REQUIRE(lr_actor >= 0.0f && lr_critic >= 0.0f && noise_scale >= 0.0f, SHEMS_ERR_INVALID,
          "ddpg_set_hparams: lr_actor=%g lr_critic=%g noise_scale=%g must be >= 0", (double)lr_actor, (double)lr_critic, (double)noise_scale);
  REQUIRE(gamma >= 0.0f && gamma <= 1.0f && tau >= 0.0f && tau <= 1.0f, SHEMS_ERR_INVALID, "ddpg_set_hparams: gamma=%g tau=%g outside [0, 1]",
          (double)gamma, (double)tau);
  GUARD(h->device);
  const DdpgHparams v{{lr_critic, lr_actor}, gamma, tau, noise_scale};
  // pageable source: the runtime stages the copy before returning (no synchronisation, which a data-parallel peer could be waiting on)
  CUDA_TRY(cudaMemcpyAsync((char*)(h->ctrl + h->sel) + offsetof(DdpgCtrl, hp), &v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
  h->hp[h->sel] = v;
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_hparams(Ddpg* h, float* lr_actor, float* lr_critic, float* gamma, float* tau, float* noise_scale) {
  REQUIRE(h && lr_actor && lr_critic && gamma && tau && noise_scale, SHEMS_ERR_INVALID, "ddpg_get_hparams: NULL argument");
  if (h->hp_stale) {   // after ddpg_exploit: the device values of every learner (a ddpg_set_hparams enqueued later has landed too)
    GUARD(h->device);
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaMemcpy2D(h->hp, sizeof(DdpgHparams), (const char*)h->ctrl + offsetof(DdpgCtrl, hp), sizeof(DdpgCtrl), sizeof(DdpgHparams),
                          (size_t)h->pop, cudaMemcpyDeviceToHost));
    h->hp_stale = false;
  }
  const DdpgHparams& v = h->hp[h->sel];
  *lr_actor = v.eta[1]; *lr_critic = v.eta[0]; *gamma = v.gamma; *tau = v.tau; *noise_scale = v.noise_scale;
  return SHEMS_OK;
}

extern "C" int32_t ddpg_set_stream(Ddpg* h, void* s) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_set_stream: NULL handle");
  h->stream = (cudaStream_t)s;
  return SHEMS_OK;
}
extern "C" int32_t ddpg_sync(Ddpg* h) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_sync: NULL handle");
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (h->dp_on) {  // a gradient exchange that gave up (a peer never arrived) skipped its update on purpose: tell the caller
    int e = 0;
    CUDA_TRY(cudaMemcpy(&e, &h->ctrl->dp_error, sizeof(int), cudaMemcpyDeviceToHost));
    REQUIRE(e == 0, SHEMS_ERR_STATE, "ddpg_sync: a data-parallel gradient exchange timed out (a peer did not arrive); the replicas' updates were skipped");
  }
  return SHEMS_OK;
}
extern "C" int32_t ddpg_set_fused(Ddpg* h, int32_t on) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_set_fused: NULL handle");
  GUARD(h->device);
  const bool want = on != 0 && h->parts[0] && h->parts[1];   // shapes outside the fused plan keep the tiled-GEMM path
  if (want != h->fused) {
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }   // re-captured by the next ddpg_update
    if (h->graph_dp_exec) { cudaGraphExecDestroy(h->graph_dp_exec); h->graph_dp_exec = nullptr; }
    h->fused = want;
  }
  return h->fused ? 1 : 0;
}
extern "C" int32_t ddpg_set_prioritized(Ddpg* h, int32_t on, float alpha, float beta, float eps) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_set_prioritized: NULL handle");
  if (on) {
    REQUIRE(isfinite(alpha) && isfinite(beta) && isfinite(eps) && alpha >= 0.0f && beta >= 0.0f && beta <= 1.0f && eps > 0.0f, SHEMS_ERR_INVALID,
            "ddpg_set_prioritized: alpha=%g beta=%g eps=%g (finite, alpha >= 0, beta in [0, 1], eps > 0)", (double)alpha, (double)beta, (double)eps);
    REQUIRE(!h->dp_on, SHEMS_ERR_STATE, "ddpg_set_prioritized: not available for a data-parallel learner");
  }
  GUARD(h->device);
  if (on) {
    const float v[3] = {alpha, beta, eps};
    // pageable source: staged before the call returns; ordered like ddpg_set_hparams, so a captured update reads the new values
    CUDA_TRY(cudaMemcpyAsync(h->per_knobs, v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
    memcpy(h->per_host, v, sizeof(v));
  }
  if ((on != 0) != h->per) {   // the update's graph gains or loses the prioritized kernels: re-captured by the next update
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
    h->per = on != 0;
  }
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_prioritized(Ddpg* h, int32_t* on, float* alpha, float* beta, float* eps) {
  REQUIRE(h && on && alpha && beta && eps, SHEMS_ERR_INVALID, "ddpg_get_prioritized: NULL argument");
  *on = h->per ? 1 : 0;
  *alpha = h->per_host[0]; *beta = h->per_host[1]; *eps = h->per_host[2];
  return SHEMS_OK;
}

extern "C" int32_t ddpg_set_nstep(Ddpg* h, int32_t n) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_set_nstep: NULL handle");
  REQUIRE(n >= 1 && n <= NSTEP_MAX, SHEMS_ERR_INVALID, "ddpg_set_nstep: n=%d outside 1..%d", n, NSTEP_MAX);
  REQUIRE(n == 1 || !h->dp_on, SHEMS_ERR_STATE, "ddpg_set_nstep: not available for a data-parallel learner");
  GUARD(h->device);
  // pageable source: staged before the call returns; ordered like ddpg_set_hparams, so a captured update reads the new n
  CUDA_TRY(cudaMemcpyAsync(h->nstep_knob, &n, sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if ((n > 1) != (h->nstep > 1)) {   // the update's graph gains or loses the walking gather: re-captured by the next update
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
  }
  h->nstep = n;
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_nstep(const Ddpg* h) { return h ? h->nstep : 0; }

extern "C" int64_t ddpg_num_params(const Ddpg* h, int32_t net) {
  return (h && net >= 0 && net <= DDPG_NET_ACTOR_BEST) ? dims_of(h, net).n_params : 0;   // ACTOR_BEST has the actor's shape
}
// the selected learner's copy of a net; DDPG_NET_ACTOR_BEST: its best-actor slot (outside the slab)
static inline float* net_of(const Ddpg* h, int net) {
  return net == DDPG_NET_ACTOR_BEST ? h->best + (long long)h->sel * h->best_stride : h->net[net] + sel_off(h);
}

extern "C" int32_t ddpg_set_layer(Ddpg* h, int32_t net, int32_t layer, const float* w_host, const float* b_host) {
  REQUIRE(h && net >= 0 && net <= DDPG_NET_ACTOR_BEST && layer >= 0 && layer < 3, SHEMS_ERR_INVALID, "ddpg_set_layer: net=%d layer=%d", net, layer);
  GUARD(h->device);
  const LayerDims& L = dims_of(h, net).l[layer];
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (w_host) CUDA_TRY(cudaMemcpy(net_of(h, net) + L.w_off, w_host, sizeof(float) * (size_t)L.in * L.out, cudaMemcpyHostToDevice));
  if (b_host) CUDA_TRY(cudaMemcpy(net_of(h, net) + L.b_off, b_host, sizeof(float) * (size_t)L.out, cudaMemcpyHostToDevice));
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_layer(Ddpg* h, int32_t net, int32_t layer, float* w_host, float* b_host) {
  REQUIRE(h && net >= 0 && net <= DDPG_NET_ACTOR_BEST && layer >= 0 && layer < 3, SHEMS_ERR_INVALID, "ddpg_get_layer: net=%d layer=%d", net, layer);
  GUARD(h->device);
  const LayerDims& L = dims_of(h, net).l[layer];
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (w_host) CUDA_TRY(cudaMemcpy(w_host, net_of(h, net) + L.w_off, sizeof(float) * (size_t)L.in * L.out, cudaMemcpyDeviceToHost));
  if (b_host) CUDA_TRY(cudaMemcpy(b_host, net_of(h, net) + L.b_off, sizeof(float) * (size_t)L.out, cudaMemcpyDeviceToHost));
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_grad(Ddpg* h, int32_t net, int32_t layer, float* w_host, float* b_host) {
  REQUIRE(h && (net == DDPG_NET_ACTOR || net == DDPG_NET_CRITIC) && layer >= 0 && layer < 3, SHEMS_ERR_INVALID, "ddpg_get_grad: net=%d layer=%d", net, layer);
  GUARD(h->device);
  const LayerDims& L = dims_of(h, net).l[layer];
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (w_host) CUDA_TRY(cudaMemcpy(w_host, h->grad[net] + sel_off(h) + L.w_off, sizeof(float) * (size_t)L.in * L.out, cudaMemcpyDeviceToHost));
  if (b_host) CUDA_TRY(cudaMemcpy(b_host, h->grad[net] + sel_off(h) + L.b_off, sizeof(float) * (size_t)L.out, cudaMemcpyDeviceToHost));
  return SHEMS_OK;
}
extern "C" int32_t ddpg_set_norm(Ddpg* h, const float* s_min_host, const float* s_max_host) {
  REQUIRE(h && s_min_host && s_max_host, SHEMS_ERR_INVALID, "ddpg_set_norm: NULL argument");
  GUARD(h->device);
  float nm[18];
  memcpy(nm, s_min_host, sizeof(float) * 9);
  memcpy(nm + 9, s_max_host, sizeof(float) * 9);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(h->norm + sel_off(h), nm, sizeof(nm), cudaMemcpyHostToDevice));
  return SHEMS_OK;
}

// βp of both optimisers of learner l (Flux.ADAM state: βp = β^t after t - 1 updates) into the device control block, with the
// reciprocals the optimiser kernels use; [0] = critic, [1] = actor
static int write_opt_state(Ddpg* h, int l, double c_b1, double c_b2, double a_b1, double a_b2) {
  double v[8] = {c_b1, c_b2, a_b1, a_b2, 1.0 / (1.0 - c_b1), 1.0 / (1.0 - c_b2), 1.0 / (1.0 - a_b1), 1.0 / (1.0 - a_b2)};
  CUDA_TRY(cudaMemcpyAsync((char*)(h->ctrl + l) + offsetof(DdpgCtrl, bp), v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));   // v lives on this stack frame
  return SHEMS_OK;
}

// init: glorot_uniform hidden layers / U(-3e-3, 3e-3) last layer / zero bias (DDPG.jl:21-22, 30-46)
__global__ void ddpg_init_kernel(float* __restrict__ w, long long n, int in, int out, int last, unsigned long long seed, unsigned layer_id) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  uint32_t r[4];
  philox4x32_10(seed, (uint64_t)e, layer_id, STREAM_INIT, r);
  const float u = (float)(r[0] >> 8) * (1.0f / 16777216.0f);
  if (!last) w[e] = __fmul_rn(__fsub_rn(u, 0.5f), sqrtf(24.0f / (float)(in + out)));
  else w[e] = __fsub_rn(__fmul_rn(6e-3f, u), 3e-3f);
}
extern "C" int32_t ddpg_init(Ddpg* h, uint64_t seed) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_init: NULL handle");
  GUARD(h->device);
  for (int l = 0; l < h->pop; ++l) {  // learner l of a population draws from Philox(seed + l): independent seeds
    const long long lo = (long long)l * h->pop_stride;
    for (int n = 0; n < 2; ++n) {
      const NetDims& d = h->dims[n];
      CUDA_TRY(cudaMemsetAsync(h->net[n] + lo, 0, sizeof(float) * (size_t)d.n_params, h->stream));
      for (int k = 0; k < 3; ++k) {
        const long long nw = (long long)d.l[k].in * d.l[k].out;
        ddpg_init_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, h->stream>>>(h->net[n] + lo + d.l[k].w_off, nw, d.l[k].in, d.l[k].out, k == 2,
                                                                              seed + (uint64_t)l, (unsigned)(n * 3 + k));
      }
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaMemcpyAsync(h->net[n + 2] + lo, h->net[n] + lo, sizeof(float) * (size_t)d.n_params, cudaMemcpyDeviceToDevice, h->stream));  // deepcopy :38,:46
      // fresh optimisers (opt_crit = ADAM(η_crit), opt_act = ADAM(η_act), input.jl:126-127): no moments, βp = β
      CUDA_TRY(cudaMemsetAsync(h->adam_m[n] + lo, 0, sizeof(float) * (size_t)d.n_params, h->stream));
      CUDA_TRY(cudaMemsetAsync(h->adam_v[n] + lo, 0, sizeof(float) * (size_t)d.n_params, h->stream));
    }
    { const int st_ = write_opt_state(h, l, h->p.adam_beta1, h->p.adam_beta2, h->p.adam_beta1, h->p.adam_beta2); if (st_) return st_; }
  }
  h->n_updates = 0;
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- minibatch gather + normalize
// getData() + normalize() (memory_plotting_saving.jl:31-42, 55-57): builds xs = [s_n; a], xs2[:, :9] = s'_n,
// xspi[:, :9] = s_n, r, done for the B sampled transitions.  src arrays are SoA with leading dim `ld`.
// src: either the replay ring (tiled layout, ring != NULL) or caller-supplied SoA arrays with leading dim ld (direct).
// One thread per (sample j, state field k): thread k == 0 also moves a, r, done.
// PER: the ring rows come from the learner's sum tree (trees[blockIdx.y], ring_draw_prioritized; caller-supplied indices as they are),
// and thread k == 0 of row j records its slot and priority in per_slot / per_leaf [pop][B] for ddpg_per_kernel.
// NSTEP: every thread of row j walks the chain from the drawn record (ring_nstep over links[blockIdx.y], n = *nstep, the learner's γ):
// s and a stay the drawn record's, s' is the last record's, and thread k == 0 sums r and folds γ^{k-1} into done.
template <bool PER, bool NSTEP = false>
__device__ __forceinline__ void gather_body(const float* const* __restrict__ rings, const float* __restrict__ rs, const float* __restrict__ ra,
                                            const float* __restrict__ rr, const float* __restrict__ rs2, const float* __restrict__ rd, long long ld,
                                            DdpgCtrl* __restrict__ ctrl, const int32_t* __restrict__ idx, long long idx_stride,
                                            const float* __restrict__ norm, int B, float* __restrict__ xs, float* __restrict__ xs2,
                                            float* __restrict__ xspi, float* __restrict__ r, float* __restrict__ done, long long pop_stride,
                                            const float* const* __restrict__ trees, int32_t* __restrict__ per_slot, float* __restrict__ per_leaf,
                                            const int32_t* const* __restrict__ links = nullptr, const int* __restrict__ nstep = nullptr) {
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");   // the forward-chain launch after it stages its weights under this kernel
  const unsigned g = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = g / 9, k = g % 9;  // unsigned: k is known to be < 9, which folds ring_field's field-range tests
  if (j >= B) return;
  {  // blockIdx.y = learner of a population: own ring, control block, indices and slab
    const long long lo = (long long)blockIdx.y * pop_stride;
    ctrl += blockIdx.y; idx += (long long)blockIdx.y * idx_stride;
    norm += lo; xs += lo; xs2 += lo; xspi += lo; r += lo; done += lo;
  }
  const float* ring = rings ? rings[blockIdx.y] : nullptr;
  float sv, s2v, a0 = 0.f, a1 = 0.f, rv = 0.f, dv = 0.f;
  if (ring) {
    const long long len = ctrl->len, head = ctrl->head, cap = ctrl->cap;
    long long slot;
    if (PER) {
      const float* tree = trees[blockIdx.y];
      const long long p2 = prio_p2(cap);
      float leaf;
      if (ctrl->use_idx) {
        slot = ring_slot(idx[(long long)ctrl->idx_cursor * B + j], head, len, cap);
        leaf = tree[p2 + slot];
      } else {
        slot = ring_draw_prioritized(tree, p2, ctrl->seed, j, ctrl->update, B, &leaf);
      }
      if (k == 0) { per_slot[(long long)blockIdx.y * B + j] = (int32_t)slot; per_leaf[(long long)blockIdx.y * B + j] = leaf; }
    } else {
      const long long li = ctrl->use_idx ? idx[(long long)ctrl->idx_cursor * B + j] : ring_draw(ctrl->seed, j, ctrl->update, len);
      slot = ring_slot(li, head, len, cap);
    }
    const float* q = ring + ring_base(slot);
    const float* row = ring_row(ring_table(ring), q);
    sv = ring_field(q, row, RING_S + k); s2v = ring_field(q, row, RING_S2 + k);
    if (k == 0) {
      a0 = ring_field(q, row, RING_A); a1 = ring_field(q, row, RING_A + 1); rv = ring_field(q, row, RING_R); dv = ring_field(q, row, RING_DONE);
    }
    if (NSTEP) {
      const RingNstep w = ring_nstep(ring, ring_table(ring), links[blockIdx.y], slot, *nstep, ctrl->hp.gamma, k == 0);
      const float* q2 = ring + ring_base(w.last);
      s2v = ring_field(q2, ring_row(ring_table(ring), q2), RING_S2 + k);
      if (k == 0) { rv = w.r; dv = w.done; }
    }
  } else {
    sv = rs[k * ld + j]; s2v = rs2[k * ld + j];
    if (k == 0) { a0 = ra[j]; a1 = ra[ld + j]; rv = rr[j]; dv = rd ? rd[j] : 0.0f; }
  }
  const float den = __fadd_rn(__fsub_rn(norm[9 + k], norm[k]), 1e-8f);
  const float sn = __fdiv_rn(__fsub_rn(sv, norm[k]), den);
  const float s2n = __fdiv_rn(__fsub_rn(s2v, norm[k]), den);
  xs[j * 11 + k] = sn; xspi[j * 11 + k] = sn; xs2[j * 11 + k] = s2n;
  if (k == 0) { xs[j * 11 + 9] = a0; xs[j * 11 + 10] = a1; r[j] = rv; done[j] = dv; }
}
__global__ void __launch_bounds__(128)
ddpg_gather_kernel(const float* const* __restrict__ rings, const float* __restrict__ rs, const float* __restrict__ ra, const float* __restrict__ rr,
                   const float* __restrict__ rs2, const float* __restrict__ rd, long long ld, DdpgCtrl* __restrict__ ctrl,
                   const int32_t* __restrict__ idx, long long idx_stride, const float* __restrict__ norm, int B, float* __restrict__ xs,
                   float* __restrict__ xs2, float* __restrict__ xspi, float* __restrict__ r, float* __restrict__ done, long long pop_stride) {
  gather_body<false>(rings, rs, ra, rr, rs2, rd, ld, ctrl, idx, idx_stride, norm, B, xs, xs2, xspi, r, done, pop_stride, nullptr, nullptr, nullptr);
}
__global__ void __launch_bounds__(128)
ddpg_gather_per_kernel(const float* const* __restrict__ rings, DdpgCtrl* __restrict__ ctrl, const int32_t* __restrict__ idx, long long idx_stride,
                       const float* __restrict__ norm, int B, float* __restrict__ xs, float* __restrict__ xs2, float* __restrict__ xspi,
                       float* __restrict__ r, float* __restrict__ done, long long pop_stride, const float* const* __restrict__ trees,
                       int32_t* __restrict__ per_slot, float* __restrict__ per_leaf) {
  gather_body<true>(rings, nullptr, nullptr, nullptr, nullptr, nullptr, 0, ctrl, idx, idx_stride, norm, B, xs, xs2, xspi, r, done, pop_stride, trees,
                    per_slot, per_leaf);
}
// n-step instantiations: uniform draws and PER draws, each row walked over its memory's successor links
__global__ void __launch_bounds__(128)
ddpg_gather_nstep_kernel(const float* const* __restrict__ rings, DdpgCtrl* __restrict__ ctrl, const int32_t* __restrict__ idx, long long idx_stride,
                         const float* __restrict__ norm, int B, float* __restrict__ xs, float* __restrict__ xs2, float* __restrict__ xspi,
                         float* __restrict__ r, float* __restrict__ done, long long pop_stride, const int32_t* const* __restrict__ links,
                         const int* __restrict__ nstep) {
  gather_body<false, true>(rings, nullptr, nullptr, nullptr, nullptr, nullptr, 0, ctrl, idx, idx_stride, norm, B, xs, xs2, xspi, r, done, pop_stride,
                           nullptr, nullptr, nullptr, links, nstep);
}
__global__ void __launch_bounds__(128)
ddpg_gather_per_nstep_kernel(const float* const* __restrict__ rings, DdpgCtrl* __restrict__ ctrl, const int32_t* __restrict__ idx, long long idx_stride,
                             const float* __restrict__ norm, int B, float* __restrict__ xs, float* __restrict__ xs2, float* __restrict__ xspi,
                             float* __restrict__ r, float* __restrict__ done, long long pop_stride, const float* const* __restrict__ trees,
                             int32_t* __restrict__ per_slot, float* __restrict__ per_leaf, const int32_t* const* __restrict__ links,
                             const int* __restrict__ nstep) {
  gather_body<true, true>(rings, nullptr, nullptr, nullptr, nullptr, nullptr, 0, ctrl, idx, idx_stride, norm, B, xs, xs2, xspi, r, done, pop_stride,
                          trees, per_slot, per_leaf, links, nstep);
}

// Prioritized replay between the TD target and the critic's backward pass, one block per learner (blockIdx.y):
//   w_j = RN32((leaf_j len / root)^-β / max_k (leaf_k len / root)^-β)  (Float64, the max over the B rows);  dq_j = RN32(dq_j w_j)
//   p_j = RN32((|RN32(y_j - q_j)| + ε)^α);  each drawn slot's leaf = the largest p_j of the rows that drew it;  p_max = max(p_max, p_j)
//   then the nodes above the drawn leaves, level by level (every node from its two children, as a full rebuild computes it)
#define PER_THREADS 1024
__global__ void __launch_bounds__(PER_THREADS)
ddpg_per_kernel(float* const* __restrict__ trees, const DdpgCtrl* __restrict__ ctrl, const float* __restrict__ knobs, const int32_t* __restrict__ per_slot,
                const float* __restrict__ per_leaf, const float* __restrict__ q, const float* __restrict__ y, float* __restrict__ dq, int B,
                long long pop_stride) {
  __shared__ double red_w[PER_THREADS / 32];
  __shared__ float red_p[PER_THREADS / 32];
  const long long lo = (long long)blockIdx.y * pop_stride;
  float* const tree = trees[blockIdx.y];
  ctrl += blockIdx.y; per_slot += (long long)blockIdx.y * B; per_leaf += (long long)blockIdx.y * B;
  q += lo; y += lo; dq += lo;
  const long long len = ctrl->len, p2 = prio_p2(ctrl->cap);
  const float alpha = knobs[0], beta = knobs[1], eps = knobs[2];
  const float root = tree[1];
  double wmax = 0.0;
  float pmax = 0.0f;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    wmax = fmax(wmax, ring_is_weight(per_leaf[j], len, root, beta));
    pmax = fmaxf(pmax, ring_priority(y[j], q[j], alpha, eps));
  }
  for (int o = 16; o > 0; o >>= 1) {
    wmax = fmax(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
  }
  if ((threadIdx.x & 31) == 0) { red_w[threadIdx.x >> 5] = wmax; red_p[threadIdx.x >> 5] = pmax; }
  __syncthreads();   // also: every thread has read the root before a leaf changes
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { wmax = fmax(wmax, red_w[i]); pmax = fmaxf(pmax, red_p[i]); }
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    dq[j] = __fmul_rn(dq[j], (float)(ring_is_weight(per_leaf[j], len, root, beta) / wmax));
    tree[p2 + per_slot[j]] = 0.0f;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < B; j += blockDim.x)   // priorities are >= 0: their bits order as signed integers
    atomicMax(reinterpret_cast<int*>(tree + p2 + per_slot[j]), __float_as_int(ring_priority(y[j], q[j], alpha, eps)));
  if (threadIdx.x == 0) prio_header(tree)[PRIO_PMAX] = fmaxf(prio_header(tree)[PRIO_PMAX], pmax);
  for (long long level = p2 >> 1; level >= 1; level >>= 1) {
    __syncthreads();
    const int shift = 63 - __clzll(p2 / level);
    for (int j = threadIdx.x; j < B; j += blockDim.x) {
      const long long n = (p2 + per_slot[j]) >> shift;
      tree[n] = __fadd_rn(tree[2 * n], tree[2 * n + 1]);
    }
  }
}

// ----------------------------------------------------------------------------- Adam + Polyak
// Flux.Optimise.ADAM apply! + update! with Float64 β, ϵ (element math in Float64, stored Float32), then
// soft_update! p_t = (1-τ) p_t + τ p_m for the target of the same net (DDPG.jl:99-108).
// βp = β^t is read from the device control block so graph replays stay valid.
template <bool FAST>
__device__ __forceinline__ float adam_element(float x, float gj, float* __restrict__ m, float* __restrict__ v, double b1, double b2, double eps, float eta,
                                              double c1, double c2, double r1, double r2) {
  const float g2 = __fmul_rn(gj, gj);
  if (FAST) {  // tensor-core mode: the gradients carry TF32 noise (1e-3 relative), so the whole step is evaluated in IEEE fp32
               // (no DDIV / DSQRT, no Float32<->Float64 conversions on the XU pipe)
    const float mj = __fmaf_rn((float)b1, *m, __fmul_rn((float)(1.0 - b1), gj));
    const float vj = __fmaf_rn((float)b2, *v, __fmul_rn((float)(1.0 - b2), g2));
    *m = mj; *v = vj;
    const float qm = __fmul_rn(mj, (float)r1), qv = __fmul_rn(vj, (float)r2);
    return __fsub_rn(x, __fmul_rn(__fdiv_rn(qm, __fadd_rn(__fsqrt_rn(qv), (float)eps)), eta));
  }
  const float mj = (float)__dadd_rn(__dmul_rn(b1, (double)*m), __dmul_rn(1.0 - b1, (double)gj));
  const float vj = (float)__dadd_rn(__dmul_rn(b2, (double)*v), __dmul_rn(1.0 - b2, (double)g2));
  *m = mj; *v = vj;
  double qm = __dmul_rn((double)mj, r1); qm = __fma_rn(__fma_rn(-qm, c1, (double)mj), r1, qm);   // mt / (1 - βp[1])
  double qv = __dmul_rn((double)vj, r2); qv = __fma_rn(__fma_rn(-qv, c2, (double)vj), r2, qv);   // vt / (1 - βp[2])
  const double d = __dmul_rn(__ddiv_rn(qm, __dadd_rn(__dsqrt_rn(qv), eps)), (double)eta);
  return __fsub_rn(x, (float)d);
}
// the last block to finish the final kernel of an update advances the device-side counters
// (`βp .= βp .* β` of Flux.ADAM for both optimisers, the Philox update counter, the host-index cursor)
__device__ __forceinline__ void adam_advance(DdpgCtrl* ctrl, double b1, double b2) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned done = atomicAdd(&ctrl->blocks_done, 1u);
    if (done == gridDim.x - 1) {
      ctrl->blocks_done = 0;
      ctrl->update += 1; ctrl->idx_cursor += 1;
      for (int o = 0; o < 2; ++o) {
        ctrl->bp[o][0] *= b1; ctrl->bp[o][1] *= b2;
        ctrl->rc[o][0] = 1.0 / (1.0 - ctrl->bp[o][0]); ctrl->rc[o][1] = 1.0 / (1.0 - ctrl->bp[o][1]);
      }
    }
  }
}
template <bool FAST>
__global__ void __launch_bounds__(256)
adam_polyak_kernel(float* __restrict__ x, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n, double b1,
                   double b2, double eps, DdpgCtrl* __restrict__ ctrl, int opt, float* __restrict__ target,
                   float* __restrict__ target2, const float* __restrict__ model2, long long n2, int advance, float gscale, long long pop_stride) {
  {  // blockIdx.y = learner of a population
    const long long lo = (long long)blockIdx.y * pop_stride;
    x += lo; g += lo; m += lo; v += lo; ctrl += blockIdx.y;
    if (target) target += lo;
    if (target2) { target2 += lo; model2 += lo; }
  }
  // mt / (1 - βp[1]) and vt / (1 - βp[2]) divide every element by the same two numbers: with r = RN(1/c) the sequence
  // q = a*r; e = fma(-q, c, a); q' = fma(e, r, q) is the correctly rounded quotient (Markstein), at 3 DFMA instead of a DDIV
  const double c1 = 1.0 - ctrl->bp[opt][0], c2 = 1.0 - ctrl->bp[opt][1];
  const double r1 = ctrl->rc[opt][0], r2 = ctrl->rc[opt][1];
  // this learner's η of optimiser `opt` and τ (ddpg_set_hparams) are read inside every loop, after the element's own loads: read once
  // up front, they are moved to uniform registers before the first element load is issued, and each thread waits for them first
#define ETA_TAU const float eta = ctrl->hp.eta[opt], tau = ctrl->hp.tau, omt = __fsub_rn(1.0f, tau); (void)eta
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long j0 = 0, k0 = 0;  // scalar loops start here (FAST: after the float4 body)
  if (FAST) {  // memory-bound fp32 variant: 16-byte accesses (every slab buffer starts on a 256-byte boundary)
    const long long n4 = n >> 2;
    for (long long q = tid; q < n4; q += stride) {
      float4 xv = reinterpret_cast<float4*>(x)[q], mv = reinterpret_cast<float4*>(m)[q], vv = reinterpret_cast<float4*>(v)[q];
      const float4 gv = reinterpret_cast<const float4*>(g)[q];
      ETA_TAU;
      float xs[4] = {xv.x, xv.y, xv.z, xv.w}, ms[4] = {mv.x, mv.y, mv.z, mv.w}, vs[4] = {vv.x, vv.y, vv.z, vv.w};
      const float gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
        xs[u] = adam_element<true>(xs[u], (gscale == 1.0f) ? gs[u] : __fmul_rn(gs[u], gscale), &ms[u], &vs[u], b1, b2, eps, eta, c1, c2, r1, r2);
      reinterpret_cast<float4*>(x)[q] = make_float4(xs[0], xs[1], xs[2], xs[3]);
      reinterpret_cast<float4*>(m)[q] = make_float4(ms[0], ms[1], ms[2], ms[3]);
      reinterpret_cast<float4*>(v)[q] = make_float4(vs[0], vs[1], vs[2], vs[3]);
      if (target) {
        float4 t = reinterpret_cast<float4*>(target)[q];
        t.x = __fadd_rn(__fmul_rn(omt, t.x), __fmul_rn(tau, xs[0])); t.y = __fadd_rn(__fmul_rn(omt, t.y), __fmul_rn(tau, xs[1]));
        t.z = __fadd_rn(__fmul_rn(omt, t.z), __fmul_rn(tau, xs[2])); t.w = __fadd_rn(__fmul_rn(omt, t.w), __fmul_rn(tau, xs[3]));
        reinterpret_cast<float4*>(target)[q] = t;
      }
    }
    j0 = n4 << 2;
    const long long m4 = n2 >> 2;
    for (long long q = tid; q < m4; q += stride) {
      float4 t = reinterpret_cast<float4*>(target2)[q];
      const float4 w = reinterpret_cast<const float4*>(model2)[q];
      ETA_TAU;
      t.x = __fadd_rn(__fmul_rn(omt, t.x), __fmul_rn(tau, w.x)); t.y = __fadd_rn(__fmul_rn(omt, t.y), __fmul_rn(tau, w.y));
      t.z = __fadd_rn(__fmul_rn(omt, t.z), __fmul_rn(tau, w.z)); t.w = __fadd_rn(__fmul_rn(omt, t.w), __fmul_rn(tau, w.w));
      reinterpret_cast<float4*>(target2)[q] = t;
    }
    k0 = m4 << 2;
  }
  for (long long j = j0 + tid; j < n; j += stride) {
    const float gj = (gscale == 1.0f) ? g[j] : __fmul_rn(g[j], gscale);  // data-parallel: mean of the ranks' summed gradients
    ETA_TAU;
    const float xn = adam_element<FAST>(x[j], gj, m + j, v + j, b1, b2, eps, eta, c1, c2, r1, r2);
    x[j] = xn;
    if (target) target[j] = __fadd_rn(__fmul_rn(omt, target[j]), __fmul_rn(tau, xn));
  }
  // second Polyak pair: the critic target moves together with the actor step (DDPG.jl:142-143)
  for (long long j = k0 + tid; j < n2; j += stride) {
    ETA_TAU;
    target2[j] = __fadd_rn(__fmul_rn(omt, target2[j]), __fmul_rn(tau, model2[j]));
  }
#undef ETA_TAU
  if (advance) adam_advance(ctrl, b1, b2);
}

// Cluster-fused small-batch path: the gradient of element j is the sum of `nparts` per-cluster partial copies, added here in a
// fixed order (deterministic) — the reduction over the minibatch that ends the fused backward pass — then ADAM (+ Polyak) as
// above.  The summed gradient is also stored to g_out (ddpg_get_grad).
__global__ void __launch_bounds__(256)
adam_polyak_parts_kernel(float* __restrict__ x, const float* __restrict__ parts, int nparts, long long part_stride, float* __restrict__ g_out,
                         float* __restrict__ m, float* __restrict__ v, long long n, double b1, double b2, double eps,
                         DdpgCtrl* __restrict__ ctrl, int opt, float* __restrict__ target, float* __restrict__ target2,
                         const float* __restrict__ model2, long long n2, int advance) {
  // the fused actor pass is a programmatic dependent of ADAM(critic): its actor forward pass may run beside this kernel
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
  const double c1 = 1.0 - ctrl->bp[opt][0], c2 = 1.0 - ctrl->bp[opt][1];
  const double r1 = ctrl->rc[opt][0], r2 = ctrl->rc[opt][1];
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // one element per thread at the reference's sizes: every load of the element (partials, parameter, moments, both Polyak
  // pairs) is issued before the first use, the partials eight at a time
  for (long long j = tid; j < n || j < n2; j += stride) {
    const bool in1 = j < n, in2 = j < n2;
    float t2 = 0.0f, w2 = 0.0f, xj = 0.0f, tj = 0.0f;
    if (in2) { t2 = target2[j]; w2 = model2[j]; }
    if (in1) { xj = x[j]; if (target) tj = target[j]; }
    // η and τ are read here rather than before the loop: live across it they cost an 8-byte spill at this kernel's 48 registers
    const float eta = ctrl->hp.eta[opt], tau = ctrl->hp.tau, omt = __fsub_rn(1.0f, tau);
    if (in1) {
      float gj = 0.0f;
      for (int c0 = 0; c0 < nparts; c0 += 8) {
        float t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = (c0 + q < nparts) ? parts[(long long)(c0 + q) * part_stride + j] : 0.0f;
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (c0 + q < nparts) gj = (c0 + q == 0) ? t[q] : __fadd_rn(gj, t[q]);
      }
      g_out[j] = gj;
      const float xn = adam_element<false>(xj, gj, m + j, v + j, b1, b2, eps, eta, c1, c2, r1, r2);
      x[j] = xn;
      if (target) target[j] = __fadd_rn(__fmul_rn(omt, tj), __fmul_rn(tau, xn));
    }
    if (in2) target2[j] = __fadd_rn(__fmul_rn(omt, t2), __fmul_rn(tau, w2));
  }
  if (advance) adam_advance(ctrl, b1, b2);
}

// Data-parallel learner: gradient all-reduce FUSED into the optimiser step, over NVLink peer memory (no NCCL call, no
// reduced-gradient round trip through HBM).  Every rank runs this ONE kernel per gradient segment at the same point of its stream,
// with the same grid.  The exchange is PUSH style:
//   0. every block sums its elements of this rank's gradient (cluster-fused path: the fixed-order sum of the per-cluster partial
//      copies), keeps them in the flat gradient buffer and writes them into row [rank] of every peer's inbox — posted NVLink
//      stores that travel while the rest of the grid is still summing;
//   1. the LAST block to finish step 0 publishes "rank `rank` is in": st.release.sys of the exchange number into every peer's flag
//      word [rank];
//   2. every block waits for all peers' flags in its own, LOCAL flag words (ld.acquire.sys);
//   3. element j: g = (sum over ranks r = 0..W-1 of [own sum | inbox[r][j]]) / W — all LOCAL loads, summed in rank order (the same
//      order everywhere -> bit-identical replicas); then ADAM (+ Polyak) as in adam_polyak_kernel.
// (Round 1 / early round 2 pulled: after the flags, W peer loads per element — one more NVLink round trip on every element's
// critical path, and at W = 8 a read burst of 7 x 516 KB per rank right when everybody waits for it.)
// An inbox segment is rewritten two exchanges later (critic and actor segments alternate).  By then the writer has completed the
// exchange in between, i.e. has seen that exchange's flags of every peer, and a peer starts an exchange kernel only after its previous
// one — all its inbox reads — has finished: no second barrier is needed.
// A peer that never arrives: ONLY block 0 runs the clock; when it gives up it records the abort for this exchange number in the
// control block, every other block sees it in its wait loop (or, having passed it, before it applies anything: see below), and NO
// block applies the step (a half-updated parameter vector would silently break the replicas' identity).  dp_error stays set;
// ddpg_sync / ddpg_dp_status report it.
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ float ld_peer(const float* p) {  // never served from a stale local cache line; no memory clobber: independent
  float v;                                                   // loads may be issued back to back
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];\n" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ unsigned ld_relaxed_sys_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys(unsigned* p, unsigned v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_volatile_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.volatile.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// -DDP_TRACE (tools/time_dp.py --trace builds that variant): globaltimer stamps of block 0 / the publishing block per segment
#ifdef DP_TRACE
__device__ unsigned long long dp_trace[2][8];
#define DP_STAMP_T(i) do { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t_)); dp_trace[opt][i] = t_; } while (0)
#define DP_STAMP(i) do { if (threadIdx.x == 0) DP_STAMP_T(i); } while (0)
extern "C" __attribute__((visibility("default"))) int ddpg_dp_trace_read(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, dp_trace, sizeof(dp_trace));
}
#else
#define DP_STAMP(i) do { } while (0)
#define DP_STAMP_T(i) do { } while (0)
#endif
template <int W>
__global__ void __launch_bounds__(256)
adam_polyak_dp_kernel(const DpPeers peers, long long seg_off, const float* __restrict__ parts, int nparts, long long part_stride,
                      float* __restrict__ g_own, float* __restrict__ x, float* __restrict__ m, float* __restrict__ v, long long n, double b1,
                      double b2, double eps, DdpgCtrl* __restrict__ ctrl, int opt, float* __restrict__ target,
                      float* __restrict__ target2, const float* __restrict__ model2, long long n2, int advance) {
  __shared__ int ok_s, last_s;
  // the fused actor pass is a programmatic dependent of the critic exchange: its actor forward pass (which does not read the critic)
  // may run beside this kernel; all blocks of this grid are resident before the dependent can start, so the waits below stay safe
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
  const unsigned epoch = ctrl->dp_epoch + 1u;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int rank = peers.rank;
  if (threadIdx.x == 0) ok_s = 1;
  if (blockIdx.x == 0) DP_STAMP(0);
  // 0. this rank's sums of the block's elements: kept locally, pushed into row [rank] of every peer's inbox
  {
    float* out[W];
#pragma unroll
    for (int r = 0; r < W; ++r)
      out[r] = reinterpret_cast<float*>(peers.box[r] + DP_BOX_FLAG_WORDS) + (long long)rank * peers.in_stride + seg_off;
    for (long long j = tid0; j < n; j += stride) {
      float gj;
      if (parts) {
        gj = 0.0f;
        for (int c0 = 0; c0 < nparts; c0 += 8) {
          float t[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) t[q] = (c0 + q < nparts) ? parts[(long long)(c0 + q) * part_stride + j] : 0.0f;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (c0 + q < nparts) gj = (c0 + q == 0) ? t[q] : __fadd_rn(gj, t[q]);
        }
        g_own[j] = gj;
      } else {
        gj = g_own[j];
      }
#pragma unroll
      for (int r = 0; r < W; ++r)
        if (r != rank) out[r][j] = gj;
    }
  }
  // 1. the last block to get here publishes: its system-scope release covers every block's inbox stores (each block fenced them
  //    before it counted itself in).  Lane r tells rank r — W - 1 lanes = one ~2 us system round trip, not W - 1 serialised ones.
  //    (Measured and dropped: a flag per block — 500 blocks x (W - 1) release stores at once took 3.5-4 us each and the slowest
  //    10 us; one fence + relaxed flag stores — the relaxed stores reached the peer 10-16 us later.)
  __syncthreads();
  if (blockIdx.x == 0) DP_STAMP(1);
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned arrived = atomicAdd(&ctrl->dp_ready, 1u);
    last_s = (arrived == gridDim.x - 1);
    if (last_s) { ctrl->dp_ready = 0; DP_STAMP_T(2); }
  }
  __syncthreads();
  if (last_s && threadIdx.x < W && (int)threadIdx.x != rank) {
    st_release_sys(peers.box[threadIdx.x] + rank, epoch);
    if ((int)threadIdx.x == (rank == 0 ? 1 : 0)) DP_STAMP_T(3);
  }
  // 2. lane r waits for rank r's flag (local memory); block 0 alone decides to give up
  if (threadIdx.x < W && (int)threadIdx.x != rank) {
    const unsigned* f = peers.box[rank] + threadIdx.x;
    unsigned long long t0 = 0, t = 0;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t0));
    unsigned spins = 0;
    while ((int)(ld_acquire_sys(f) - epoch) < 0) {
      if ((++spins & 63u) == 0u) {
        if (ld_volatile_u32(&ctrl->dp_abort) == epoch) { ok_s = 0; break; }
        asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
        if (blockIdx.x == 0 && t - t0 > peers.timeout_ns) {
          if ((int)(ld_acquire_sys(f) - epoch) >= 0) break;   // it arrived after all
          ctrl->dp_abort = epoch; ctrl->dp_error = 1;
          __threadfence();
          ok_s = 0;
          break;
        }
        if (blockIdx.x != 0 && t - t0 > 4ull * peers.timeout_ns) { ok_s = 0; break; }   // backstop: block 0 never ran its clock
      }
    }
  }
  __syncthreads();
  if (blockIdx.x == 0) DP_STAMP(4);
  // Every block waits for the same W - 1 flags and only block 0 runs the clock, so the decision is the grid's: if block 0 gave up on this
  // exchange, a block whose own polls happened to see the flags later skips as well (dp_error is set; the replica must be restored).
  const bool ok = ok_s && ld_volatile_u32(&ctrl->dp_abort) != epoch;
  const double c1 = 1.0 - ctrl->bp[opt][0], c2 = 1.0 - ctrl->bp[opt][1];
  const double r1 = ctrl->rc[opt][0], r2 = ctrl->rc[opt][1];
  const float eta = ctrl->hp.eta[opt], tau = ctrl->hp.tau;
  const float omt = __fsub_rn(1.0f, tau), inv_w = 1.0f / (float)W;
  if (ok) {
    const float* in = reinterpret_cast<const float*>(peers.box[rank] + DP_BOX_FLAG_WORDS) + seg_off;
    for (long long j = tid0; j < n || j < n2; j += stride) {
      const bool in1 = j < n, in2 = j < n2;
      float t2 = 0.0f, w2 = 0.0f, xj = 0.0f, tj = 0.0f, gr[W];
      if (in1) {
#pragma unroll
        for (int r = 0; r < W; ++r) gr[r] = ld_peer((r == rank ? g_own : in + (long long)r * peers.in_stride) + j);   // local, past L1
        xj = x[j];
        if (target) tj = target[j];
      }
      if (in2) { t2 = target2[j]; w2 = model2[j]; }
      if (in1) {
        float gs = gr[0];
#pragma unroll
        for (int r = 1; r < W; ++r) gs = __fadd_rn(gs, gr[r]);
        const float xn = adam_element<false>(xj, __fmul_rn(gs, inv_w), m + j, v + j, b1, b2, eps, eta, c1, c2, r1, r2);
        x[j] = xn;
        if (target) target[j] = __fadd_rn(__fmul_rn(omt, tj), __fmul_rn(tau, xn));
      }
      if (in2) target2[j] = __fadd_rn(__fmul_rn(omt, t2), __fmul_rn(tau, w2));
    }
  }
  __syncthreads();
  if (blockIdx.x == 0) DP_STAMP(5);
  if (threadIdx.x == 0) {  // the last block closes this exchange
    __threadfence();
    const unsigned done = atomicAdd(&ctrl->dp_blocks_done, 1u);
    if (done == gridDim.x - 1) { ctrl->dp_blocks_done = 0; ctrl->dp_epoch = epoch; DP_STAMP(6); }
  }
  if (advance) adam_advance(ctrl, b1, b2);
}
// host-side dispatch on the world size (the gather loop is unrolled per W); grid: one element per thread, capped at the number
// of blocks that are co-resident (the blocks wait for one another in step 1)
static int dp_grid_cap = 0;
static int launch_adam_dp(cudaStream_t st, const DpPeers& peers, long long seg_off, const float* parts, int nparts, long long part_stride, float* g_own,
                          float* x, float* m, float* v, long long n, double b1, double b2, double eps, DdpgCtrl* ctrl, int opt,
                          float* target, float* target2, const float* model2, long long n2, int advance) {
#define DP_CASE(WW)                                                                                                                          \
  case WW: {                                                                                                                                 \
    if (!dp_grid_cap) {                                                                                                                      \
      int per_sm = 0, dev = 0, sms = 0;                                                                                                      \
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, adam_polyak_dp_kernel<WW>, 256, 0));                                   \
      CUDA_TRY(cudaGetDevice(&dev));                                                                                                         \
      CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));                                                           \
      dp_grid_cap = per_sm * sms > 0 ? per_sm * sms : 148;                                                                                   \
    }                                                                                                                                        \
    const long long want = ((n > n2 ? n : n2) + 255) / 256;                                                                                  \
    const unsigned grid = (unsigned)(want < dp_grid_cap ? want : dp_grid_cap);                                                               \
    adam_polyak_dp_kernel<WW><<<grid, 256, 0, st>>>(peers, seg_off, parts, nparts, part_stride, g_own, x, m, v, n, b1, b2, eps, ctrl, opt, target, \
                                                    target2, model2, n2, advance);                                                    \
  } break;
  switch (peers.world) {
    DP_CASE(1) DP_CASE(2) DP_CASE(3) DP_CASE(4) DP_CASE(5) DP_CASE(6) DP_CASE(7) DP_CASE(8) DP_CASE(16)
    default: shems_set_error("ddpg_update_dp: world size %d has no kernel instance (1-8, 16)", peers.world); return SHEMS_ERR_INVALID;
  }
#undef DP_CASE
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- update sequence
static inline GemmProblem gp_fwd(const float* X, long long ldx, int M, const float* net, const LayerDims& L, float* Y, long long ldy, int epi) {
  GemmProblem g; memset(&g, 0, sizeof(g));
  g.A = X; g.sAm = ldx; g.sAk = 1;
  g.B = net + L.w_off; g.sBk = L.out; g.sBn = 1;  // Wt[in][out]
  g.C = Y; g.ldc = ldy; g.M = M; g.N = L.out; g.K = L.in; g.epi = epi; g.bias = net + L.b_off;
  return g;
}
// dW[i][o] = sum_b X[b][i] dZ[b][o]   (+ db[o] = sum_b dZ[b][o])
static inline GemmProblem gp_dw(const float* X, long long ldx, const float* dZ, long long lddz, int B, const LayerDims& L, float* grad) {
  GemmProblem g; memset(&g, 0, sizeof(g));
  g.A = X; g.sAm = 1; g.sAk = ldx;
  g.B = dZ; g.sBk = lddz; g.sBn = 1;
  g.C = grad + L.w_off; g.ldc = L.out; g.M = L.in; g.N = L.out; g.K = B; g.epi = EPI_NONE; g.dbias = grad + L.b_off;
  return g;
}
// dX[b][i] = sum_o dZ[b][o] Wt[i][o]  (rows i0..i0+ni-1 of Wt), then the epilogue
static inline GemmProblem gp_dx(const float* dZ, long long lddz, int B, const float* net, const LayerDims& L, int i0, int ni, float* dX, long long lddx,
                                int epi, const float* aux, long long auxld) {
  GemmProblem g; memset(&g, 0, sizeof(g));
  g.A = dZ; g.sAm = lddz; g.sAk = 1;
  g.B = net + L.w_off + (long long)i0 * L.out; g.sBk = 1; g.sBn = L.out;
  g.C = dX; g.ldc = lddx; g.M = B; g.N = ni; g.K = L.out; g.epi = epi; g.aux = aux; g.auxld = auxld;
  return g;
}
static int launch_gemms(cudaStream_t st, const GemmProblem* ps, int count, int pop = 1, long long ls_w = 0, long long ls_x = 0) {
  GemmBatch gb; memset(&gb, 0, sizeof(gb));
  gb.count = count; gb.ksplit = 1; gb.pop = pop; gb.ls_w = ls_w; gb.ls_x = ls_x;
  bool skinny = true;
  int maxM = 1, maxN = 1;
  long long ctas32 = 0;
  for (int i = 0; i < count; ++i) {
    gb.p[i] = ps[i];
    skinny = skinny && ps[i].N <= 2 && ps[i].sAk == 1 && ps[i].dbias == nullptr && ps[i].K >= 32;
    maxM = max(maxM, ps[i].M); maxN = max(maxN, ps[i].N);
    ctas32 += (long long)((ps[i].M + 31) / 32) * ((ps[i].N + 31) / 32);
  }
  if (skinny) {
    gemm_skinny_kernel<<<dim3((maxM + 7) / 8, count, pop), 256, 0, st>>>(gb);
  } else if (ctas32 * pop < 296) {  // fewer than two CTAs per SM with 32x32 tiles: use 16x16 tiles (4x the CTAs, 1/4 of the serial work each)
    gemm_batch_kernel<16, 16><<<dim3((maxM + 15) / 16, (maxN + 15) / 16, count * pop), 128, 0, st>>>(gb);
  } else {
    gemm_batch_kernel<32, 32><<<dim3((maxM + 31) / 32, (maxN + 31) / 32, count * pop), 512, 0, st>>>(gb);
  }
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// the same problems for every learner of the handle, each on the weights and activations of its own slab
static inline int slab_gemms(const Ddpg* h, cudaStream_t st, const GemmProblem* ps, int count) {
  return launch_gemms(st, ps, count, h->pop, h->pop_stride, h->pop_stride);
}
#define TRY(x) do { int _s = (x); if (_s) return _s; } while (0)

// dW-type product (K = batch) with its bias gradient.  From SPLITK_MIN_BATCH rows on the batch dimension is split over
// blockIdx.z: every split writes [tile sums | column sums] into the workspace, splitk_reduce_kernel adds them in order.
static int launch_dw(Ddpg* h, cudaStream_t st, const GemmProblem& g, bool side = false) {
  const int B = g.K;
  float* const ws = side ? h->ws_side : h->ws;
  if (B < SPLITK_MIN_BATCH) return slab_gemms(h, st, &g, 1);
  const long long mn = (long long)g.M * g.N, stride = mn + g.N;
  REQUIRE(g.ldc == g.N && g.dbias == g.C + mn && g.epi == EPI_NONE, SHEMS_ERR_INVALID, "launch_dw: not a contiguous [W|b] gradient block");
  const int ksplit = min(SPLITK_MAX, B / 256);
  REQUIRE(stride * ksplit <= h->ws_floats, SHEMS_ERR_INVALID, "launch_dw: workspace too small");
  GemmBatch gb; memset(&gb, 0, sizeof(gb));
  gb.count = 1; gb.ksplit = ksplit; gb.split_stride = stride;
  gb.p[0] = g; gb.p[0].C = ws; gb.p[0].dbias = ws + mn;
  const long long ctas32 = (long long)((g.M + 31) / 32) * ((g.N + 31) / 32) * ksplit;
  if (ctas32 < 296) gemm_batch_kernel<16, 16><<<dim3((g.M + 15) / 16, (g.N + 15) / 16, ksplit), 128, 0, st>>>(gb);
  else gemm_batch_kernel<32, 32><<<dim3((g.M + 31) / 32, (g.N + 31) / 32, ksplit), 512, 0, st>>>(gb);
  CUDA_TRY(cudaGetLastError());
  splitk_reduce_kernel<<<(unsigned)((stride + 255) / 256), 256, 0, st>>>(ws, stride, ksplit, g.C, stride);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

// ---- layer-2 contractions on TF32 tensor cores (csrc/tc_gemm.cu); operands are used where they lie in HBM.  A population
// handle runs all learners' products in one launch (grid.z = learner): weights/gradients/activations of learner l sit
// l*pop_stride floats behind learner 0's; act() scratch uses its own stride (enqueue_forward's xstride).
// dX =(dZ · W^T) masked by relu'(H):  dZ [M][lddz] K-major, Wt[in][out] K-major (k = out)
static int tc_dx(const Ddpg* h, cudaStream_t st, const float* dZ, int lddz, int M, const float* net, const LayerDims& L, float* dX, int lddx, const float* H, int ldh) {
  TcOperand A{dZ, lddz, false}, Bo{net + L.w_off, L.out, false};
  TcBatch bt; bt.count = h->pop; bt.sA = bt.sB = bt.sD = bt.sAux = h->pop_stride;
  bt.pdl = true;   // a programmatic dependent of the outer_mask launch before it: its set-up (barriers, TMEM, tensor maps) runs under that kernel's tail
  return tc_gemm(st, A, Bo, dX, lddx, M, L.in, L.out, TC_EPI_RELU_MASK, nullptr, H, ldh, 1, nullptr, bt);
}
// dW = X^T · dZ (both MN-major, K = batch, split-K for one large-batch learner), db = column sums of dZ
static int tc_dw(Ddpg* h, cudaStream_t st, const float* X, int ldx, const float* dZ, int lddz, int B, const LayerDims& L, float* grad, bool side = false) {
  float* const ws = side ? h->ws_side : h->ws;
  unsigned* const counters = side ? h->counters_side : h->counters;
  const int tiles = ((L.in + 127) / 128) * ((L.out + 127) / 128), kb = (B + 31) / 32;
  const int splits = h->pop > 1 ? 1 : max(1, min(min(kb / 4, (148 + tiles - 1) / tiles), SPLITK_MAX));
  TcOperand A{X, ldx, true}, Bo{dZ, lddz, true};
  TcBatch bt; bt.count = h->pop; bt.sA = bt.sB = bt.sD = h->pop_stride;
  TRY(tc_gemm(st, A, Bo, grad + L.w_off, L.out, L.in, L.out, B, TC_EPI_NONE, nullptr, nullptr, 0, splits, splits > 1 ? ws : nullptr, bt));
  const int slabs = h->pop > 1 ? 1 : max(1, min(SPLITK_MAX, B / 128)), rows_per = (B + slabs - 1) / slabs;
  if (slabs == 1) {  // small batch: the column sums are the bias gradient (every learner of a population in one launch)
    wcolsum_partial_kernel<0><<<dim3((L.out + 31) / 32, 1, h->pop), 256, 0, st>>>(dZ, lddz, B, L.out, nullptr, rows_per, L.out, grad + L.b_off, h->pop_stride,
                                                                                 nullptr, nullptr);
    CUDA_TRY(cudaGetLastError());
    return SHEMS_OK;
  }
  REQUIRE((L.out + 31) / 32 <= WS_COUNTERS, SHEMS_ERR_INVALID, "tc_dw: layer too wide for the reduction counters");
  wcolsum_partial_kernel<0><<<dim3((L.out + 31) / 32, slabs), 256, 0, st>>>(dZ, lddz, B, L.out, nullptr, rows_per, L.out, ws, 0, grad + L.b_off,
                                                                            counters);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// one net of a forward pass: inputs X -> h1 -> h2 -> output layer (out: TC_OUT_TANH / TC_OUT_ID / TC_OUT_TD) into y [rows][ldy].
// keep: a backward pass reads h1 and h2 (the chain kernel stores them only then; the layer-by-layer products always go through them)
struct FwdNet { const float* X; const float* w; const NetDims* d; float *h1, *h2; bool keep; int out; float* y; int ldy; };
// large-batch first layer (up to 3 nets): see l1_fwd_kernel
static int big_l1(cudaStream_t st, const FwdNet* nets, int count, int ldx, int M, int ldy, int pop, long long ls_w, long long ls_x) {
  L1Batch a; memset(&a, 0, sizeof(a));
  a.count = count; a.ls_w = ls_w; a.ls_x = ls_x;
  for (int i = 0; i < count; ++i) {
    const LayerDims& L = nets[i].d->l[0];
    a.X[i] = nets[i].X; a.W[i] = nets[i].w + L.w_off; a.bias[i] = nets[i].w + L.b_off; a.Y[i] = nets[i].h1; a.K[i] = L.in;
    REQUIRE(L.in <= 12 && L.out == nets[0].d->l[0].out, SHEMS_ERR_INVALID, "big_l1: unsupported first-layer shape");
  }
  a.M = M; a.N = nets[0].d->l[0].out; a.ldx = ldx; a.ldy = ldy;
  l1_fwd_kernel<<<dim3((M + 31) / 32, (a.N + 255) / 256, count * pop), 256, 0, st>>>(a);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// output layer backward: dW3 (+db3) by weighted column sums, dX by the masked outer product (large batches and populations)
static int launch_outer_mask(Ddpg* h, cudaStream_t st, const float* dZ, int J, const float* W, const float* H, int ld, int B, int N, float* dX) {
  const long long ne = (long long)B * ((N + 3) / 4);
  REQUIRE(ne < (1ll << 31), SHEMS_ERR_INVALID, "launch_outer_mask: batch x width too large");
  const dim3 grid((unsigned)((ne + 255) / 256), h->pop);
  if (J == 1) outer_mask_kernel<1><<<grid, 256, 0, st>>>(dZ, W, H, ld, B, N, dX, h->pop_stride);
  else outer_mask_kernel<2><<<grid, 256, 0, st>>>(dZ, W, H, ld, B, N, dX, h->pop_stride);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// dW3 (+db3) of an output layer with J <= 2 units by weighted column sums over slabs of rows
static int out_bwd_dw(Ddpg* h, cudaStream_t st, const float* H, int ldh, const float* dZ, int J, int B, const LayerDims& L, float* grad, bool side = false) {
  REQUIRE(J == L.out && (J == 1 || J == 2), SHEMS_ERR_INVALID, "out_bwd_dw: output layer must have 1 or 2 units");
  float* const ws = side ? h->ws_side : h->ws;
  unsigned* const counters = side ? h->counters_side : h->counters;
  const int N = L.in, slabs = h->pop > 1 ? 1 : max(1, min(SPLITK_MAX, B / 128)), rows_per = (B + slabs - 1) / slabs;
  const long long stride = (long long)N * J + J;
  const dim3 grid((N + 31) / 32, slabs, h->pop);
  float* out = slabs == 1 ? grad + L.w_off : ws;  // a single slab is the gradient block [W3 | b3] itself
  REQUIRE((N + 31) / 32 <= WS_COUNTERS, SHEMS_ERR_INVALID, "out_bwd_dw: layer too wide for the reduction counters");
  if (J == 1) wcolsum_partial_kernel<1><<<grid, 256, 0, st>>>(H, ldh, B, N, dZ, rows_per, stride, out, h->pop_stride, grad + L.w_off, counters);
  else wcolsum_partial_kernel<2><<<grid, 256, 0, st>>>(H, ldh, B, N, dZ, rows_per, stride, out, h->pop_stride, grad + L.w_off, counters);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// fork / join of the side stream (inside a stream capture these become parallel branches of the graph)
static int side_after(Ddpg* h, cudaStream_t st, cudaEvent_t ev) {   // the side stream continues after what `st` has enqueued so far
  CUDA_TRY(cudaEventRecord(ev, st));
  CUDA_TRY(cudaStreamWaitEvent(h->side, ev, 0));
  return SHEMS_OK;
}
static int side_join(Ddpg* h, cudaStream_t st) {                     // `st` continues after everything enqueued on the side stream
  CUDA_TRY(cudaEventRecord(h->ev_join, h->side));
  CUDA_TRY(cudaStreamWaitEvent(st, h->ev_join, 0));
  return SHEMS_OK;
}
static inline bool use_tc(const Ddpg* h, long long rows) { return h->tc && rows * h->pop >= TC_MIN_ROWS; }
// how the passes of a call run, as the caller decides it: chain: a net's whole forward pass is one kernel (tc_fwd_chain); tc: the
// layer-2 products on TF32 tensor cores; big: streaming kernels for the thin products, the weight gradients of a backward pass on the
// side stream
struct Regime { bool chain, tc, big; };
static inline Regime update_regime(const Ddpg* h) {
  const int B = h->p.batch;
  const bool tc = use_tc(h, B);
  return Regime{tc && h->chain, tc, tc || B >= SPLITK_MIN_BATCH || h->pop > 1};
}

// The forward passes of up to 3 nets of one width on M rows of inputs [M][ldx], sharing launches: layer 1 -> layer 2 -> output layer,
// or with rg.chain one whole-net kernel (csrc/tc_gemm.cu tc_fwd_chain_kernel) launched with the flags pdl / early_weights.  The
// activations of learner l lie xstride floats behind learner 0's, its weights pop_stride.  defer_out: without the chain kernel the
// output layer is left to the caller.
static int enqueue_forward(const Ddpg* h, cudaStream_t st, const Regime& rg, const FwdNet* nets, int count, int ldx, int M, long long xstride,
                           int pdl = 0, int early_weights = 0, bool defer_out = false) {
  if (rg.chain) {
    TcFwdChainArgs a; memset(&a, 0, sizeof(a));
    a.M = M; a.L1 = h->p.l1; a.L2 = h->p.l2; a.nprob = count; a.ldx = ldx; a.ldh1 = h->ld1; a.ldh2 = h->ld2;
    a.pop = h->pop; a.pop_stride = h->pop_stride;
    // few row tiles: two CTAs (a cluster) per tile, half of the layer-2 units each, so that the launch covers the SMs
    a.nsplit = (long long)((M + 127) / 128) * count * h->pop * 2 <= 148 ? 2 : 1;
    for (int q = 0; q < count; ++q) {
      const FwdNet& n = nets[q]; const NetDims& d = *n.d;
      a.X[q] = n.X; a.K1[q] = d.l[0].in;
      a.W1[q] = n.w + d.l[0].w_off; a.b1[q] = n.w + d.l[0].b_off; a.W2[q] = n.w + d.l[1].w_off; a.b2[q] = n.w + d.l[1].b_off;
      a.W3[q] = n.w + d.l[2].w_off; a.b3[q] = n.w + d.l[2].b_off; a.J[q] = d.l[2].out;
      a.H1[q] = n.keep ? n.h1 : nullptr; a.H2[q] = n.keep ? n.h2 : nullptr; a.out_mode[q] = n.out; a.out[q] = n.y; a.ldo[q] = n.ldy;
      if (n.out == TC_OUT_TD) {
        a.td_r = h->r; a.td_done = h->done; a.td_q = h->q; a.td_dq = h->dq; a.inv_batch = 1.0f / (float)M;
        a.td_gamma = &h->ctrl->hp.gamma; a.td_gamma_stride = sizeof(DdpgCtrl) / sizeof(float);
      }
    }
    a.pdl = pdl; a.early_weights = early_weights;
    return tc_fwd_chain(st, a);
  }
  const int l1 = h->ld1, l2 = h->ld2;
  GemmProblem g[TC_MAX_PROBLEMS];
  if (rg.big) TRY(big_l1(st, nets, count, ldx, M, l1, h->pop, h->pop_stride, xstride));
  else {
    for (int q = 0; q < count; ++q) g[q] = gp_fwd(nets[q].X, ldx, M, nets[q].w, nets[q].d->l[0], nets[q].h1, l1, EPI_BIAS_RELU);
    TRY(launch_gemms(st, g, count, h->pop, h->pop_stride, xstride));
  }
  if (rg.tc) {  // the layer-2 products have one shape: a single persistent launch deals their tiles over the SMs
    TcOperand A[TC_MAX_PROBLEMS], W[TC_MAX_PROBLEMS]; float* D[TC_MAX_PROBLEMS]; const float* bias[TC_MAX_PROBLEMS];
    for (int q = 0; q < count; ++q) {   // Y = relu(X · W + b):  X [M][ld1] K-major, Flux weight Wt[in][out] MN-major
      const LayerDims& L = nets[q].d->l[1];
      A[q] = TcOperand{nets[q].h1, l1, false}; W[q] = TcOperand{nets[q].w + L.w_off, L.out, true};
      D[q] = nets[q].h2; bias[q] = nets[q].w + L.b_off;
    }
    TcBatch bt; bt.count = h->pop; bt.sA = bt.sD = xstride; bt.sB = bt.sBias = h->pop_stride;
    const LayerDims& L = nets[0].d->l[1];
    TRY(tc_gemm_multi(st, count, A, W, D, l2, M, L.out, L.in, TC_EPI_BIAS_RELU, bias, nullptr, 0, 1, nullptr, bt));
  } else {
    for (int q = 0; q < count; ++q) g[q] = gp_fwd(nets[q].h1, l1, M, nets[q].w, nets[q].d->l[1], nets[q].h2, l2, EPI_BIAS_RELU);
    TRY(launch_gemms(st, g, count, h->pop, h->pop_stride, xstride));
  }
  if (defer_out) return SHEMS_OK;
  for (int q = 0; q < count; ++q) {
    const FwdNet& n = nets[q];
    g[q] = gp_fwd(n.h2, l2, M, n.w, n.d->l[2], n.y, n.ldy, n.out == TC_OUT_TANH ? EPI_BIAS_TANH : n.out == TC_OUT_ID ? EPI_BIAS_ID : EPI_TD_TARGET);
    if (n.out == TC_OUT_TD) { g[q].aux = h->r; g[q].aux2 = h->done; g[q].aux3 = h->q; g[q].out2 = h->dq; g[q].ctrl = h->ctrl; g[q].inv_batch = 1.0f / (float)M; }
  }
  return launch_gemms(st, g, count, h->pop, h->pop_stride, xstride);
}

// The backward pass of one net from dout = d loss / d output [B][J] to its weight gradients in grad, through dz2 [B][ld2] and dz1 [B][ld1],
// on the activations h1, h2 of its forward pass and the minibatch xs (the actor's first layer reads its 9 state columns).  extra: a
// product that is no part of the pass (the actor's reporting-only q(s, actor(s))), enqueued off the critical path.
static int enqueue_backward(Ddpg* h, cudaStream_t st, const Regime& rg, const float* w, const NetDims& d, const float* h1, const float* h2,
                            const float* dout, float* dz2, float* dz1, float* grad, const GemmProblem* extra = nullptr) {
  const int B = h->p.batch, l1 = h->ld1, l2 = h->ld2, J = d.l[2].out;
  GemmProblem g[2];
  if (rg.big) {
    // the dX chain (dz2 -> dz1 -> dW1) is the critical path; dW3, dW2 and their bias sums run beside it on the side stream
    TRY(side_after(h, st, h->ev_fork));                                                                       // dout, h2 are ready
    TRY(out_bwd_dw(h, h->side, h2, l2, dout, J, B, d.l[2], grad, true));
    if (extra) TRY(slab_gemms(h, h->side, extra, 1));
    TRY(launch_outer_mask(h, st, dout, J, w + d.l[2].w_off, h2, l2, B, d.l[2].in, dz2));
    TRY(side_after(h, st, h->ev_mid));                                                                        // dz2 is ready
    if (rg.tc) {
      TRY(tc_dw(h, h->side, h1, l1, dz2, l2, B, d.l[1], grad, true));
      TRY(tc_dx(h, st, dz2, l2, B, w, d.l[1], dz1, l1, h1, l1));
    } else {
      g[0] = gp_dw(h1, l1, dz2, l2, B, d.l[1], grad);
      g[1] = gp_dx(dz2, l2, B, w, d.l[1], 0, d.l[1].in, dz1, l1, EPI_RELU_MASK, h1, l1);
      TRY(launch_dw(h, h->side, g[0], true));
      TRY(slab_gemms(h, st, g + 1, 1));
    }
    TRY(launch_dw(h, st, gp_dw(h->xs, 11, dz1, l1, B, d.l[0], grad)));
    return side_join(h, st);
  }
  g[0] = gp_dw(h2, l2, dout, J, B, d.l[2], grad);
  g[1] = gp_dx(dout, J, B, w, d.l[2], 0, d.l[2].in, dz2, l2, EPI_RELU_MASK, h2, l2);
  TRY(slab_gemms(h, st, g, 2));
  g[0] = gp_dw(h1, l1, dz2, l2, B, d.l[1], grad);
  g[1] = gp_dx(dz2, l2, B, w, d.l[1], 0, d.l[1].in, dz1, l1, EPI_RELU_MASK, h1, l1);
  TRY(slab_gemms(h, st, g, 2));
  TRY(launch_dw(h, st, gp_dw(h->xs, 11, dz1, l1, B, d.l[0], grad)));
  if (extra) TRY(slab_gemms(h, st, extra, 1));
  return SHEMS_OK;
}

// ADAM on the critic (opt 0) or on the actor (opt 1: with soft_update! of both targets and the advance of the update counters).
// dp: the gradient exchange over NVLink fused into the step; parts: the gradient is the sum of the cluster-fused passes' per-cluster
// partials, added in the same kernel.  One element per thread (the Float64 div/sqrt chains need TLP); the grids of both steps are sized
// from the critic's parameter count.
#ifndef ADAM_PARTS_THREADS
#define ADAM_PARTS_THREADS 256
#endif
static int enqueue_adam(Ddpg* h, cudaStream_t st, int opt, float gscale, bool dp, bool parts) {
  const DdpgParams& p = h->p;
  const int k = opt == 0 ? 1 : 0;   // index of the net in grad, adam_m, adam_v, parts and dims (0 actor, 1 critic)
  const long long n = h->dims[k].n_params, nc = h->dims[1].n_params;
  float* const x = h->net[opt == 0 ? DDPG_NET_CRITIC : DDPG_NET_ACTOR];
  float* const target = opt ? h->net[DDPG_NET_ACTOR_TARGET] : nullptr;
  float* const target2 = opt ? h->net[DDPG_NET_CRITIC_TARGET] : nullptr;   // the critic target moves with the actor step (DDPG.jl:142-143)
  const float* const model2 = opt ? h->net[DDPG_NET_CRITIC] : nullptr;
  const long long n2 = opt ? nc : 0;
  const int nparts = parts ? p.batch / FUSED_ROWS : 0;
  const float* const part = parts ? h->parts[k] : nullptr;
  if (dp)  // the flat gradient buffer holds the critic's segment, then the actor's
    return launch_adam_dp(st, h->dp, h->grad[k] - h->gradbuf, part, nparts, parts ? n : 0, h->grad[k], x, h->adam_m[k], h->adam_v[k], n,
                          p.adam_beta1, p.adam_beta2, p.adam_eps, h->ctrl, opt, target, target2, model2, n2, opt);
  const unsigned blocks = (unsigned)((nc + 255) / 256);
  if (parts)
    adam_polyak_parts_kernel<<<(unsigned)((nc + ADAM_PARTS_THREADS - 1) / ADAM_PARTS_THREADS), ADAM_PARTS_THREADS, 0, st>>>(
        x, part, nparts, n, h->grad[k], h->adam_m[k], h->adam_v[k], n, p.adam_beta1, p.adam_beta2, p.adam_eps, h->ctrl, opt, target, target2,
        model2, n2, opt);
  else if (h->tc)
    adam_polyak_kernel<true><<<dim3((blocks + 3) / 4, h->pop), 256, 0, st>>>(x, h->grad[k], h->adam_m[k], h->adam_v[k], n, p.adam_beta1, p.adam_beta2,
                                                                            p.adam_eps, h->ctrl, opt, target, target2, model2, n2, opt, gscale, h->pop_stride);
  else
    adam_polyak_kernel<false><<<dim3(blocks, h->pop), 256, 0, st>>>(x, h->grad[k], h->adam_m[k], h->adam_v[k], n, p.adam_beta1, p.adam_beta2,
                                                                   p.adam_eps, h->ctrl, opt, target, target2, model2, n2, opt, gscale, h->pop_stride);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

// one replay() after the minibatch has been gathered (DESIGN.md, "DDPG update"), in three phases so that a data-parallel
// learner can all-reduce the flat gradient buffer between them:
//   phase 0: targets, TD target, critic forward/backward            -> grad[critic]
//   phase 1: ADAM(critic), actor-loss forward/backward through the UPDATED critic -> grad[actor]
//   phase 2: ADAM(actor), soft_update! of both targets, counters
// Small batches (the reference's B = 120) are latency bound: independent problems share launches (up to 4 per kernel).
// Large batches run one problem per launch; the 250x500 contractions go to the TF32 tensor-core kernel when enabled and
// every product whose K is the batch is split over the batch.
static int enqueue_phase0(Ddpg* h, cudaStream_t st) {
  const Regime rg = update_regime(h);
  const int B = h->p.batch;
  const NetDims& da = h->dims[0]; const NetDims& dc = h->dims[1];
  float *actor = h->net[DDPG_NET_ACTOR], *critic = h->net[DDPG_NET_CRITIC], *actor_t = h->net[DDPG_NET_ACTOR_TARGET], *critic_t = h->net[DDPG_NET_CRITIC_TARGET];
  // P1-P3: actor_target(s'_n) -> a' | critic(s_n, a) -> q | actor(s_n) -> vcat(s_n, actions)      (DDPG.jl:131, :114, :117)
  // Programmatic dependent launches (the tcgen05 kernels only: their set-up is worth hiding, and a CTA of theirs fills an SM, so
  // a grid scheduled early takes nothing from the side branch.  The thin kernels as dependents were measured and dropped: their
  // early-resident blocks starve the side branch, 209 -> 226 us).  After the gather only the rows' inputs are its output.
  const FwdNet fwd[3] = {{h->xs2, actor_t, &da, h->t_h1, h->t_h2, false, TC_OUT_TANH, h->xs2 + 9, 11},
                         {h->xs, critic, &dc, h->c_h1, h->c_h2, true, TC_OUT_ID, h->q, 1},
                         {h->xs, actor, &da, h->a_h1, h->a_h2, true, TC_OUT_TANH, h->xspi + 9, 11}};
  TRY(enqueue_forward(h, st, rg, fwd, 3, 11, B, h->pop_stride, 1, 1));
  // P4-P6: q' = critic_target(vcat(s'_n, a'));  y = r + γ(1-done) q';  dq = 2(q-y)/B     (:132-133)
  // (after the three-net launch: a' and q are its output, critic_target's weights are not)
  const FwdNet td = {h->xs2, critic_t, &dc, h->tc_h1, h->tc_h2, false, TC_OUT_TD, h->y, 1};
  TRY(enqueue_forward(h, st, rg, &td, 1, 11, B, h->pop_stride, 1, 1));
  if (h->per) {   // prioritized replay: importance weights on dq, the rows' priorities back into the sum trees
    ddpg_per_kernel<<<dim3(1, h->pop), PER_THREADS, 0, st>>>(h->trees_dev, h->ctrl, h->per_knobs, h->per_slot, h->per_leaf, h->q, h->y, h->dq, B,
                                                             h->pop_stride);
    CUDA_TRY(cudaGetLastError());
  }
  // P7-P9: critic backward (:137, :105-108)
  return enqueue_backward(h, st, rg, critic, dc, h->c_h1, h->c_h2, h->dq, h->dz2, h->dz1, h->grad[1]);
}

static int enqueue_phase1(Ddpg* h, cudaStream_t st, float gscale, bool dp = false) {
  const Regime rg = update_regime(h);
  const DdpgParams& p = h->p;
  const int B = p.batch, l1 = h->ld1, l2 = h->ld2;
  const NetDims& da = h->dims[0]; const NetDims& dc = h->dims[1];
  float *actor = h->net[DDPG_NET_ACTOR], *critic = h->net[DDPG_NET_CRITIC];
  // the fused dX chain through the critic below: with few row tiles two CTAs share a tile and ADD their shares of the action-input gradient
  const int bwd_split = (rg.chain && h->pop == 1 && ((B + 127) / 128) * 2 <= 148) ? 2 : 1;
  if (bwd_split == 2) CUDA_TRY(cudaMemsetAsync(h->dza3, 0, sizeof(float) * 2 * (size_t)B, st));
  // P10: ADAM(η_crit) on the critic
  TRY(enqueue_adam(h, st, 0, gscale, dp, false));
  // P11-P13: critic(vcat(s_n, actor(s_n))) with the UPDATED critic (:116-119); loss_act = -mean(q) => dq = -1/B.  The chain kernel
  // also yields q(s, actor(s)) itself (reporting); layer by layer, that product is left for the actor's backward pass below
  // (chain: after ADAM(critic), the weights are the predecessor's output)
  const FwdNet fwd = {h->xspi, critic, &dc, h->p_h1, h->p_h2, true, TC_OUT_ID, h->qpi, 1};
  TRY(enqueue_forward(h, st, rg, &fwd, 1, 11, B, h->pop_stride, 1, 0, true));
  GemmProblem g;
  if (rg.chain) {
    // dX through the critic only, as ONE kernel (csrc/tc_gemm.cu tc_bwd_chain_kernel): dq -> dz2 -> dz1 -> the action inputs, times tanh';
    // nothing of it is kept (no weight gradient of the critic in the actor's loss)
    TcBwdChainArgs b; memset(&b, 0, sizeof(b));
    b.M = B; b.L1 = p.l1; b.L2 = p.l2; b.J = 1; b.ldh1 = l1; b.ldh2 = l2; b.pdl = 1; b.nsplit = bwd_split;
    b.dout = h->dqpi; b.W3 = critic + dc.l[2].w_off; b.W2 = critic + dc.l[1].w_off; b.H2 = h->p_h2; b.H1 = h->p_h1;
    b.W1a = critic + dc.l[0].w_off + 9ll * p.l1; b.act = h->xspi + 9; b.ld_act = 11; b.dA = h->dza3;
    b.pop = h->pop; b.pop_stride = h->pop_stride;
    TRY(tc_bwd_chain(st, b));
  } else {
    if (rg.big) {                                                                                            // dX through the critic only
      TRY(launch_outer_mask(h, st, h->dqpi, 1, critic + dc.l[2].w_off, h->p_h2, l2, B, p.l2, h->dzp2));
    } else {
      g = gp_dx(h->dqpi, 1, B, critic, dc.l[2], 0, p.l2, h->dzp2, l2, EPI_RELU_MASK, h->p_h2, l2);
      TRY(slab_gemms(h, st, &g, 1));
    }
    // P14-P15: back through critic layers 2, 1 down to the action inputs, times tanh'
    if (rg.tc) TRY(tc_dx(h, st, h->dzp2, l2, B, critic, dc.l[1], h->dzp1, l1, h->p_h1, l1));
    else {
      g = gp_dx(h->dzp2, l2, B, critic, dc.l[1], 0, p.l1, h->dzp1, l1, EPI_RELU_MASK, h->p_h1, l1);
      TRY(slab_gemms(h, st, &g, 1));
    }
    g = gp_dx(h->dzp1, l1, B, critic, dc.l[0], 9, 2, h->dza3, 2, EPI_TANH_GRAD, h->xspi + 9, 11);
    TRY(slab_gemms(h, st, &g, 1));
  }
  // P16-P18: actor backward, with q(s, actor(s)) beside it when the chain kernel has not produced it
  const GemmProblem qpi = gp_fwd(h->p_h2, l2, B, critic, dc.l[2], h->qpi, 1, EPI_BIAS_ID);
  return enqueue_backward(h, st, rg, actor, da, h->a_h1, h->a_h2, h->dza3, h->dza2, h->dza1, h->grad[0], rg.chain ? nullptr : &qpi);
}

static int enqueue_phase2(Ddpg* h, cudaStream_t st, float gscale, bool dp = false) {
  // P19: ADAM(η_act) on the actor + soft_update! of both targets (:140-143)
  return enqueue_adam(h, st, 1, gscale, dp, false);
}

// One learner at a small batch: critic pass -> ADAM(critic) -> actor pass -> ADAM(actor) + soft_update!, the two passes as
// thread-block-cluster kernels that keep a row's whole forward/backward chain on chip (csrc/ddpg_fused.cu)
static inline bool use_fused(const Ddpg* h) { return h->fused && h->parts[0] && h->parts[1]; }
static inline FusedNetOff fused_off(const NetDims& d) {
  return FusedNetOff{(int)d.l[0].w_off, (int)d.l[0].b_off, (int)d.l[1].w_off, (int)d.l[1].b_off, (int)d.l[2].w_off, (int)d.l[2].b_off};
}
struct GatherSrc { bool from_rings; const float *s, *a, *r, *s2, *done; long long ld; };
static int enqueue_update_fused(Ddpg* h, cudaStream_t st, bool dp, const GatherSrc& src) {
  const DdpgParams& p = h->p;
  FusedArgs a; memset(&a, 0, sizeof(a));
  a.actor = h->net[DDPG_NET_ACTOR]; a.critic = h->net[DDPG_NET_CRITIC]; a.actor_t = h->net[DDPG_NET_ACTOR_TARGET]; a.critic_t = h->net[DDPG_NET_CRITIC_TARGET];
  a.ao = fused_off(h->dims[0]); a.co = fused_off(h->dims[1]);
  a.l1 = p.l1; a.l2 = p.l2; a.B = p.batch;
  a.xs = h->xs; a.xs2 = h->xs2; a.xspi = h->xspi; a.r = h->r; a.done = h->done; a.q = h->q; a.y = h->y; a.qpi = h->qpi;
  a.inv_batch = 1.0f / (float)p.batch;
  a.rings = src.from_rings ? h->rings_dev : nullptr;
  a.src_s = src.s; a.src_a = src.a; a.src_r = src.r; a.src_s2 = src.s2; a.src_d = src.done; a.src_ld = src.ld;
  a.ctrl = h->ctrl; a.idx = h->idx_dev; a.norm = h->norm; a.xs_w = h->xs;
  a.vec16 = w2_vec16(h) ? 1 : 0;
  if (src.from_rings && h->nstep > 1) { a.links = h->links_dev; a.nstep = h->nstep_knob; }
  // each pass is followed by the reduction of its partial sums and the optimiser step (dp: with the gradient exchange) in ONE kernel
  a.part = h->parts[1]; a.part_stride = h->dims[1].n_params;
  TRY(ddpg_fused_critic(st, a));
  TRY(enqueue_adam(h, st, 0, 1.0f, dp, true));
  a.part = h->parts[0]; a.part_stride = h->dims[0].n_params;
  TRY(ddpg_fused_actor(st, a));
  return enqueue_adam(h, st, 1, 1.0f, dp, true);
}

static int enqueue_update_body(Ddpg* h, cudaStream_t st, bool dp = false) {
  int s0 = enqueue_phase0(h, st);
  if (!s0) s0 = enqueue_phase1(h, st, 1.0f, dp);
  if (!s0) s0 = enqueue_phase2(h, st, 1.0f, dp);
  return s0;
}

// from_rings: every learner samples its own replay ring (h->rings_dev); else one caller-supplied minibatch (single learner)
static int enqueue_gather(Ddpg* h, cudaStream_t st, bool from_rings, const float* s, const float* a, const float* r, const float* s2,
                          const float* done, long long ld) {
  const int B = h->p.batch;
  if (from_rings && h->nstep > 1) {
    if (h->per)
      ddpg_gather_per_nstep_kernel<<<dim3((B * 9 + 127) / 128, h->pop), 128, 0, st>>>(h->rings_dev, h->ctrl, h->idx_dev, h->idx_stride, h->norm, B,
                                                                                     h->xs, h->xs2, h->xspi, h->r, h->done, h->pop_stride, h->trees_dev,
                                                                                     h->per_slot, h->per_leaf, h->links_dev, h->nstep_knob);
    else
      ddpg_gather_nstep_kernel<<<dim3((B * 9 + 127) / 128, h->pop), 128, 0, st>>>(h->rings_dev, h->ctrl, h->idx_dev, h->idx_stride, h->norm, B, h->xs,
                                                                                 h->xs2, h->xspi, h->r, h->done, h->pop_stride, h->links_dev,
                                                                                 h->nstep_knob);
    CUDA_TRY(cudaGetLastError());
    return SHEMS_OK;
  }
  if (h->per && from_rings) {
    ddpg_gather_per_kernel<<<dim3((B * 9 + 127) / 128, h->pop), 128, 0, st>>>(h->rings_dev, h->ctrl, h->idx_dev, h->idx_stride, h->norm, B, h->xs,
                                                                             h->xs2, h->xspi, h->r, h->done, h->pop_stride, h->trees_dev,
                                                                             h->per_slot, h->per_leaf);
    CUDA_TRY(cudaGetLastError());
    return SHEMS_OK;
  }
  ddpg_gather_kernel<<<dim3((B * 9 + 127) / 128, from_rings ? h->pop : 1), 128, 0, st>>>(from_rings ? h->rings_dev : nullptr, s, a, r, s2, done, ld,
                                                                                     h->ctrl, h->idx_dev, h->idx_stride, h->norm, B, h->xs,
                                                                                     h->xs2, h->xspi, h->r, h->done, h->pop_stride);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

// one whole replay(): sample + update.  Fused path: 4 launches (the critic pass gathers); tiled path: gather kernel + the GEMM sequence
static int enqueue_update(Ddpg* h, cudaStream_t st, bool dp, bool from_rings, const float* s, const float* a, const float* r, const float* s2,
                          const float* done, long long ld) {
  // prioritized replay weighs dq between the passes of the tiled sequence: its updates never take the fused passes
  if (use_fused(h) && !h->per) return enqueue_update_fused(h, st, dp, GatherSrc{from_rings, s, a, r, s2, done, ld});
  TRY(enqueue_gather(h, st, from_rings, s, a, r, s2, done, ld));
  return enqueue_update_body(h, st, dp);
}

// capture gather(from the replay rings) + body once; replays read everything that changes from the device control blocks
static int ensure_graph(Ddpg* h, bool dp = false) {
  cudaGraph_t& graph = dp ? h->graph_dp : h->graph;
  cudaGraphExec_t& graph_exec = dp ? h->graph_dp_exec : h->graph_exec;
  if (graph_exec) return SHEMS_OK;
  if (graph) { cudaGraphDestroy(graph); graph = nullptr; }
  cudaStream_t cs;
  CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { cudaStreamDestroy(cs); shems_set_error("cudaStreamBeginCapture: %s", cudaGetErrorString(e)); return SHEMS_ERR_CUDA; }
  int st = enqueue_update(h, cs, dp, true, nullptr, nullptr, nullptr, nullptr, nullptr, 0);
  e = cudaStreamEndCapture(cs, &graph);
  cudaStreamDestroy(cs);
  if (st) return st;
  if (e != cudaSuccess) { shems_set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e)); return SHEMS_ERR_CUDA; }
  CUDA_TRY(cudaGraphInstantiate(&graph_exec, graph, 0));
  return SHEMS_OK;
}

// a prioritized learner writes priorities back into its memory's tree: every learner needs a memory with priorities of its own
static int per_memories_ok(const Ddpg* h, ShemsReplay* const* rps, const char* who) {
  if (!h->per) return SHEMS_OK;
  for (int l = 0; l < h->pop; ++l) {
    REQUIRE(rps[l], SHEMS_ERR_INVALID, "%s: learner %d has no replay memory", who, l);
    REQUIRE(rps[l]->prio, SHEMS_ERR_STATE, "%s: prioritized learner, but the memory of learner %d has no priorities (replay_enable_priorities)", who, l);
    for (int k = 0; k < l; ++k)
      REQUIRE(rps[k] != rps[l], SHEMS_ERR_INVALID, "%s: prioritized learners %d and %d share one memory", who, k, l);
  }
  return SHEMS_OK;
}

// an n-step learner walks its memory's successor links: every learner needs a memory with links
static int nstep_memories_ok(const Ddpg* h, ShemsReplay* const* rps, const char* who) {
  if (h->nstep == 1) return SHEMS_OK;
  for (int l = 0; l < h->pop; ++l) {
    REQUIRE(rps[l], SHEMS_ERR_INVALID, "%s: learner %d has no replay memory", who, l);
    REQUIRE(rps[l]->next, SHEMS_ERR_STATE, "%s: n-step learner (n = %d), but the memory of learner %d has no successor links (replay_enable_successors)",
            who, h->nstep, l);
  }
  return SHEMS_OK;
}

struct CtrlHostPart { unsigned long long seed; unsigned update; int use_idx; long long len, head, cap; int idx_cursor; unsigned blocks_done; };
static_assert(sizeof(CtrlHostPart) == offsetof(DdpgCtrl, bp), "control block layout");

// host-owned part of every learner's control block (seed, ring geometry, index mode) + ring pointers + optional indices;
// update/bp stay device-owned.  rps[l], seeds[l]: learner l's replay memory and Philox seed; idx_host [pop][per_learner] or NULL.
static int stage_update_inputs(Ddpg* h, ShemsReplay* const* rps, const uint64_t* seeds, const int32_t* idx_host, long long per_learner) {
  const int pop = h->pop;
  std::vector<CtrlHostPart> hp((size_t)pop);
  std::vector<const float*> rings((size_t)pop);
  std::vector<float*> trees((size_t)pop);
  std::vector<const int32_t*> links((size_t)pop);
  TRY(per_memories_ok(h, rps, "ddpg_update"));
  TRY(nstep_memories_ok(h, rps, "ddpg_update"));
  for (int l = 0; l < pop; ++l) {
    ShemsReplay* rp = rps[l];
    REQUIRE(rp, SHEMS_ERR_INVALID, "ddpg_update: learner %d has no replay memory", l);
    REQUIRE(rp->device == h->device, SHEMS_ERR_INVALID, "ddpg_update: replay on device %d, learner on %d", rp->device, h->device);
    REQUIRE(rp->length > 0, SHEMS_ERR_STATE, "ddpg_update: memory is empty");
    trees[l] = rp->prio;
    links[l] = rp->next;
    if (idx_host)
      for (long long j = 0; j < per_learner; ++j) {
        const int32_t v = idx_host[(long long)l * per_learner + j];
        REQUIRE(v >= 0 && v < rp->length, SHEMS_ERR_INVALID, "ddpg_update: idx[%d][%lld]=%d outside 0..%lld", l, j, v, (long long)rp->length - 1);
      }
    // minibatch stream: Philox(seed, draw j, counter = index of the update inside THIS call) — replay(rng_rpl = r) trains on the
    // minibatch replay_sample(seed = r) returns, as getData(rng) is one sample in both uses (memory_plotting_saving.jl:31-42)
    hp[l].seed = seeds[l]; hp[l].update = 0u; hp[l].use_idx = idx_host ? 1 : 0;
    hp[l].len = rp->length; hp[l].head = rp->head; hp[l].cap = rp->capacity; hp[l].idx_cursor = 0; hp[l].blocks_done = 0;
    rings[l] = rp->ring;
  }
  if (idx_host) {
    const long long need = (long long)pop * per_learner;
    if (h->idx_cap < need) {
      CUDA_TRY(cudaStreamSynchronize(h->stream));
      cudaFree(h->idx_dev); h->idx_dev = nullptr; h->idx_cap = 0;
      CUDA_TRY(cudaMalloc(&h->idx_dev, sizeof(int32_t) * (size_t)need));
      h->idx_cap = need;
      if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }  // idx pointer is baked into the graphs
      if (h->graph_dp_exec) { cudaGraphExecDestroy(h->graph_dp_exec); h->graph_dp_exec = nullptr; }
    }
    if (h->idx_stride != per_learner && h->pop > 1) {  // the stride between learners' index blocks is baked in as well
      if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
      if (h->graph_dp_exec) { cudaGraphExecDestroy(h->graph_dp_exec); h->graph_dp_exec = nullptr; }
    }
    h->idx_stride = per_learner;
    CUDA_TRY(cudaMemcpyAsync(h->idx_dev, idx_host, sizeof(int32_t) * (size_t)need, cudaMemcpyHostToDevice, h->stream));
  }
  // pageable sources: the runtime stages these small copies before returning, so the vectors may go out of scope
  CUDA_TRY(cudaMemcpy2DAsync(h->ctrl, sizeof(DdpgCtrl), hp.data(), sizeof(CtrlHostPart), sizeof(CtrlHostPart), (size_t)pop, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaMemcpyAsync((void*)h->rings_dev, rings.data(), sizeof(const float*) * (size_t)pop, cudaMemcpyHostToDevice, h->stream));
  if (h->per) CUDA_TRY(cudaMemcpyAsync(h->trees_dev, trees.data(), sizeof(float*) * (size_t)pop, cudaMemcpyHostToDevice, h->stream));
  if (h->nstep > 1) CUDA_TRY(cudaMemcpyAsync((void*)h->links_dev, links.data(), sizeof(const int32_t*) * (size_t)pop, cudaMemcpyHostToDevice, h->stream));
  return SHEMS_OK;
}

extern "C" int32_t ddpg_update_population(Ddpg* h, ShemsReplay* const* rps, int32_t n_updates, const int32_t* idx_host, const uint64_t* seeds) {
  REQUIRE(h && rps && seeds, SHEMS_ERR_INVALID, "ddpg_update_population: NULL argument");
  REQUIRE(n_updates >= 1, SHEMS_ERR_INVALID, "ddpg_update_population: n_updates=%d", n_updates);
  GUARD(h->device);
  TRY(stage_update_inputs(h, rps, seeds, idx_host, (long long)n_updates * h->p.batch));
  TRY(ensure_graph(h));
  for (int u = 0; u < n_updates; ++u) CUDA_TRY(cudaGraphLaunch(h->graph_exec, h->stream));
  h->n_updates += n_updates;
  return SHEMS_OK;
}

extern "C" int32_t ddpg_update(Ddpg* h, ShemsReplay* rp, int32_t n_updates, const int32_t* idx_host, uint64_t seed) {
  REQUIRE(h && rp, SHEMS_ERR_INVALID, "ddpg_update: NULL argument");
  REQUIRE(h->pop == 1, SHEMS_ERR_INVALID, "ddpg_update: this handle holds %d learners, use ddpg_update_population", h->pop);
  return ddpg_update_population(h, &rp, n_updates, idx_host, &seed);
}

// Data-parallel learner: one replay() in three calls; between them the caller all-reduces (sum) the gradient buffer
// (ddpg_grad_buffer: critic part after phase 0, actor part after phase 1) and passes grad_scale = 1/world_size.
extern "C" int32_t ddpg_update_phase(Ddpg* h, ShemsReplay* rp, int32_t phase, const int32_t* idx_host, uint64_t seed, float grad_scale) {
  REQUIRE(h, SHEMS_ERR_INVALID, "ddpg_update_phase: NULL handle");
  REQUIRE(phase >= 0 && phase <= 2, SHEMS_ERR_INVALID, "ddpg_update_phase: phase=%d", phase);
  REQUIRE(h->pop == 1, SHEMS_ERR_INVALID, "ddpg_update_phase: not available for a population handle");
  REQUIRE(!h->per, SHEMS_ERR_STATE, "ddpg_update_phase: not available for a prioritized learner");
  REQUIRE(h->nstep == 1, SHEMS_ERR_STATE, "ddpg_update_phase: not available for an n-step learner");
  GUARD(h->device);
  if (phase == 0) {
    REQUIRE(rp, SHEMS_ERR_STATE, "ddpg_update_phase: replay missing");
    TRY(stage_update_inputs(h, &rp, &seed, idx_host, h->p.batch));
    TRY(enqueue_gather(h, h->stream, true, nullptr, nullptr, nullptr, nullptr, nullptr, 0));
    return enqueue_phase0(h, h->stream);
  }
  if (phase == 1) return enqueue_phase1(h, h->stream, grad_scale);
  TRY(enqueue_phase2(h, h->stream, grad_scale));
  h->n_updates += 1;
  return SHEMS_OK;
}

// ---- data-parallel learner over NVLink peer memory
struct DpExport {  // what one rank tells the others (ddpg_dp_export), DDPG_DP_HANDLE_BYTES bytes
  cudaIpcMemHandle_t box;          // the rank's exchange box (flags + inbox rows), written by its peers
  unsigned long long raw_box;      // the same address for peers living in THIS process (tests: two handles, one process)
  long long in_stride;             // floats per inbox row (the flat gradient buffer's length): must agree between the ranks
  int pid, device;
};
static_assert(sizeof(DpExport) <= DDPG_DP_HANDLE_BYTES, "DDPG_DP_HANDLE_BYTES too small");
static inline long long dp_in_stride(const Ddpg* h) { return (((h->grad[0] - h->gradbuf) + h->dims[0].n_params) + 63) & ~63ll; }

extern "C" int32_t ddpg_dp_export(Ddpg* h, void* handle_out) {
  REQUIRE(h && handle_out, SHEMS_ERR_INVALID, "ddpg_dp_export: NULL argument");
  REQUIRE(h->pop == 1, SHEMS_ERR_INVALID, "ddpg_dp_export: not available for a population handle");
  GUARD(h->device);
  if (!h->dp_box) {  // flags, then one inbox row per possible source rank; zeroed: exchange numbers start at 1
    const size_t bytes = sizeof(unsigned) * (size_t)DP_BOX_FLAG_WORDS + sizeof(float) * (size_t)DP_MAX_WORLD * (size_t)dp_in_stride(h);
    CUDA_TRY(cudaMalloc((void**)&h->dp_box, bytes));
    CUDA_TRY(cudaMemset(h->dp_box, 0, bytes));
    CUDA_TRY(cudaDeviceSynchronize());
  }
  DpExport e; memset(&e, 0, sizeof(e));
  CUDA_TRY(cudaIpcGetMemHandle(&e.box, h->dp_box));
  e.raw_box = (unsigned long long)(uintptr_t)h->dp_box;
  e.in_stride = dp_in_stride(h);
  e.pid = (int)getpid(); e.device = h->device;
  memset(handle_out, 0, DDPG_DP_HANDLE_BYTES);
  memcpy(handle_out, &e, sizeof(e));
  return SHEMS_OK;
}

extern "C" int32_t ddpg_dp_connect(Ddpg* h, int32_t rank, int32_t world, const void* handles) {
  REQUIRE(h && handles, SHEMS_ERR_INVALID, "ddpg_dp_connect: NULL argument");
  REQUIRE(world >= 1 && world <= DP_MAX_WORLD && rank >= 0 && rank < world, SHEMS_ERR_INVALID, "ddpg_dp_connect: rank=%d world=%d (max %d)", rank, world, DP_MAX_WORLD);
  REQUIRE(h->pop == 1 && !h->dp_on, SHEMS_ERR_STATE, "ddpg_dp_connect: population handle, or already connected");
  REQUIRE(!h->per, SHEMS_ERR_STATE, "ddpg_dp_connect: not available for a prioritized learner");
  REQUIRE(h->nstep == 1, SHEMS_ERR_STATE, "ddpg_dp_connect: not available for an n-step learner");
  REQUIRE(h->dp_box, SHEMS_ERR_STATE, "ddpg_dp_connect: call ddpg_dp_export on this handle first");
  GUARD(h->device);
  memset(&h->dp, 0, sizeof(h->dp));
  h->dp.world = world; h->dp.rank = rank; h->dp.in_stride = dp_in_stride(h);
  h->dp.timeout_ns = DP_TIMEOUT_NS;
  if (const char* ev = getenv("SHEMS_DP_TIMEOUT_MS")) {   // tests: a short clock for the missing-peer case
    const long long ms = atoll(ev);
    if (ms > 0) h->dp.timeout_ns = (unsigned long long)ms * 1000000ull;
  }
  for (int r = 0; r < world; ++r) {
    DpExport e;
    memcpy(&e, (const char*)handles + (size_t)r * DDPG_DP_HANDLE_BYTES, sizeof(e));
    REQUIRE(e.in_stride == h->dp.in_stride, SHEMS_ERR_INVALID, "ddpg_dp_connect: rank %d has a different network shape (%lld gradient floats, here %lld)", r,
            e.in_stride, h->dp.in_stride);
    if (r == rank) { h->dp.box[r] = h->dp_box; continue; }
    if (e.pid == (int)getpid()) {  // same process: plain pointers (peer access between the two devices if they differ)
      if (e.device != h->device) {
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, h->device, e.device));
        REQUIRE(can, SHEMS_ERR_CUDA, "ddpg_dp_connect: device %d cannot access device %d", h->device, e.device);
        cudaError_t pe = cudaDeviceEnablePeerAccess(e.device, 0);
        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(pe);
        cudaGetLastError();
      }
      h->dp.box[r] = (unsigned*)(uintptr_t)e.raw_box;
      continue;
    }
    void* pb = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&pb, e.box, cudaIpcMemLazyEnablePeerAccess));
    h->dp_opened[h->dp_n_opened++] = pb;
    h->dp.box[r] = (unsigned*)pb;
  }
  h->dp_on = true;
  return SHEMS_OK;
}

// Everything ddpg_update_dp may have to allocate or instantiate (index staging for idx_ints host-supplied indices per call, the
// captured graph), done up front: cudaMalloc / graph instantiation can synchronise the device, which must not happen while a
// peer that shares this GPU (two ranks in one process) already spins in its exchange kernel.
extern "C" int32_t ddpg_dp_prepare(Ddpg* h, int64_t idx_ints) {
  REQUIRE(h && h->dp_on, SHEMS_ERR_STATE, "ddpg_dp_prepare: call ddpg_dp_connect first");
  GUARD(h->device);
  if (idx_ints > h->idx_cap) {
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->idx_dev); h->idx_dev = nullptr; h->idx_cap = 0;
    CUDA_TRY(cudaMalloc(&h->idx_dev, sizeof(int32_t) * (size_t)idx_ints));
    h->idx_cap = idx_ints;
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
    if (h->graph_dp_exec) { cudaGraphExecDestroy(h->graph_dp_exec); h->graph_dp_exec = nullptr; }
  }
  TRY(ensure_graph(h, true));
  CUDA_TRY(cudaGraphUpload(h->graph_dp_exec, h->stream));  // the first launch would otherwise upload (and may synchronise)
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return SHEMS_OK;
}

// replay() n_updates times on a connected data-parallel learner: every rank samples its own replay shard, the two gradient
// exchanges run inside the optimiser kernels over NVLink (adam_polyak_dp_kernel); every rank must make the same calls.
extern "C" int32_t ddpg_update_dp(Ddpg* h, ShemsReplay* rp, int32_t n_updates, const int32_t* idx_host, uint64_t seed) {
  REQUIRE(h && rp, SHEMS_ERR_INVALID, "ddpg_update_dp: NULL argument");
  REQUIRE(h->dp_on, SHEMS_ERR_STATE, "ddpg_update_dp: call ddpg_dp_connect first");
  REQUIRE(!h->per, SHEMS_ERR_STATE, "ddpg_update_dp: not available for a prioritized learner");
  REQUIRE(h->nstep == 1, SHEMS_ERR_STATE, "ddpg_update_dp: not available for an n-step learner");
  REQUIRE(n_updates >= 1, SHEMS_ERR_INVALID, "ddpg_update_dp: n_updates=%d", n_updates);
  GUARD(h->device);
  TRY(stage_update_inputs(h, &rp, &seed, idx_host, (long long)n_updates * h->p.batch));
  TRY(ensure_graph(h, true));
  for (int u = 0; u < n_updates; ++u) CUDA_TRY(cudaGraphLaunch(h->graph_dp_exec, h->stream));
  h->n_updates += n_updates;
  return SHEMS_OK;
}
// 0 while every gradient exchange completed; 1 after a peer failed to arrive within the spin limit (the update was skipped)
extern "C" int32_t ddpg_dp_status(Ddpg* h, int32_t* error_out) {
  REQUIRE(h && error_out, SHEMS_ERR_INVALID, "ddpg_dp_status: NULL argument");
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  int e = 0;
  CUDA_TRY(cudaMemcpy(&e, &h->ctrl->dp_error, sizeof(int), cudaMemcpyDeviceToHost));
  *error_out = e;
  return SHEMS_OK;
}

extern "C" int32_t ddpg_update_batch(Ddpg* h, const float* s_dev, const float* a_dev, const float* r_dev, const float* s2_dev, const float* done_dev) {
  REQUIRE(h && s_dev && a_dev && r_dev && s2_dev, SHEMS_ERR_INVALID, "ddpg_update_batch: NULL argument");
  REQUIRE(h->pop == 1, SHEMS_ERR_INVALID, "ddpg_update_batch: not available for a population handle");
  REQUIRE(!h->per, SHEMS_ERR_STATE, "ddpg_update_batch: a prioritized learner samples its replay memory (no priorities come with a caller's minibatch)");
  GUARD(h->device);
  TRY(enqueue_update(h, h->stream, false, false, s_dev, a_dev, r_dev, s2_dev, done_dev, h->p.batch));
  h->n_updates += 1;
  return SHEMS_OK;
}

// loss_crit = mean((q - y)^2) and loss_act = -mean(q_pi) of the last update (DDPG.jl:114-119)
__global__ void ddpg_loss_kernel(const float* __restrict__ q, const float* __restrict__ y, const float* __restrict__ qpi, int B, float* __restrict__ out) {
  double lc = 0.0, la = 0.0;
  for (int j = threadIdx.x; j < B; j += 32) { const float d = q[j] - y[j]; lc += (double)(d * d); la += (double)qpi[j]; }
  for (int o = 16; o > 0; o >>= 1) { lc += __shfl_xor_sync(0xffffffffu, lc, o); la += __shfl_xor_sync(0xffffffffu, la, o); }
  if (threadIdx.x == 0) { out[0] = (float)(lc / B); out[1] = (float)(-la / B); }
}
extern "C" int32_t ddpg_get_losses(Ddpg* h, float* loss_crit, float* loss_act) {
  REQUIRE(h && loss_crit && loss_act, SHEMS_ERR_INVALID, "ddpg_get_losses: NULL argument");
  GUARD(h->device);
  ddpg_loss_kernel<<<1, 32, 0, h->stream>>>(h->q + sel_off(h), h->y + sel_off(h), h->qpi + sel_off(h), h->p.batch, h->loss_scratch);
  CUDA_TRY(cudaGetLastError());
  float out[2];
  CUDA_TRY(cudaMemcpyAsync(out, h->loss_scratch, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  *loss_crit = out[0]; *loss_act = out[1];
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- act
// normalize (memory_plotting_saving.jl:55-57) of SoA obs [9][n] -> x [n][9]
__global__ void __launch_bounds__(256)
ddpg_normalize_kernel(const float* __restrict__ obs, long long n, const float* __restrict__ norm, float* __restrict__ x, long long pop_stride,
                      long long act_stride, long long osl, long long osk) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  // learner l = blockIdx.y; state field k of its instance j sits at obs[l*osl + k*osk + j]
  // (packed [P][9][n]: osl = 9n, osk = n; one SoA over all N = P*n instances, as an env handle stores it: osl = n, osk = N)
  obs += (long long)blockIdx.y * osl; norm += (long long)blockIdx.y * pop_stride; x += (long long)blockIdx.y * act_stride;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const float den = __fadd_rn(__fsub_rn(norm[9 + k], norm[k]), 1e-8f);
    x[j * 9 + k] = __fdiv_rn(__fsub_rn(obs[k * osk + j], norm[k]), den);
  }
}
// clamp(actor + noise, -1, 1) and scale_action (DDPG.jl:172-184); noise: given, or σ_eff·N(0,1) by Box-Muller on Philox, where
// σ_eff = RN32(σ × noise_scale of the learner)
__global__ void __launch_bounds__(256)
ddpg_act_epilogue_kernel(const float* __restrict__ y /*[n][2]*/, long long n, float sigma, const DdpgCtrl* __restrict__ ctrl, unsigned long long seed, long long step,
                         long long env_id_base, const float* __restrict__ noise, float lo0, float lo1, float hi0, float hi1,
                         float* __restrict__ a_out, float* __restrict__ scaled_out, long long act_stride, long long asl, long long ask,
                         float* __restrict__ noise_acc, int noise_first) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (noise_acc) noise_acc += (long long)blockIdx.y * n;   // [P*n], instance j of learner l at l*n + j
  {  // blockIdx.y = learner l of a population: component k of its instance j sits at [l*asl + k*ask + j] in noise / a / scaled
     // (packed [P][2][n]: asl = 2n, ask = n; SoA over all instances: asl = n, ask = N); noise streams are keyed by the global env id
    const long long l = blockIdx.y;
    y += l * act_stride; a_out += l * asl; env_id_base += l * n;
    sigma = __fmul_rn(sigma, ctrl[l].hp.noise_scale);
    if (noise) noise += l * asl;
    if (scaled_out) scaled_out += l * asl;
  }
  const bool have = noise != nullptr;
  const ActOut o = act_gauss_epilogue(y[j * 2 + 0], y[j * 2 + 1], have, have ? noise[j] : 0.0f, have ? noise[ask + j] : 0.0f, sigma, seed, step,
                                      env_id_base + j, lo0, lo1, hi0, hi1);
  a_out[j] = o.a0; a_out[ask + j] = o.a1;
  if (scaled_out) { scaled_out[j] = o.s0; scaled_out[ask + j] = o.s1; }
  if (noise_acc) noise_acc[j] = __fadd_rn(noise_first ? 0.0f : noise_acc[j], o.noise_mean);   // noise_eps += noise (DDPG.jl:224)
}

// OUNoise (DDPG.jl:49-55, input.jl:190-234) with Julia's types: θ, μ, σ, dt and X are Float32, randn is Float64:
//   dx = θ .* (μ .- X) .* dt              (Float32)
//   dx .+= σ .* sqrt(dt) .* randn(2)      (Float32(σ·√dt) · z in Float64, added in Float64, stored Float32; σ = RN32(σ × noise_scale))
//   X .+= dx;  noise = Float32.(X)        (X persists across steps AND episodes: the reference never resets it)
// Every instance carries its own X (ou_x [2][n]); z: caller-supplied standard normal draws or Philox + Box-Muller.
__global__ void __launch_bounds__(256)
ddpg_act_ou_epilogue_kernel(const float* __restrict__ y /*[n][2]*/, long long n, float theta, float mu, float sigma, const DdpgCtrl* __restrict__ ctrl,
                            float dt, float* __restrict__ ou_x,
                            unsigned long long seed, long long step, long long env_id_base, const double* __restrict__ z, float lo0, float lo1,
                            float hi0, float hi1, float* __restrict__ a_out, float* __restrict__ scaled_out, long long act_stride,
                            long long asl, long long ask, float* __restrict__ noise_acc, int noise_first) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (noise_acc) noise_acc += (long long)blockIdx.y * n;
  {  // learner l = blockIdx.y; component k of its instance j at [l*asl + k*ask + j] (packed: asl = 2n, ask = n; SoA: asl = n, ask = N)
    const long long l = blockIdx.y;
    y += l * act_stride; a_out += l * asl; ou_x += l * asl; env_id_base += l * n;
    sigma = __fmul_rn(sigma, ctrl[l].hp.noise_scale);
    if (z) z += l * asl;
    if (scaled_out) scaled_out += l * asl;
  }
  double z0, z1;
  if (z) { z0 = z[j]; z1 = z[ask + j]; }
  else {
    uint32_t w[4];
    philox4x32_10(seed, (uint64_t)(env_id_base + j), (uint32_t)step, STREAM_NOISE, w);
    const double u1 = 1.0 - u53(w[0], w[1]), u2 = u53(w[2], w[3]);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    z0 = rad * cs; z1 = rad * sn;
  }
  const float ssd = __fmul_rn(sigma, __fsqrt_rn(dt));
  float nz[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float x = ou_x[k * ask + j];
    float dx = __fmul_rn(__fmul_rn(theta, __fsub_rn(mu, x)), dt);
    dx = (float)__dadd_rn((double)dx, __dmul_rn((double)ssd, k == 0 ? z0 : z1));
    nz[k] = __fadd_rn(x, dx);
    ou_x[k * ask + j] = nz[k];
  }
  if (noise_acc) noise_acc[j] = __fadd_rn(noise_first ? 0.0f : noise_acc[j], __fmul_rn(__fadd_rn(nz[0], nz[1]), 0.5f));   // mean(Float32.(ou.X))
  float a0 = __fadd_rn(y[j * 2 + 0], nz[0]), a1 = __fadd_rn(y[j * 2 + 1], nz[1]);
  a0 = a0 > 1.0f ? 1.0f : (a0 < -1.0f ? -1.0f : a0);
  a1 = a1 > 1.0f ? 1.0f : (a1 < -1.0f ? -1.0f : a1);
  a_out[j] = a0; a_out[ask + j] = a1;
  if (scaled_out) {
    const double sp0 = (double)__fsub_rn(hi0, lo0), sp1 = (double)__fsub_rn(hi1, lo1);
    scaled_out[j] = (float)__dadd_rn((double)lo0, __dmul_rn(__dmul_rn(__dadd_rn((double)a0, 1.0), 0.5), sp0));
    scaled_out[ask + j] = (float)__dadd_rn((double)lo1, __dmul_rn(__dmul_rn(__dadd_rn((double)a1, 1.0), 0.5), sp1));
  }
}

// actor(normalize(s)) for n states per learner -> h->act_y [n][2] (pre-noise); shared by the noise variants of act()
// act() on a handful of states of one learner runs as one cluster kernel (csrc/ddpg_fused.cu)
static inline bool fused_act_ok(const Ddpg* h, int64_t n) { return use_fused(h) && h->pop == 1 && n <= FUSED_ACT_MAX_ROWS; }
static FusedActArgs fused_act_args(const Ddpg* h, const float* obs_dev, int64_t n, long long osk) {
  FusedActArgs a; memset(&a, 0, sizeof(a));
  a.actor = h->net[DDPG_NET_ACTOR];
  a.ao = fused_off(h->dims[0]);
  a.l1 = h->p.l1; a.l2 = h->p.l2;
  a.vec16 = w2_vec16(h) ? 1 : 0;
  a.n = n; a.obs = obs_dev; a.osk = osk; a.norm = h->norm; a.y = h->act_y;
  return a;
}
static int act_forward(Ddpg* h, const float* obs_dev, int64_t n, long long osl, long long osk) {
  const int l1 = h->ld1, l2 = h->ld2, pop = h->pop;
  if (h->act_cap < n) {  // scratch: per learner [x n*9 | h1 n*ld1 | h2 n*ld2 | y n*2], each part at a 256-byte boundary
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->act_x);
    h->act_x = h->act_h1 = h->act_h2 = h->act_y = nullptr; h->act_cap = 0;
    const long long o1 = (9 * n + 63) & ~63ll, o2 = o1 + (((long long)l1 * n + 63) & ~63ll), o3 = o2 + (((long long)l2 * n + 63) & ~63ll);
    h->act_stride = o3 + ((2 * n + 63) & ~63ll);
    CUDA_TRY(cudaMalloc(&h->act_x, sizeof(float) * (size_t)h->act_stride * (size_t)pop));
    h->act_h1 = h->act_x + o1; h->act_h2 = h->act_x + o2; h->act_y = h->act_x + o3;
    h->act_cap = n;
  }
  if (fused_act_ok(h, n)) {  // a handful of states (the reference acts on one): one cluster kernel
    FusedActArgs a = fused_act_args(h, obs_dev, n, osk);
    return ddpg_fused_act(h->stream, a);
  }
  const dim3 gn((unsigned)((n + 255) / 256), pop);
  ddpg_normalize_kernel<<<gn, 256, 0, h->stream>>>(obs_dev, n, h->norm, h->act_x, h->pop_stride, h->act_stride, osl, osk);
  CUDA_TRY(cudaGetLastError());
  const Regime rg{false, use_tc(h, n), n * pop >= SPLITK_MIN_BATCH};
  const FwdNet fwd = {h->act_x, h->net[DDPG_NET_ACTOR], &h->dims[0], h->act_h1, h->act_h2, false, TC_OUT_TANH, h->act_y, 2};
  return enqueue_forward(h, h->stream, rg, &fwd, 1, 9, (int)n, h->act_stride);
}

// sprev_dev (optional, [9][N]): receives a copy of the raw states — the episode loop's s for `remember`
static int act_gauss(Ddpg* h, const float* obs_dev, int64_t n, float sigma, uint64_t seed, int64_t step, int64_t env_id_base,
                     const float* noise_dev, float* a_dev, float* scaled_dev, bool soa, float* sprev_dev = nullptr, float* noise_acc = nullptr,
                     int noise_first = 0) {
  REQUIRE(h && obs_dev && a_dev, SHEMS_ERR_INVALID, "ddpg_act: NULL argument");
  REQUIRE(n >= 1 && n < (1ll << 31), SHEMS_ERR_INVALID, "ddpg_act: n=%lld", (long long)n);
  GUARD(h->device);
  const long long N = (long long)n * h->pop;
  if (fused_act_ok(h, n)) {  // normalize, the actor's three layers, noise, clamp, scale_action (and the copy of s) in ONE cluster kernel
    FusedActArgs a = fused_act_args(h, obs_dev, n, n);   // one learner: packed [9][n] and SoA [9][N] coincide
    a.a_out = a_dev; a.scaled_out = scaled_dev; a.noise = noise_dev; a.ask = n;
    a.sigma = sigma * h->hp[0].noise_scale; a.seed = seed; a.step = step; a.env_id_base = env_id_base;   // RN32, as the kernels form it
    a.lo0 = h->p.act_lo[0]; a.lo1 = h->p.act_lo[1]; a.hi0 = h->p.act_hi[0]; a.hi1 = h->p.act_hi[1];
    a.sprev = sprev_dev; a.noise_acc = noise_acc; a.noise_first = noise_first;
    return ddpg_fused_act(h->stream, a);
  }
  if (sprev_dev) CUDA_TRY(cudaMemcpyAsync(sprev_dev, obs_dev, sizeof(float) * 9 * (size_t)N, cudaMemcpyDeviceToDevice, h->stream));
  TRY(act_forward(h, obs_dev, n, soa ? n : 9 * n, soa ? N : n));
  const dim3 gn((unsigned)((n + 255) / 256), h->pop);
  ddpg_act_epilogue_kernel<<<gn, 256, 0, h->stream>>>(h->act_y, n, sigma, h->ctrl, seed, step, env_id_base, noise_dev, h->p.act_lo[0], h->p.act_lo[1],
                                                      h->p.act_hi[0], h->p.act_hi[1], a_dev, scaled_dev, h->act_stride, soa ? n : 2 * n,
                                                      soa ? N : n, noise_acc, noise_first);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
extern "C" int32_t ddpg_act(Ddpg* h, const float* obs_dev, int64_t n, float sigma, uint64_t seed, int64_t step, int64_t env_id_base,
                            const float* noise_dev, float* a_dev, float* scaled_dev) {
  return act_gauss(h, obs_dev, n, sigma, seed, step, env_id_base, noise_dev, a_dev, scaled_dev, false);
}
// the same with every array laid out as ONE structure-of-arrays over all N = P*n instances of the population (learner l owns
// instances l*n .. l*n+n-1): obs [9][N] is exactly the state array of an environment handle, scaled_dev [2][N] its action input
extern "C" int32_t ddpg_act_soa(Ddpg* h, const float* obs_dev, int64_t n, float sigma, uint64_t seed, int64_t step, int64_t env_id_base,
                                const float* noise_dev, float* a_dev, float* scaled_dev) {
  return act_gauss(h, obs_dev, n, sigma, seed, step, env_id_base, noise_dev, a_dev, scaled_dev, true);
}

static int act_ou(Ddpg* h, const float* obs_dev, int64_t n, float theta, float mu, float sigma, float dt, float* ou_x_dev, uint64_t seed,
                  int64_t step, int64_t env_id_base, const double* z_dev, float* a_dev, float* scaled_dev, bool soa, float* noise_acc = nullptr,
                  int noise_first = 0) {
  REQUIRE(h && obs_dev && a_dev && ou_x_dev, SHEMS_ERR_INVALID, "ddpg_act_ou: NULL argument");
  REQUIRE(n >= 1 && n < (1ll << 31), SHEMS_ERR_INVALID, "ddpg_act_ou: n=%lld", (long long)n);
  REQUIRE(dt >= 0.0f, SHEMS_ERR_INVALID, "ddpg_act_ou: dt=%g (sqrt(dt) raises DomainError in the reference)", (double)dt);
  GUARD(h->device);
  const long long N = (long long)n * h->pop;
  TRY(act_forward(h, obs_dev, n, soa ? n : 9 * n, soa ? N : n));
  const dim3 gn((unsigned)((n + 255) / 256), h->pop);
  ddpg_act_ou_epilogue_kernel<<<gn, 256, 0, h->stream>>>(h->act_y, n, theta, mu, sigma, h->ctrl, dt, ou_x_dev, seed, step, env_id_base, z_dev,
                                                         h->p.act_lo[0], h->p.act_lo[1], h->p.act_hi[0], h->p.act_hi[1], a_dev, scaled_dev,
                                                         h->act_stride, soa ? n : 2 * n, soa ? N : n, noise_acc, noise_first);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
extern "C" int32_t ddpg_act_ou(Ddpg* h, const float* obs_dev, int64_t n, float theta, float mu, float sigma, float dt, float* ou_x_dev,
                               uint64_t seed, int64_t step, int64_t env_id_base, const double* z_dev, float* a_dev, float* scaled_dev) {
  return act_ou(h, obs_dev, n, theta, mu, sigma, dt, ou_x_dev, seed, step, env_id_base, z_dev, a_dev, scaled_dev, false);
}
// noise_type of ddpg_episode (input.jl:111): 0 = "gn" (GNoise, the default), 1 = "ou" (OUNoise(mu, sigma, theta, dt, X), input.jl:190-234;
// X lives in the handle, one pair per instance, and — like the reference's global `ou` — is never reset)
extern "C" int32_t ddpg_set_noise(Ddpg* h, int32_t kind, float theta, float mu, float dt) {
  REQUIRE(h && (kind == 0 || kind == 1), SHEMS_ERR_INVALID, "ddpg_set_noise: kind=%d (0 gn, 1 ou)", kind);
  REQUIRE(dt >= 0.0f, SHEMS_ERR_INVALID, "ddpg_set_noise: dt=%g", (double)dt);
  h->noise_kind = kind; h->ou_theta = theta; h->ou_mu = mu; h->ou_dt = dt;
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- episode!
// reward_eps += r (DDPG.jl:223): the Float64 env.reward of every step (shems_LU1.jl:171) is summed in Float64; the replay memory
// keeps Float32(r), which is what `cu` makes of it when getData uploads the minibatch (memory_plotting_saving.jl:37)
__global__ void __launch_bounds__(256)
ddpg_accum_return_kernel(const double* __restrict__ r, double* __restrict__ ret, long long n, int first) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ret[i] = (first ? 0.0 : ret[i]) + r[i];
}

// One learner's episode loop, after step!: remember (DDPG.jl:229 — the n transitions go to ring slots head .. head+n-1), reward_eps += r
// (:223) and the host-owned part of the control block of the replay() that follows (seed, update number, ring geometry), all
// passed BY VALUE: one launch in place of two kernels and three small host-to-device copies per step.
__global__ void __launch_bounds__(256)
ddpg_episode_post_step_kernel(float* __restrict__ ring, long long cap, long long head, const float* __restrict__ s, const float* __restrict__ a,
                              const float* __restrict__ r, const double* __restrict__ r64, const float* __restrict__ s2, long long n,
                              double* __restrict__ ep_ret, int first, DdpgCtrl* __restrict__ ctrl, CtrlHostPart hp,
                              const float** __restrict__ rings_dev) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && ctrl) { *reinterpret_cast<CtrlHostPart*>(ctrl) = hp; rings_dev[0] = ring; }
  if (i >= n) return;
  float* q = ring + ring_base(ring_push_slot(head, i, cap));
  float si[9], s2i[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { si[k] = s[k * n + i]; s2i[k] = s2[k * n + i]; }
  ring_store_full(q, si, a[i], a[n + i], r[i], s2i, 0.0f);
  if (ep_ret) ep_ret[i] = (first ? 0.0 : ep_ret[i]) + r64[i];
}

// episode!(env; NUM_STEPS, train, track = 0, rng_ep) (DDPG.jl:186-242) for all instances of `env`, enqueued in one call with no host
// round trip per step: act(normalize(s)) [+ gn noise when train] -> scale_action -> step! -> remember -> replay() x updates_per_step.
// The environment must have been reset by the caller (reset! is :189).  env holds N = P*n instances, learner l owns instances
// l*n .. l*n+n-1 and the replay memory rps[l].  Per-step seeds: rng_step = (seed*1000003 + step) mod 2^63 feeds the noise stream
// (keyed by the global env id) and, as rng_step + l, learner l's minibatch stream — the same rule the Python Driver uses.
// All three handles must be bound to the same CUDA stream.  ep_return_dev [N] (Float64) receives the summed rewards, or NULL.
extern "C" int32_t ddpg_episode(Ddpg* h, ShemsEnv* env, ShemsReplay* const* rps, int32_t n_steps, int32_t train, float sigma, uint64_t seed,
                                int32_t updates_per_step, int64_t env_id_base, double* ep_return_dev, float* noise_eps_dev) {
  REQUIRE(h && env, SHEMS_ERR_INVALID, "ddpg_episode: NULL argument");
  REQUIRE(n_steps >= 1 && updates_per_step >= 0, SHEMS_ERR_INVALID, "ddpg_episode: n_steps=%d updates_per_step=%d", n_steps, updates_per_step);
  REQUIRE(!train || rps, SHEMS_ERR_INVALID, "ddpg_episode: training needs the replay memories");
  REQUIRE(env->device == h->device, SHEMS_ERR_INVALID, "ddpg_episode: env on device %d, learner on %d", env->device, h->device);
  REQUIRE(env->n % h->pop == 0, SHEMS_ERR_INVALID, "ddpg_episode: %lld instances do not split over %d learners", (long long)env->n, h->pop);
  REQUIRE(env->stream == h->stream && (!train || rps[0]->stream == h->stream), SHEMS_ERR_STATE,
          "ddpg_episode: bind the environment, the learner and the replay memories to one CUDA stream");
  REQUIRE(env->was_reset, SHEMS_ERR_STATE, "ddpg_episode: reset! must come first");
  if (train) TRY(per_memories_ok(h, rps, "ddpg_episode"));
  if (train) TRY(nstep_memories_ok(h, rps, "ddpg_episode"));
  if (ensure_rows(env, n_steps)) {  // nothing is enqueued for an episode that would leave the series
    shems_set_error("BoundsError: episode of %d steps from row %d leaves the %d-row series (next_state!, shems_LU1.jl:266-268)", n_steps, env->max_idx,
                    env->nrows);
    return SHEMS_ERR_BOUNDS;
  }
  GUARD(h->device);
  const long long N = env->n, n = N / h->pop;
  if (h->ep_cap < N) {
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->ep_a); h->ep_a = nullptr; h->ep_cap = 0;
    CUDA_TRY(cudaMalloc(&h->ep_a, sizeof(float) * 16 * (size_t)N));
    h->ep_scaled = h->ep_a + 2 * N; h->ep_sprev = h->ep_a + 4 * N; h->ep_r = h->ep_a + 13 * N;
    h->ep_r64 = reinterpret_cast<double*>(h->ep_a + 14 * N);   // 8-byte aligned: cudaMalloc base + 56 N bytes
    h->ep_cap = N;
  }
  if (train && h->noise_kind == 1 && h->ou_cap != N) {  // first use (or another environment size): X = zeros (input.jl:234)
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->ou_x); h->ou_x = nullptr; h->ou_cap = 0;
    CUDA_TRY(cudaMalloc(&h->ou_x, sizeof(float) * 2 * (size_t)N));
    CUDA_TRY(cudaMemsetAsync(h->ou_x, 0, sizeof(float) * 2 * (size_t)N, h->stream));
    h->ou_cap = N;
  }
  std::vector<uint64_t> seeds((size_t)h->pop);
  if (train && h->per && h->pop == 1 && updates_per_step > 0)   // the post-step kernel below stages the ring, not the tree
    CUDA_TRY(cudaMemcpyAsync(h->trees_dev, &rps[0]->prio, sizeof(float*), cudaMemcpyHostToDevice, h->stream));
  if (train && h->nstep > 1 && h->pop == 1 && updates_per_step > 0)   // and not the links either
    CUDA_TRY(cudaMemcpyAsync((void*)h->links_dev, &rps[0]->next, sizeof(const int32_t*), cudaMemcpyHostToDevice, h->stream));
  for (int step = 1; step <= n_steps; ++step) {
    const uint64_t rng_step = (seed * 1000003ull + (uint64_t)step) & 0x7fffffffffffffffull;
    if (train && h->noise_kind == 1) {
      TRY(act_ou(h, env->obs, n, h->ou_theta, h->ou_mu, sigma, h->ou_dt, h->ou_x, rng_step, step, env_id_base, nullptr, h->ep_a, h->ep_scaled, true,
                 noise_eps_dev, step == 1));
      CUDA_TRY(cudaMemcpyAsync(h->ep_sprev, env->obs, sizeof(float) * 9 * (size_t)N, cudaMemcpyDeviceToDevice, h->stream));
    } else {
      TRY(act_gauss(h, env->obs, n, train ? sigma : 0.0f, rng_step, step, env_id_base, nullptr, h->ep_a, h->ep_scaled, true,
                    train ? h->ep_sprev : nullptr, noise_eps_dev, step == 1));
    }
    TRY(shems_step(env, h->ep_scaled, 0, h->ep_r, h->ep_r64, nullptr, nullptr));
    if (train && h->pop == 1 && !h->dp_on) {  // one learner: remember + reward_eps + the next replay()'s control block in one launch
      ShemsReplay* rp = rps[0];
      REQUIRE(rp && rp->device == h->device, SHEMS_ERR_INVALID, "ddpg_episode: replay memory missing or on another device");
      REQUIRE(N <= rp->capacity, SHEMS_ERR_INVALID, "ddpg_episode: %lld instances exceed the memory's capacity %lld", N, (long long)rp->capacity);
      const long long head = rp->head, cap = rp->capacity;
      CtrlHostPart hp; memset(&hp, 0, sizeof(hp));
      hp.seed = rng_step; hp.update = 0u; hp.use_idx = 0;
      hp.len = rp->length + N > cap ? cap : rp->length + N; hp.head = (head + N) % cap; hp.cap = cap;   // the ring after this step's push
      ddpg_episode_post_step_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(rp->ring, rp->capacity, head, h->ep_sprev, h->ep_a, h->ep_r,
                                                                                       h->ep_r64, env->obs, N, ep_return_dev, step == 1,
                                                                                       updates_per_step > 0 ? h->ctrl : nullptr, hp, h->rings_dev);
      CUDA_TRY(cudaGetLastError());
      TRY(replay_after_rollout(rp, N, N, h->stream));   // after the kernel: the link pass reads the records it wrote
      if (updates_per_step > 0) {
        TRY(ensure_graph(h));
        for (int u = 0; u < updates_per_step; ++u) CUDA_TRY(cudaGraphLaunch(h->graph_exec, h->stream));
        h->n_updates += updates_per_step;
      }
      continue;
    }
    if (ep_return_dev) {
      ddpg_accum_return_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->ep_r64, ep_return_dev, N, step == 1);
      CUDA_TRY(cudaGetLastError());
    }
    if (train) {
      TRY(replay_push_groups(rps, h->pop, h->ep_sprev, h->ep_a, h->ep_r, env->obs, nullptr, n));   // the unscaled action is stored (:229)
      if (updates_per_step > 0 && h->dp_on) {
        // a connected data-parallel learner: every rank steps its own instances and memory, the update exchanges gradients
        // (all ranks make the same calls) — never the local-only graph, which would let the replicas drift apart
        TRY(ddpg_update_dp(h, rps[0], updates_per_step, nullptr, rng_step));
      } else if (updates_per_step > 0) {
        for (int l = 0; l < h->pop; ++l) seeds[l] = rng_step + (uint64_t)l;
        TRY(ddpg_update_population(h, rps, updates_per_step, nullptr, seeds.data()));                  // replay(rng_rpl = rng_step) (:231)
      }
    }
  }
  return SHEMS_OK;
}

// The persistent cluster kernel (csrc/actor_rollout.cu) over every instance group of `env`, one launch per group: ddpg_rollout's
// one-learner branch and ddpg_evaluate share it.  actor: learner 0's copy of the net to run, actor_stride floats between learners'
// copies.  One learner: the whole group is one segment; populations: learner l owns instances l*n .. l*n+n-1, which the caller has
// checked lie inside one group.
static int rollout_launch(Ddpg* h, ShemsEnv* env, const float* actor, long long actor_stride, int32_t n_steps, float sigma, uint64_t seed,
                          int64_t env_id_base, double* ep_return_dev, double* trace_dev, float* act_traj_dev) {
  const long long N = env->n, n = N / h->pop;
  ActorRolloutArgs a; memset(&a, 0, sizeof(a));
  a.actor = actor;
  a.ao = fused_off(h->dims[0]);
  a.l1 = h->p.l1; a.l2 = h->p.l2;
  a.vec16 = w2_vec16(h) ? 1 : 0;
  a.norm = h->norm; a.actor_stride = actor_stride; a.norm_stride = h->pop_stride;
  a.N = N; a.obs = env->obs; a.idx = env->idx; a.T = n_steps; a.step0 = env->step;
  a.sigma = sigma * h->hp[0].noise_scale; a.seed = seed; a.env_id_base = env_id_base;
  a.lo0 = h->p.act_lo[0]; a.lo1 = h->p.act_lo[1]; a.hi0 = h->p.act_hi[0]; a.hi1 = h->p.act_hi[1];
  a.ep_return = ep_return_dev; a.trace = trace_dev; a.act_traj = act_traj_dev;
  for (int g = 0; g < env->n_groups; ++g) {
    a.P = env->gdp[g]; a.series = env->gseries[g]; a.n0 = env->gstart[g]; a.n1 = env->gstart[g + 1];
    a.seg = h->pop == 1 ? a.n1 - a.n0 : n;
    a.l0 = h->pop == 1 ? 0 : a.n0 / n;
    TRY(actor_rollout_launch(h->stream, a));
  }
  return SHEMS_OK;
}

// episode!(env; NUM_STEPS, train = false, track, rng_ep) (DDPG.jl:186-242) / inference(env; track = 1) (memory_plotting_saving.jl:62-89)
// for every instance of `env`: act(normalize(s)) [+ GNoise when sigma > 0] -> scale_action -> step!, n_steps times, by ONE call.
// One learner at the fused shapes: a single persistent cluster kernel per group of instances (csrc/actor_rollout.cu) — no launch,
// no host round trip per step.  Populations / wider nets: one act + step! launch pair per step.
extern "C" int32_t ddpg_rollout(Ddpg* h, ShemsEnv* env, int32_t n_steps, float sigma, uint64_t seed, int64_t env_id_base, double* ep_return_dev,
                                double* trace_dev, float* act_traj_dev) {
  REQUIRE(h && env, SHEMS_ERR_INVALID, "ddpg_rollout: NULL argument");
  REQUIRE(n_steps >= 1, SHEMS_ERR_INVALID, "ddpg_rollout: n_steps=%d", n_steps);
  REQUIRE(env->device == h->device, SHEMS_ERR_INVALID, "ddpg_rollout: env on device %d, learner on %d", env->device, h->device);
  REQUIRE(env->n % h->pop == 0, SHEMS_ERR_INVALID, "ddpg_rollout: %lld instances do not split over %d learners", (long long)env->n, h->pop);
  REQUIRE(env->stream == h->stream, SHEMS_ERR_STATE, "ddpg_rollout: bind the environment and the learner to one CUDA stream");
  REQUIRE(env->was_reset, SHEMS_ERR_STATE, "ddpg_rollout: reset! must come first");
  if (ensure_rows(env, n_steps)) {
    shems_set_error("BoundsError: rollout of %d steps from row %d leaves the %d-row series (next_state!, shems_LU1.jl:266-268)", n_steps, env->max_idx,
                    env->nrows);
    return SHEMS_ERR_BOUNDS;
  }
  GUARD(h->device);
  const long long N = env->n, n = N / h->pop;
  if (h->pop == 1 && h->rollout_ok) {
    TRY(rollout_launch(h, env, h->net[DDPG_NET_ACTOR], 0, n_steps, sigma, seed, env_id_base, ep_return_dev, trace_dev, act_traj_dev));
    env->max_idx += n_steps; env->step += n_steps; env->consistent = true;
    return SHEMS_OK;
  }
  if (h->ep_cap < N) {
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->ep_a); h->ep_a = nullptr; h->ep_cap = 0;
    CUDA_TRY(cudaMalloc(&h->ep_a, sizeof(float) * 16 * (size_t)N));
    h->ep_scaled = h->ep_a + 2 * N; h->ep_sprev = h->ep_a + 4 * N; h->ep_r = h->ep_a + 13 * N;
    h->ep_r64 = reinterpret_cast<double*>(h->ep_a + 14 * N);
    h->ep_cap = N;
  }
  for (int t = 0; t < n_steps; ++t) {
    const int step = env->step + 1;
    const uint64_t rng_step = (seed * 1000003ull + (uint64_t)step) & 0x7fffffffffffffffull;
    float* a_out = act_traj_dev ? act_traj_dev + (size_t)t * 2 * N : h->ep_a;
    TRY(act_gauss(h, env->obs, n, sigma, rng_step, step, env_id_base, nullptr, a_out, h->ep_scaled, true, nullptr));
    TRY(shems_step(env, h->ep_scaled, trace_dev ? 1 : 0, nullptr, h->ep_r64, nullptr, trace_dev ? trace_dev + (size_t)t * SHEMS_TRACE_COLS * N : nullptr));
    if (ep_return_dev) {
      ddpg_accum_return_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->ep_r64, ep_return_dev, N, t == 0);
      CUDA_TRY(cudaGetLastError());
    }
  }
  return SHEMS_OK;
}

// episode!(env; train = false) (DDPG.jl:266-271) / inference(env; track = 1) for EVERY learner of the handle, noise-free, by one call: the
// persistent cluster kernel with a learner dimension (every cluster serves 8 instances of one learner and reads that learner's actor and
// s_min / s_max), so a learner's evaluation inside a population has the bits of its evaluation on a one-learner handle.
// net: DDPG_NET_ACTOR or DDPG_NET_ACTOR_BEST (the slot ddpg_keep_best fills).
extern "C" int32_t ddpg_evaluate(Ddpg* h, ShemsEnv* env, int32_t net, int32_t n_steps, int64_t env_id_base, double* ep_return_dev, double* trace_dev,
                                 float* act_traj_dev) {
  REQUIRE(h && env, SHEMS_ERR_INVALID, "ddpg_evaluate: NULL argument");
  REQUIRE(net == DDPG_NET_ACTOR || net == DDPG_NET_ACTOR_BEST, SHEMS_ERR_INVALID, "ddpg_evaluate: net=%d (ACTOR or ACTOR_BEST)", net);
  REQUIRE(n_steps >= 1, SHEMS_ERR_INVALID, "ddpg_evaluate: n_steps=%d", n_steps);
  REQUIRE(env->device == h->device, SHEMS_ERR_INVALID, "ddpg_evaluate: env on device %d, learner on %d", env->device, h->device);
  REQUIRE(env->n % h->pop == 0, SHEMS_ERR_INVALID, "ddpg_evaluate: %lld instances do not split over %d learners", (long long)env->n, h->pop);
  REQUIRE(h->rollout_ok, SHEMS_ERR_INVALID, "ddpg_evaluate: widths l1=%d l2=%d outside the cluster kernel's plan (l1 <= %d, l2 <= %d)", h->p.l1,
          h->p.l2, FUSED_MAX_L1, FUSED_MAX_L2);
  const long long N = env->n, n = N / h->pop;
  for (int g = 1; g < env->n_groups && h->pop > 1; ++g)   // one learner: every group is a segment of its own (as ddpg_rollout)
    REQUIRE(env->gstart[g] % n == 0, SHEMS_ERR_INVALID, "ddpg_evaluate: the group starting at instance %lld splits the %lld instances of learner %lld",
            (long long)env->gstart[g], n, (long long)(env->gstart[g] / n));
  REQUIRE(env->stream == h->stream, SHEMS_ERR_STATE, "ddpg_evaluate: bind the environment and the learner to one CUDA stream");
  REQUIRE(env->was_reset, SHEMS_ERR_STATE, "ddpg_evaluate: reset! must come first");
  if (ensure_rows(env, n_steps)) {
    shems_set_error("BoundsError: evaluation of %d steps from row %d leaves the %d-row series (next_state!, shems_LU1.jl:266-268)", n_steps, env->max_idx,
                    env->nrows);
    return SHEMS_ERR_BOUNDS;
  }
  GUARD(h->device);
  const float* actor = net == DDPG_NET_ACTOR ? h->net[DDPG_NET_ACTOR] : h->best;
  const long long stride = net == DDPG_NET_ACTOR ? h->pop_stride : h->best_stride;
  TRY(rollout_launch(h, env, actor, stride, n_steps, 0.0f, 0, env_id_base, ep_return_dev, trace_dev, act_traj_dev));
  env->max_idx += n_steps; env->step += n_steps; env->consistent = true;
  return SHEMS_OK;
}

// run_episodes' bookkeeping after an evaluation round (DDPG.jl:273, :282-289) for every learner: one block per learner, so the
// decision and the copy it gates are made by the same block.  Thread 0 forms score = (Σ_k ep_return[l·n + k]) / n in index order in
// Float64 and, when score > best_score (strict: ties and NaN never win), records it with the episode; then the block copies the
// learner's actor into its best-actor slot.
__global__ void __launch_bounds__(256)
ddpg_keep_best_kernel(const double* __restrict__ ep_return, long long n, int episode, double* __restrict__ score_out, double* __restrict__ best_score,
                      int32_t* __restrict__ best_run, const float* __restrict__ actor, long long pop_stride, float* __restrict__ best,
                      long long best_stride, long long na) {
  __shared__ int take;
  const long long l = blockIdx.x;
  if (threadIdx.x == 0) {
    double sum = 0.0;
    for (long long k = 0; k < n; ++k) sum += ep_return[l * n + k];
    const double score = sum / (double)n;
    if (score_out) score_out[l] = score;
    take = score > best_score[l];
    if (take) { best_score[l] = score; best_run[l] = episode; }
  }
  __syncthreads();
  if (!take) return;
  const float* src = actor + l * pop_stride;   // both copies start on 256-byte boundaries
  float* dst = best + l * best_stride;
  const long long n4 = na / 4;
  for (long long i = threadIdx.x; i < n4; i += blockDim.x) reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src)[i];
  for (long long i = 4 * n4 + threadIdx.x; i < na; i += blockDim.x) dst[i] = src[i];
}
extern "C" int32_t ddpg_keep_best(Ddpg* h, const double* ep_return_dev, int64_t n, int32_t episode, double* score_dev) {
  REQUIRE(h && ep_return_dev, SHEMS_ERR_INVALID, "ddpg_keep_best: NULL argument");
  REQUIRE(n >= 1, SHEMS_ERR_INVALID, "ddpg_keep_best: n=%lld", (long long)n);
  GUARD(h->device);
  ddpg_keep_best_kernel<<<h->pop, 256, 0, h->stream>>>(ep_return_dev, n, episode, score_dev, h->best_score, h->best_run, h->net[DDPG_NET_ACTOR],
                                                       h->pop_stride, h->best, h->best_stride, h->dims[0].n_params);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_best(Ddpg* h, double* best_score_host, int32_t* best_run_host) {
  REQUIRE(h && best_score_host && best_run_host, SHEMS_ERR_INVALID, "ddpg_get_best: NULL argument");
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(best_score_host, h->best_score, sizeof(double) * (size_t)h->pop, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(best_run_host, h->best_run, sizeof(int32_t) * (size_t)h->pop, cudaMemcpyDeviceToHost));
  return SHEMS_OK;
}
extern "C" int32_t ddpg_set_best(Ddpg* h, const double* best_score_host, const int32_t* best_run_host) {
  REQUIRE(h && best_score_host && best_run_host, SHEMS_ERR_INVALID, "ddpg_set_best: NULL argument");
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(h->best_score, best_score_host, sizeof(double) * (size_t)h->pop, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->best_run, best_run_host, sizeof(int32_t) * (size_t)h->pop, cudaMemcpyHostToDevice));
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- population-based training (exploit + explore)
// ddpg_exploit: inside every group of learners the bottom share takes over the learner state of a learner drawn from the top share and
// perturbs its hyper-parameters.  Grid (copy chunks x P), blockIdx.y = learner d.  Every block works out d's decision itself from the
// scores (a pure function of scores, seed, round and d), so all blocks of d agree without talking to each other and the call is one
// launch.  Top (rank < k) and bottom (rank >= m - k) sets are disjoint for k <= m / 2: no learner is read and written in one call.
#define EXPLOIT_THREADS 256
#define EXPLOIT_UNROLL 8
#define EXPLOIT_CHUNK (EXPLOIT_THREADS * EXPLOIT_UNROLL)   // float4 per block
#define EXPLOIT_PARTS 9
struct ExploitArgs {
  const double* score; float* slab; long long pop_stride; DdpgCtrl* ctrl; int32_t* parent;
  long long part_off[EXPLOIT_PARTS], part_n4[EXPLOIT_PARTS];   // float4 offset of a part inside a learner's slab, float4 count
  double frac; float factor_lo, factor_hi; int keys; unsigned round; unsigned long long seed;
  int n_groups; int group_start[DDPG_EXPLOIT_MAX_GROUPS + 1];
};
// the sort key: the score with NaN as -inf; learner i ranks before learner j on a larger key, ties to the lower index
__device__ __forceinline__ double pbt_key(double s) { return isnan(s) ? -INFINITY : s; }
__device__ __forceinline__ bool pbt_before(double ki, int i, double kj, int j) { return ki > kj || (ki == kj && i < j); }
// hyper-parameter j of the source (bit j of keys set): x * factor in one fp32 multiply; gamma and tau then at most 1
__device__ __forceinline__ float pbt_perturb(float x, int j, int keys, unsigned w1, float lo, float hi) {
  if (!((keys >> j) & 1)) return x;
  const float y = __fmul_rn(x, ((w1 >> j) & 1u) ? hi : lo);
  return (j == 2 || j == 3) ? fminf(y, 1.0f) : y;
}
__device__ __forceinline__ int block_sum(int v, int* red) {
  v = __reduce_add_sync(0xffffffffu, v);
  __syncthreads();   // red may still be read from an earlier call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  int s = 0;
#pragma unroll
  for (int w = 0; w < EXPLOIT_THREADS / 32; ++w) s += red[w];
  return s;
}

__global__ void __launch_bounds__(EXPLOIT_THREADS) ddpg_exploit_kernel(const ExploitArgs a) {
  __shared__ int red[EXPLOIT_THREADS / 32];
  __shared__ int s_src;
  const int d = blockIdx.y, tid = threadIdx.x;
  int g = 0;
  while (d >= a.group_start[g + 1]) ++g;
  const int g0 = a.group_start[g], m = a.group_start[g + 1] - g0;
  const int k = (int)floor(a.frac * (double)m);
  // rank of d inside its group: the learners that rank before it
  const double kd = pbt_key(a.score[d]);
  int c = 0;
  for (int i = g0 + tid; i < g0 + m; i += EXPLOIT_THREADS) c += pbt_before(pbt_key(a.score[i]), i, kd, d);
  const int rank = block_sum(c, red);
  if (k == 0 || rank < m - k) {   // kept
    if (blockIdx.x == 0 && tid == 0 && a.parent) a.parent[d] = -1;
    return;
  }
  uint32_t w[4];
  philox4x32_10(a.seed, (uint64_t)d, a.round, STREAM_PBT, w);
  const int r_src = (int)(uint32_t)(((uint64_t)w[0] * (uint64_t)k) >> 32);
  // the source is the group's learner of rank r_src: every thread ranks its candidates (ranks are a permutation: one thread finds it)
  for (int j = g0 + tid; j < g0 + m; j += EXPLOIT_THREADS) {
    const double kj = pbt_key(a.score[j]);
    int rj = 0;
    for (int i = g0; i < g0 + m && rj <= r_src; ++i) rj += pbt_before(pbt_key(a.score[i]), i, kj, j);
    if (rj == r_src) s_src = j;
  }
  __syncthreads();
  const int src = s_src;
  if (blockIdx.x == 0 && tid == 0) {   // optimiser β powers and their reciprocals, perturbed hyper-parameters, lineage
    const DdpgCtrl& cs = a.ctrl[src];
    DdpgCtrl& cd = a.ctrl[d];
#pragma unroll
    for (int n = 0; n < 2; ++n)
#pragma unroll
      for (int b = 0; b < 2; ++b) { cd.bp[n][b] = cs.bp[n][b]; cd.rc[n][b] = cs.rc[n][b]; }
    const DdpgHparams hs = cs.hp;
    DdpgHparams hd;   // bits of keys in Learner.HPARAMS order: 0 lr_actor (eta[1]), 1 lr_critic (eta[0]), 2 gamma, 3 tau, 4 noise_scale
    hd.eta[1] = pbt_perturb(hs.eta[1], 0, a.keys, w[1], a.factor_lo, a.factor_hi);
    hd.eta[0] = pbt_perturb(hs.eta[0], 1, a.keys, w[1], a.factor_lo, a.factor_hi);
    hd.gamma = pbt_perturb(hs.gamma, 2, a.keys, w[1], a.factor_lo, a.factor_hi);
    hd.tau = pbt_perturb(hs.tau, 3, a.keys, w[1], a.factor_lo, a.factor_hi);
    hd.noise_scale = pbt_perturb(hs.noise_scale, 4, a.keys, w[1], a.factor_lo, a.factor_hi);
    cd.hp = hd;
    if (a.parent) a.parent[d] = src;
  }
  // this block's chunk of the concatenated parts: every part starts on a 256-byte boundary of the slab and its float4 count covers
  // the part (the tail float4 stays inside the part's 64-float carve), so the copy is float4 only
  const float4* __restrict__ from = reinterpret_cast<const float4*>(a.slab + (long long)src * a.pop_stride);
  float4* __restrict__ to = reinterpret_cast<float4*>(a.slab + (long long)d * a.pop_stride);
  const long long c0 = (long long)blockIdx.x * EXPLOIT_CHUNK, c1 = c0 + EXPLOIT_CHUNK;
  long long p0 = 0;
#pragma unroll 1
  for (int p = 0; p < EXPLOIT_PARTS; ++p) {
    const long long p1 = p0 + a.part_n4[p], lo = max(c0, p0), hi = min(c1, p1);
    if (lo < hi) {
      const float4* s = from + a.part_off[p] + (lo - p0);
      float4* t = to + a.part_off[p] + (lo - p0);
      const long long n = hi - lo;
      float4 v[EXPLOIT_UNROLL];
#pragma unroll
      for (int u = 0; u < EXPLOIT_UNROLL; ++u) {
        const long long i = tid + (long long)u * EXPLOIT_THREADS;
        if (i < n) v[u] = __ldg(s + i);
      }
#pragma unroll
      for (int u = 0; u < EXPLOIT_UNROLL; ++u) {
        const long long i = tid + (long long)u * EXPLOIT_THREADS;
        if (i < n) t[i] = v[u];
      }
    }
    p0 = p1;
  }
}

extern "C" int32_t ddpg_exploit(Ddpg* h, const double* score_dev, const DdpgExploitParams* p, int32_t* parent_dev) {
  REQUIRE(h && score_dev && p, SHEMS_ERR_INVALID, "ddpg_exploit: NULL argument");
  REQUIRE(p->frac >= 0.0 && p->frac <= 0.5, SHEMS_ERR_INVALID, "ddpg_exploit: frac=%g outside [0, 0.5]", p->frac);
  REQUIRE(isfinite(p->factor_lo) && isfinite(p->factor_hi) && p->factor_lo > 0.0f && p->factor_hi > 0.0f, SHEMS_ERR_INVALID,
          "ddpg_exploit: factors %g, %g must be finite and > 0", (double)p->factor_lo, (double)p->factor_hi);
  REQUIRE(p->keys >= 0 && p->keys <= 31, SHEMS_ERR_INVALID, "ddpg_exploit: keys=%d outside 0..31", p->keys);
  REQUIRE(p->n_groups >= 0 && p->n_groups <= DDPG_EXPLOIT_MAX_GROUPS, SHEMS_ERR_INVALID, "ddpg_exploit: n_groups=%d outside 0..%d", p->n_groups,
          DDPG_EXPLOIT_MAX_GROUPS);
  ExploitArgs a;
  memset(&a, 0, sizeof(a));
  if (p->n_groups == 0) {
    a.n_groups = 1; a.group_start[0] = 0; a.group_start[1] = h->pop;
  } else {
    REQUIRE(p->group_start[0] == 0 && p->group_start[p->n_groups] == h->pop, SHEMS_ERR_INVALID,
            "ddpg_exploit: group starts must begin at 0 and end at P = %d (%d .. %d)", h->pop, p->group_start[0], p->group_start[p->n_groups]);
    for (int g = 0; g < p->n_groups; ++g)
      REQUIRE(p->group_start[g] < p->group_start[g + 1], SHEMS_ERR_INVALID, "ddpg_exploit: group starts do not increase at group %d (%d, %d)", g,
              p->group_start[g], p->group_start[g + 1]);
    a.n_groups = p->n_groups;
    for (int g = 0; g <= p->n_groups; ++g) a.group_start[g] = p->group_start[g];
  }
  GUARD(h->device);
  // what ddpg_get_state / ddpg_set_state move: the four nets, the four ADAM moment arrays, s_min | s_max
  const long long na = h->dims[0].n_params, nc = h->dims[1].n_params;
  float* const parts[EXPLOIT_PARTS] = {h->net[0], h->net[1], h->net[2], h->net[3], h->adam_m[0], h->adam_v[0], h->adam_m[1], h->adam_v[1], h->norm};
  const long long counts[EXPLOIT_PARTS] = {na, nc, na, nc, na, na, nc, nc, 18};
  long long total = 0;
  for (int i = 0; i < EXPLOIT_PARTS; ++i) {
    a.part_off[i] = (parts[i] - h->slab) / 4;   // every part starts on a 256-byte boundary
    a.part_n4[i] = (counts[i] + 3) / 4;
    total += a.part_n4[i];
  }
  a.score = score_dev; a.slab = h->slab; a.pop_stride = h->pop_stride; a.ctrl = h->ctrl; a.parent = parent_dev;
  a.frac = p->frac; a.factor_lo = p->factor_lo; a.factor_hi = p->factor_hi; a.keys = p->keys; a.round = p->round; a.seed = p->seed;
  const dim3 grid((unsigned)((total + EXPLOIT_CHUNK - 1) / EXPLOIT_CHUNK), (unsigned)h->pop);
  ddpg_exploit_kernel<<<grid, EXPLOIT_THREADS, 0, h->stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  h->hp_stale = true;
  return SHEMS_OK;
}

extern "C" int32_t ddpg_grad_buffer(Ddpg* h, float** grad_dev, int64_t* n) {
  REQUIRE(h && grad_dev && n, SHEMS_ERR_INVALID, "ddpg_grad_buffer: NULL argument");
  *grad_dev = h->gradbuf;
  *n = (h->grad[0] - h->gradbuf) + h->dims[0].n_params;
  return SHEMS_OK;
}

// ----------------------------------------------------------------------------- full learner snapshot (resume)
// What the reference never saves (saveBSON writes the actor and the score arrays only, memory_plotting_saving.jl:263-270, so a
// run cannot be resumed): the four nets, both optimisers' moments and β powers, the update counter and the normalisation
// constants of the selected learner.  Layout of state_host (floats):
//   [actor | critic | actor_target | critic_target | m_actor | v_actor | m_critic | v_critic | s_min (9) | s_max (9)]
// opt_host (doubles): [βp_critic[0], βp_critic[1], βp_actor[0], βp_actor[1], number of updates, 0, 0, 0]
extern "C" int64_t ddpg_state_floats(const Ddpg* h) {
  if (!h) return 0;
  return 4 * h->dims[0].n_params + 4 * h->dims[1].n_params + 18;
}
static int state_copy(Ddpg* h, float* host, bool to_host) {
  const long long na = h->dims[0].n_params, nc = h->dims[1].n_params, lo = sel_off(h);
  float* const parts[9] = {h->net[0], h->net[1], h->net[2], h->net[3], h->adam_m[0], h->adam_v[0], h->adam_m[1], h->adam_v[1], h->norm};
  const long long counts[9] = {na, nc, na, nc, na, na, nc, nc, 18};
  long long off = 0;
  for (int i = 0; i < 9; ++i) {
    if (to_host) CUDA_TRY(cudaMemcpy(host + off, parts[i] + lo, sizeof(float) * (size_t)counts[i], cudaMemcpyDeviceToHost));
    else CUDA_TRY(cudaMemcpy(parts[i] + lo, host + off, sizeof(float) * (size_t)counts[i], cudaMemcpyHostToDevice));
    off += counts[i];
  }
  return SHEMS_OK;
}
extern "C" int32_t ddpg_get_state(Ddpg* h, float* state_host, double* opt_host) {
  REQUIRE(h && state_host && opt_host, SHEMS_ERR_INVALID, "ddpg_get_state: NULL argument");
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  TRY(state_copy(h, state_host, true));
  DdpgCtrl c;
  CUDA_TRY(cudaMemcpy(&c, h->ctrl + h->sel, sizeof(c), cudaMemcpyDeviceToHost));
  opt_host[0] = c.bp[0][0]; opt_host[1] = c.bp[0][1]; opt_host[2] = c.bp[1][0]; opt_host[3] = c.bp[1][1];
  opt_host[4] = (double)h->n_updates; opt_host[5] = opt_host[6] = opt_host[7] = 0.0;
  return SHEMS_OK;
}
extern "C" int32_t ddpg_set_state(Ddpg* h, const float* state_host, const double* opt_host) {
  REQUIRE(h && state_host && opt_host, SHEMS_ERR_INVALID, "ddpg_set_state: NULL argument");
  for (int i = 0; i < 4; ++i)
    REQUIRE(opt_host[i] > 0.0 && opt_host[i] < 1.0, SHEMS_ERR_INVALID, "ddpg_set_state: beta power %d = %g outside (0, 1)", i, opt_host[i]);
  REQUIRE(opt_host[4] >= 0.0, SHEMS_ERR_INVALID, "ddpg_set_state: update counter %g", opt_host[4]);
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  TRY(state_copy(h, const_cast<float*>(state_host), false));
  TRY(write_opt_state(h, h->sel, opt_host[0], opt_host[1], opt_host[2], opt_host[3]));
  h->n_updates = (long long)opt_host[4];   // one counter per handle (the learners of a population advance together)
  return SHEMS_OK;
}
// OUNoise.X of ddpg_episode's instances ([2][n], input.jl:234; never reset by the reference): n_out receives the instance count
// (0 before the first OU episode); x_host may be NULL to query it.  ddpg_set_ou_state (re)allocates for n instances.
extern "C" int32_t ddpg_get_ou_state(Ddpg* h, float* x_host, int64_t* n_out) {
  REQUIRE(h && n_out, SHEMS_ERR_INVALID, "ddpg_get_ou_state: NULL argument");
  GUARD(h->device);
  *n_out = h->ou_cap;
  if (x_host && h->ou_cap > 0) {
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaMemcpy(x_host, h->ou_x, sizeof(float) * 2 * (size_t)h->ou_cap, cudaMemcpyDeviceToHost));
  }
  return SHEMS_OK;
}
extern "C" int32_t ddpg_set_ou_state(Ddpg* h, const float* x_host, int64_t n) {
  REQUIRE(h && x_host && n >= 1, SHEMS_ERR_INVALID, "ddpg_set_ou_state: NULL argument or n=%lld", (long long)n);
  GUARD(h->device);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (h->ou_cap != n) {
    cudaFree(h->ou_x); h->ou_x = nullptr; h->ou_cap = 0;
    CUDA_TRY(cudaMalloc(&h->ou_x, sizeof(float) * 2 * (size_t)n));
    h->ou_cap = n;
  }
  CUDA_TRY(cudaMemcpy(h->ou_x, x_host, sizeof(float) * 2 * (size_t)n, cudaMemcpyHostToDevice));
  return SHEMS_OK;
}
