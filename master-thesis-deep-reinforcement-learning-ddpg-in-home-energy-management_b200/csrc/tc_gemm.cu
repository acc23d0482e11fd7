// tc_gemm.cu — TF32 tensor-core GEMM for the large-batch DDPG update (B >= 1024): sm_100a tcgen05 + TMEM + TMA.
//
//   D[M×N] = epilogue( A · B^T-or-B ),  fp32 in HBM, TF32 multiply, fp32 accumulate in TMEM.
//
// Each operand is described the way it already sits in HBM (no transposed copies):
//   K-major  : element (row, k) at  ptr[row*ld + k]   (k contiguous)   — activations as the M operand of forward / dX
//   MN-major : element (row, k) at  ptr[k*ld + row]   (row contiguous) — Flux weights Wt[in][out] as the N operand of the
//              forward pass, and both operands of dW = X^T · dZ
// Persistent CTAs (one per SM) work through 128×128 output tiles (optionally K-splits of them).  Warp roles (192 threads):
//   warp 0   : TMA producer — cp.async.bulk.tensor into a 5-stage ring of 128B-swizzled tiles (running across tile boundaries), mbarrier expect_tx
//   warp 1   : TMEM allocator + MMA issuer — one elected lane issues 4 tcgen05.mma.kind::tf32 (K = 8 each) per 32-wide
//              k-block, tcgen05.commit releases the smem stage / signals the epilogue
//   warps 2-5: epilogue — tcgen05.ld (32 lanes × 32 columns per instruction) TMEM -> registers -> fused epilogue -> HBM
// Descriptor encodings follow cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor) of CUTLASS 3.9.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "common.h"
#include "tc_gemm.h"

namespace {

struct TcMaps { CUtensorMap a[TC_MAX_PROBLEMS], b[TC_MAX_PROBLEMS], d[TC_MAX_PROBLEMS]; };

constexpr int BLOCK_M = 128, BLOCK_N = 128, BLOCK_K = 32, UMMA_K = 8;
constexpr int STAGES = 5;                                    // 5 x 32 KB operand ring: one persistent CTA per SM keeps it full across tiles
constexpr int TILE_BYTES = BLOCK_M * BLOCK_K * 4;            // 16 KB per operand and stage
constexpr int STAGING_BYTES = 4 * 2 * 4096;                  // epilogue: 4 warps x 2 chunk buffers of 32x32 fp32
constexpr int SMEM_BYTES = STAGES * 2 * TILE_BYTES + STAGING_BYTES + 1024;   // + alignment slack
constexpr int ACC_STAGES = 2;                                // double-buffered accumulator: epilogue of tile i overlaps the k-loop of tile i+1
constexpr int TMEM_COLS = ACC_STAGES * BLOCK_N;              // 256 fp32 columns

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// operand tile load; the third coordinate is the batch entry (a learner of a population), 0 otherwise
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
                   smem_u32(smem_dst)),
               "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// smem -> global tile store (3-D map {N, M, splits}); completion is tracked by the bulk async-group of the issuing thread
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];\n" ::"l"(tm), "r"(smem_u32(smem_src)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "elect.sync _|P1, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, P1;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// SmemDescriptor (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
// layout_type [61,64): SWIZZLE_128B = 2 (K-major tiles), SWIZZLE_128B_BASE32B = 1 (the only layout for MN-major tf32)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

// Persistent, warp-specialised GEMM: grid = min(#tiles, #SMs) CTAs of 192 threads, CTA c works on tiles c, c + grid, ...
// (tile = (m-tile, n-tile, z) with z the K-split or the batch entry).  The three roles run the same tile sequence but are coupled
// only through mbarriers, so the TMA producer streams the operands of tile i+1 while the MMA lane still issues tile i and the
// epilogue warps drain tile i-1 from the other half of TMEM:
//   warp 0   : TMA producer          full[s] / empty[s]          5-stage operand ring, running across tile boundaries
//   warp 1   : tcgen05.mma issuer    acc_full[a] / acc_empty[a]  two 128-column accumulators in TMEM
//   warps 2-5: epilogue              tcgen05.ld -> fused epilogue -> swizzled smem chunk (double-buffered) -> bulk tensor store
template <bool A_MN, bool B_MN>
__global__ void __launch_bounds__(192, 1)
tc_gemm_kernel(const __grid_constant__ TcMaps maps, const TcGemmArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);  // SW128 needs 1024 B
  uint8_t* staging = smem + STAGES * 2 * TILE_BYTES;
  __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], acc_full_bar[ACC_STAGES], acc_empty_bar[ACC_STAGES];
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float bias_s[2][BLOCK_N];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mt = (p.M + BLOCK_M - 1) / BLOCK_M, nt = (p.N + BLOCK_N - 1) / BLOCK_N;
  const int nz = p.batch > 1 ? p.batch : p.splits;
  const int total_tiles = mt * nt * nz * p.nprob;  // several same-shape problems (own tensor maps / pointers) share one launch
  const int kb_total = (p.K + BLOCK_K - 1) / BLOCK_K;
  const int kb_per = (kb_total + p.splits - 1) / p.splits;
  // programmatic dependent launch (when the host asks for it): a successor may be scheduled while this grid runs, and this grid's own
  // set-up (barriers, TMEM, tensor maps) runs under the tail of its predecessor; nothing the predecessor wrote is touched before the wait
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(&acc_full_bar[a], 1); mbar_init(&acc_empty_bar[a], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    for (int q = 0; q < p.nprob; ++q) {
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.a[q]) : "memory");
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.b[q]) : "memory");
      if (p.tma_store) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.d[q]) : "memory");
    }
  }
  if (warp == 1) {  // TMEM allocation: 2 x 128 fp32 accumulator columns × 128 lanes
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_smem)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;
  asm volatile("griddepcontrol.wait;\n" ::: "memory");

// tile -> (m0, n0, split, bz, first k-block, number of k-blocks); m-tiles vary fastest so that concurrently running CTAs share B tiles in L2
#define TILE_COORDS(tile)                                                               \
  const int prob = (tile) / (mt * nt * nz), t_ = (tile) - prob * (mt * nt * nz);        \
  const int z_ = t_ / (mt * nt), r_ = t_ - z_ * (mt * nt);                              \
  const int m0 = (r_ % mt) * BLOCK_M, n0 = (r_ / mt) * BLOCK_N;                         \
  const int split = p.batch > 1 ? 0 : z_, bz = p.batch > 1 ? z_ : 0;                    \
  const int kb_begin = split * kb_per;                                                  \
  const int num_kb = max(0, min(kb_total, kb_begin + kb_per) - kb_begin);

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      int g = 0;  // k-blocks issued so far (ring position carries over tile boundaries)
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        TILE_COORDS(tile)
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int s = g % STAGES, ph = (g / STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          mbar_expect_tx(&full_bar[s], 2 * TILE_BYTES);
          uint8_t* sa = smem + s * 2 * TILE_BYTES;
          uint8_t* sb = sa + TILE_BYTES;
          const int k0 = (kb_begin + i) * BLOCK_K;
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < 4; ++j) tma_load_3d(sa + j * 4096, &maps.a[prob], &full_bar[s], m0 + j * 32, k0, bz);  // box {32 rows(MN), 32 k}
          } else {
            tma_load_3d(sa, &maps.a[prob], &full_bar[s], k0, m0, bz);                                               // box {32 k, 128 rows}
          }
          if (B_MN) {
#pragma unroll
            for (int j = 0; j < 4; ++j) tma_load_3d(sb + j * 4096, &maps.b[prob], &full_bar[s], n0 + j * 32, k0, bz);
          } else {
            tma_load_3d(sb, &maps.b[prob], &full_bar[s], k0, n0, bz);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // InstrDescriptor: c_format F32 (1) [4,6), a/b_format TF32 (2) [7,10)/[10,13), a_major [15], b_major [16], N>>3 [17,23), M>>4 [24,29)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                           ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
    if (elect_one()) {
      int g = 0, it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        TILE_COORDS(tile)
        (void)m0; (void)n0; (void)bz; (void)prob;
        const int acc = it & 1, use = it >> 1;
        mbar_wait(&acc_empty_bar[acc], (use & 1) ^ 1);  // the epilogue has drained this accumulator (passes at once on first use)
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int s = g % STAGES, ph = (g / STAGES) & 1;
          mbar_wait(&full_bar[s], ph);
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          const uint32_t sa = smem_u32(smem + s * 2 * TILE_BYTES), sb = sa + TILE_BYTES;
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            // K-major, SWIZZLE_128B: rows of 128 B (32 k), 8-row groups 1024 B apart (SBO); one UMMA_K = 32 B further along the row.
            // MN-major, SWIZZLE_128B_BASE32B: k-rows of 128 B (32 MN elements); the swizzle atom is 4 k-rows (512 B, 32-byte
            //   chunks XOR row%4), so one UMMA_K = 8 spans two atoms 512 B apart (SBO); 32-wide MN chunks are 4096 B apart (LBO).
            const uint64_t ad = A_MN ? make_smem_desc(sa + kk * 1024, 4096, 512, 1) : make_smem_desc(sa + kk * 32, 16, 1024, 2);
            const uint64_t bd = B_MN ? make_smem_desc(sb + kk * 1024, 4096, 512, 1) : make_smem_desc(sb + kk * 32, 16, 1024, 2);
            umma_tf32(tmem_d, ad, bd, idesc, (i | kk) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);  // frees the smem stage once the MMAs above have read it
        }
        umma_commit(&acc_full_bar[acc]);   // accumulator complete (arrives at once for an empty k-range)
      }
    }
  } else {
    // ===== epilogue (warps 2-5): TMEM lane quarter = warp % 4 =====
    // A thread owns one accumulator row; tcgen05.ld hands it 32 consecutive columns at a time.  With a TMA-storable D
    // (16-byte rows) the warp writes its 32x32 chunk into 128B-swizzled shared memory and one lane issues a bulk tensor
    // store: full 128-byte lines, clipped at M / N by the tensor map.  Otherwise every thread stores its row segment directly.
    const int q = warp & 3;
    const bool mask = (p.epi == TC_EPI_RELU_MASK);
    const bool aux_vec = mask && ((p.auxld & 3) == 0) && ((p.bs_aux & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.aux[0]) & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.aux[1]) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(p.aux[2]) & 15) == 0);
    uint8_t* stage = staging + q * (2 * 4096);  // this warp's two 32x32 fp32 chunk buffers (4 KB each, 1024-byte aligned)
    int it = 0, chunk_no = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      TILE_COORDS(tile)
      const int acc = it & 1, use = it >> 1;
      const int m = m0 + q * 32 + lane;
      // this tile's bias slice (double-buffered: the named barrier of tile it+1 proves everyone is done with tile it-1's slice)
      bias_s[it & 1][threadIdx.x - 64] = (p.epi == TC_EPI_BIAS_RELU && n0 + (int)threadIdx.x - 64 < p.N) ? p.bias[prob][(long long)bz * p.bs_bias + n0 + threadIdx.x - 64] : 0.0f;
      asm volatile("bar.sync 1, 128;\n" ::: "memory");
      const float* auxrow = mask ? p.aux[prob] + (long long)bz * p.bs_aux + (long long)min(m, p.M - 1) * p.auxld : nullptr;
      if (num_kb > 0) {
        mbar_wait(&acc_full_bar[acc], use & 1);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
      }
      float* Dp = p.D[prob] + (long long)(split + bz) * p.split_stride;  // split_stride doubles as the batch stride of D
#pragma unroll 1
      for (int c = 0; c < BLOCK_N / 32; ++c) {
        const int nc = n0 + c * 32;
        if (nc >= p.N) break;
        float4 hx[8];
        if (mask) {  // relu'(H): this row's 32 mask values, requested before the accumulator is read
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const int n = nc + j4 * 4;
            if (aux_vec && n + 3 < p.N) hx[j4] = *reinterpret_cast<const float4*>(auxrow + n);
            else {
              hx[j4].x = (n + 0 < p.N) ? auxrow[n + 0] : 0.0f; hx[j4].y = (n + 1 < p.N) ? auxrow[n + 1] : 0.0f;
              hx[j4].z = (n + 2 < p.N) ? auxrow[n + 2] : 0.0f; hx[j4].w = (n + 3 < p.N) ? auxrow[n + 3] : 0.0f;
            }
          }
        }
        uint32_t v[32];
        if (num_kb > 0) tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BLOCK_N + c * 32), v);
        else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        float4 o[8];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          float x[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) x[u] = __uint_as_float(v[j4 * 4 + u]);
          if (p.epi == TC_EPI_BIAS_RELU) {
            const float4 bv = *reinterpret_cast<const float4*>(&bias_s[it & 1][c * 32 + j4 * 4]);
            x[0] = fmaxf(x[0] + bv.x, 0.0f); x[1] = fmaxf(x[1] + bv.y, 0.0f); x[2] = fmaxf(x[2] + bv.z, 0.0f); x[3] = fmaxf(x[3] + bv.w, 0.0f);
          } else if (mask) {
            x[0] = hx[j4].x > 0.0f ? x[0] : 0.0f; x[1] = hx[j4].y > 0.0f ? x[1] : 0.0f;
            x[2] = hx[j4].z > 0.0f ? x[2] : 0.0f; x[3] = hx[j4].w > 0.0f ? x[3] : 0.0f;
          }
          o[j4] = make_float4(x[0], x[1], x[2], x[3]);
        }
        if (p.tma_store) {
          uint8_t* buf = stage + (chunk_no & 1) * 4096;
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");  // the store issued two chunks ago has read this buffer
          __syncwarp();
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)  // SWIZZLE_128B: 16-byte chunk j of row r sits at chunk j ^ (r & 7)
            *reinterpret_cast<float4*>(buf + lane * 128 + ((j4 ^ (lane & 7)) << 4)) = o[j4];
          asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&maps.d[prob], buf, nc, m0 + q * 32, split + bz);
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
          }
          ++chunk_no;
        } else if (m < p.M) {
          const bool vec = ((p.ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(Dp) & 15) == 0);
          float* drow = Dp + (long long)m * p.ldd;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const int n = nc + j4 * 4;
            if (vec && n + 3 < p.N) *reinterpret_cast<float4*>(drow + n) = o[j4];
            else {
              const float x[4] = {o[j4].x, o[j4].y, o[j4].z, o[j4].w};
#pragma unroll
              for (int u = 0; u < 4; ++u) if (n + u < p.N) drow[n + u] = x[u];
            }
          }
        }
      }
      // every tcgen05.ld of this accumulator has completed (wait::ld): hand it back to the MMA issuer
      asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty_bar[acc]);
    }
    if (p.tma_store && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");  // smem must outlive the reads
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  }
#undef TILE_COORDS
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}


// ---------------------------------------------------------------------------------------------------------------- forward chain
// One net's WHOLE forward pass for a 128-row tile of a large minibatch in one CTA (large-batch replay(), DDPG.jl:131-132, :114, :117):
//   h1 = relu(x W1 + b1)        fp32 SIMT by 8 producer warps (thread = 4 rows x 4 columns of a k-block, the rows' inputs held in
//                               registers for the whole kernel, W1 and b1 in shared memory), written k-block by k-block straight into a
//                               3-deep ring of 128B-swizzled K-major A-operand blocks in shared memory; when the backward pass needs h1
//                               the finished k-blocks are sent to HBM by TMA stores FROM the operand
//   h2 = relu(h1 W2 + b2)       tcgen05.mma kind::tf32, 128 x 256 x 8 per instruction; BOTH 256-column halves accumulate in TMEM at once
//                               (all 512 columns), so the tile makes ONE pass over k: W2 is streamed by TMA (MN-major, as Flux stores it)
//                               through a 4-stage ring of [16 k][512 columns] slabs = 128 KB in flight per SM.  (The first version kept the
//                               whole A operand resident — 128 KB — and walked k once per half behind a 48 KB ring: 48 KB / L2 latency =
//                               40 GB/s per SM, 19.4 us per tile.)
//   out = f(h2 W3 + b3)         in the epilogue (8 warps: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4): bias + ReLU, h2 to HBM
//                               by TMA stores staged in the then idle W2 ring (4 chunks in flight per warp), and the output layer's dot
//                               product (1 or 2 units) in registers, the two halves' partial sums joined through shared memory;
//                               f = tanh (actor -> written into the critic's input rows), identity (q), or the TD target
//                               y = r + gamma (1 - done) q' with dq = 2 (q - y) / B (DDPG.jl:133)
// Replaces l1_fwd_kernel + tc_gemm_kernel + gemm_skinny_kernel (3 launches and two round trips of the activations through HBM per net).
// Warp roles (320 threads): warp 0 TMA producer, warp 1 TMEM allocation + MMA issue (+ the h1 stores), warps 2-9 layer-1 producers, then
// the epilogue.
constexpr int FC_THREADS = 320, FC_N = 256, FC_KB = 8, FC_ASTAGES = 3, FC_BSTAGES = 4, FC_BK = 16;
constexpr int FC_A_BYTES = FC_ASTAGES * TILE_BYTES;            // 3 k-blocks x 16 KB
constexpr int FC_B_STAGE = 2 * FC_N * FC_BK * 4;               // 32 KB: 16 chunks of [16 k][32 columns], column half h at h * 16 KB
constexpr int FC_SMEM = FC_A_BYTES + FC_BSTAGES * FC_B_STAGE + 1024;
static_assert(FC_BSTAGES * FC_B_STAGE >= 8 * 4 * 4096, "the epilogue stages 4 chunks per warp in the W2 ring");

// -DFC_TRACE: globaltimer stamps of CTA 0 (tools/time_ddpg_large.py with a *fctrace* build): [0..15] TMA slab issued, [32..47] MMA slab
// committed, [64..71] layer-1 k-block written (warp 2), [72] start, [73] accumulators seen, [74] warp 2's chunks done, [76] end
#ifdef FC_TRACE
__device__ unsigned long long fc_trace[96];
#define FC_STAMP(i) do { if (blockIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t_)); fc_trace[i] = t_; } } while (0)
#else
#define FC_STAMP(i) do { } while (0)
#endif
// NS = 2: a cluster of two CTAs per row tile, each with 256 of the layer-2 units (half of the W2 stream; layer 1 is computed by both, h1
// stored by the first); the second CTA hands its share of the output layer's dot products to the first through distributed shared
// memory.  For launches whose row tiles alone would leave more than half of the SMs idle.
template <int NS>
__global__ void __launch_bounds__(FC_THREADS, 1)
tc_fwd_chain_kernel(const __grid_constant__ TcMaps maps, const TcFwdChainArgs p) {
  constexpr int NCOL = 2 * FC_N / NS;                          // layer-2 units (accumulator columns) of this CTA
  constexpr int HN = NCOL / FC_N;                              // 256-column MMA halves of this CTA
  constexpr int BST = FC_BSTAGES * NS, BSTAGE = FC_B_STAGE / NS;   // the W2 ring: the same 128 KB, in slabs of [16 k][NCOL columns]
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + FC_A_BYTES;
  __shared__ uint64_t a_full[FC_ASTAGES], a_empty[FC_ASTAGES], b_full[BST], b_empty[BST], acc_full;
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float w1s[12][FC_KB * BLOCK_K];   // rows 0..K1-1: W1 (zero beyond l1), rows K1..10: zero, row 11: b1 (its input is 1)
  __shared__ __align__(16) float b2s[2 * FC_N];
  __shared__ __align__(16) float w3s[2][2 * FC_N];            // W3[:, j] (zero beyond l2)
  __shared__ float dpart[2][BLOCK_M];                         // the upper column half's share of the output layer's dot products
  __shared__ float xpart[2][BLOCK_M];                         // NS = 2: the second CTA's share, written by it through DSMEM
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mt = (p.M + BLOCK_M - 1) / BLOCK_M;
  const int bx = blockIdx.x / NS, nh = blockIdx.x % NS;        // nh: which half of the layer-2 units (= the rank in the cluster of two)
  const int prob = bx / mt, m0 = (bx - prob * mt) * BLOCK_M;
  const int K1 = p.K1[prob], J = p.J[prob];
  const int learner = blockIdx.y;                              // a population: the learner's slab starts lo floats further, TMA coordinate 2
  const long long lo = (long long)learner * p.pop_stride;
  // γ of the TD target: requested now, used in the epilogue (loaded there, its latency would add to the kernel's tail)
  const float td_gamma = p.out_mode[prob] == TC_OUT_TD ? p.td_gamma[learner * p.td_gamma_stride] : 0.0f;
  const int nkb = (p.L1 + BLOCK_K - 1) / BLOCK_K, nslab = (p.L1 + FC_BK - 1) / FC_BK;   // k-blocks of 32 / W2 slabs of 16 that hold real units
  if (warp == 2 && lane == 0) FC_STAMP(72);
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");   // see tc_gemm_kernel
  // Programmatic dependent launch: what did the predecessor in the stream write?  Normally only the rows' inputs (early_weights): the
  // weights are staged under its tail, then the wait, then the inputs.  After an optimiser step the weights are its output: wait first
  // (then the inputs are requested before the staging so that they arrive under it).
  float x[4][12];   // layer-1 producers: the inputs of rows {lane, lane+32, lane+64, lane+96}
#define FC_LOAD_X()                                                                                                                       \
  if (warp >= 2) {                                                                                                                        \
    _Pragma("unroll") for (int rr = 0; rr < 4; ++rr) {                                                                                    \
      const int row = m0 + lane + 32 * rr;                                                                                                \
      _Pragma("unroll") for (int i = 0; i < 11; ++i)                                                                                      \
        x[rr][i] = (row < p.M && i < K1) ? __ldg(p.X[prob] + lo + (long long)row * p.ldx + i) : 0.0f;                                     \
      x[rr][11] = 1.0f; /* the bias row of w1s: fma(1, b, sum) == sum + b */                                                              \
    }                                                                                                                                     \
  }
  if (!p.early_weights) {
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    FC_LOAD_X();
  }
  for (int e = threadIdx.x; e < 12 * FC_KB * BLOCK_K; e += FC_THREADS) {
    const int i = e / (FC_KB * BLOCK_K), n = e - i * (FC_KB * BLOCK_K);
    float v = 0.0f;
    if (n < p.L1) v = i < K1 ? __ldg(p.W1[prob] + lo + (long long)i * p.L1 + n) : (i == 11 ? __ldg(p.b1[prob] + lo + n) : 0.0f);
    w1s[i][n] = v;
  }
  for (int n = threadIdx.x; n < 2 * FC_N; n += FC_THREADS) {
    const bool ok = n < p.L2;
    b2s[n] = ok ? __ldg(p.b2[prob] + lo + n) : 0.0f;
    w3s[0][n] = ok ? __ldg(p.W3[prob] + lo + (long long)n * J) : 0.0f;
    w3s[1][n] = (ok && J == 2) ? __ldg(p.W3[prob] + lo + (long long)n * J + 1) : 0.0f;
  }
  if (p.early_weights) {
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
    FC_LOAD_X();
  }
#undef FC_LOAD_X
  if (threadIdx.x == 0) {
    for (int k = 0; k < FC_ASTAGES; ++k) { mbar_init(&a_full[k], 8); mbar_init(&a_empty[k], 1); }   // a_full: one arrival per producer warp
    for (int s = 0; s < BST; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    mbar_init(&acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.b[prob]) : "memory");
    if (p.H1[prob] && nh == 0) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.a[prob]) : "memory");
    if (p.H2[prob]) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.d[prob]) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOL));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;
  const int q = warp & 3, erow = m0 + q * 32 + lane;          // epilogue: TMEM lane quarter and row of this thread
  float d0 = 0.0f, d1 = 0.0f;                                  // its share of the output layer's dot products
  bool fin = false;                                            // this thread finishes a row (warps 2-5)

  if (warp == 0) {
    // ===== TMA producer: W2[16-k slab][all columns] as the MN-major B operand, 16 boxes of {32 columns, 16 k} per slab =====
    if (elect_one()) {
      for (int g = 0; g < nslab; ++g) {
        const int s = g % BST, ph = (g / BST) & 1;
        mbar_wait(&b_empty[s], ph ^ 1);
        FC_STAMP(g);
        mbar_expect_tx(&b_full[s], BSTAGE);
        uint8_t* sb = sB + s * BSTAGE;
#pragma unroll
        for (int j = 0; j < NCOL / 32; ++j) tma_load_3d(sb + j * (FC_BK * 128), &maps.b[prob], &b_full[s], nh * NCOL + j * 32, g * FC_BK, learner);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (1u << 16) | ((uint32_t)(FC_N >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
    if (elect_one()) {
      const bool store_h1 = p.H1[prob] != nullptr && nh == 0;
      for (int g = 0; g < nslab; ++g) {
        const int kb = g >> 1, sa_i = kb % FC_ASTAGES, s = g % BST, ph = (g / BST) & 1;
        if ((g & 1) == 0) {
          mbar_wait(&a_full[sa_i], (kb / FC_ASTAGES) & 1);   // layer-1 producers have written (and fenced) this k-block of the A operand
          if (store_h1 && kb * BLOCK_K < p.ldh1) {          // ... which is also h1[m0 .. m0+127][kb*32 .. +31]: send it to HBM as it lies
            tma_store_3d(&maps.a[prob], sA + sa_i * TILE_BYTES, kb * BLOCK_K, m0, learner);
            asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
          }
        }
        mbar_wait(&b_full[s], ph);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const uint32_t sa = smem_u32(sA + sa_i * TILE_BYTES) + (uint32_t)((g & 1) * (FC_BK / UMMA_K) * 32), sb = smem_u32(sB + s * BSTAGE);
#pragma unroll
        for (int h = 0; h < HN; ++h) {
#pragma unroll
          for (int kk = 0; kk < FC_BK / UMMA_K; ++kk) {
            const uint64_t ad = make_smem_desc(sa + kk * 32, 16, 1024, 2);                                  // K-major, SWIZZLE_128B
            const uint64_t bd = make_smem_desc(sb + h * (FC_N * FC_BK * 4) + kk * 1024, FC_BK * 128, 512, 1);   // MN-major, SWIZZLE_128B_BASE32B: 32-column chunks 2 KB apart
            umma_tf32(tmem_base + (uint32_t)(h * FC_N), ad, bd, idesc, (g | kk) != 0 ? 1u : 0u);
          }
        }
        umma_commit(&b_empty[s]);
        FC_STAMP(32 + g);
        if ((g & 1) == 1 || g == nslab - 1) {   // last slab of this k-block: its ring slot is free once these MMAs (and the h1 store's read) are done
          if (store_h1) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
          umma_commit(&a_empty[sa_i]);
        }
      }
      umma_commit(&acc_full);
    }
  } else {
    // ===== layer-1 producers (warps 2-9): thread = rows {lane, lane+32, lane+64, lane+96} x 4 columns (cg = warp - 2) of every k-block =====
    const int cg = warp - 2;
    {
      for (int kb = 0; kb < nkb; ++kb) {
        const int n0 = kb * BLOCK_K + cg * 4, sa_i = kb % FC_ASTAGES;
        float4 w[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) w[i] = *reinterpret_cast<const float4*>(&w1s[i][n0]);   // same address across the warp: broadcast
        float4 o[4];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f, o3 = 0.0f;
#pragma unroll
          for (int i = 0; i < 12; ++i) {
            o0 = fmaf(x[rr][i], w[i].x, o0); o1 = fmaf(x[rr][i], w[i].y, o1); o2 = fmaf(x[rr][i], w[i].z, o2); o3 = fmaf(x[rr][i], w[i].w, o3);
          }
          o[rr] = make_float4(fmaxf(o0, 0.0f), fmaxf(o1, 0.0f), fmaxf(o2, 0.0f), fmaxf(o3, 0.0f));
        }
        if (kb >= FC_ASTAGES) mbar_wait(&a_empty[sa_i], ((kb / FC_ASTAGES) - 1) & 1);   // the MMAs (and the h1 store) of k-block kb - 3 have read the slot
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const int r = lane + 32 * rr;                       // SWIZZLE_128B: 16-byte chunk j of row r at j ^ (r & 7); units beyond l1 are relu(0) = 0
          *reinterpret_cast<float4*>(sA + sa_i * TILE_BYTES + r * 128 + ((cg ^ (r & 7)) << 4)) = o[rr];
        }
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[sa_i]);
        if (warp == 2 && lane == 0) FC_STAMP(64 + kb);
      }
    }
    // ===== epilogue (the same 8 warps; TMEM lane quarter = warp % 4, column half hh): a thread owns one row of one half =====
    const int hh = cg >> 2;
    uint8_t* buf = sB + cg * (4 * 4096);                      // the W2 ring is idle once the accumulators are final: 4 staging chunks per warp
    const bool store = p.H2[prob] != nullptr;
    mbar_wait(&acc_full, 0);
    if (warp == 2 && lane == 0) FC_STAMP(73);
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
#pragma unroll 1
    for (int c = 0; c < NCOL / 64; ++c) {
      const int lc = hh * (NCOL / 2) + c * 32, nc = nh * NCOL + lc;   // column of this CTA's accumulator / layer-2 unit
      if (nc >= p.L2) break;
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)lc, v);
      float4 o[8];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {   // columns beyond l2: accumulator 0 (TMA zero fill), b2 = W3 = 0 -> h2 = 0, no contribution
        const float4 bv = *reinterpret_cast<const float4*>(&b2s[nc + j4 * 4]);
        const float4 wa = *reinterpret_cast<const float4*>(&w3s[0][nc + j4 * 4]);
        const float4 wb = *reinterpret_cast<const float4*>(&w3s[1][nc + j4 * 4]);
        o[j4].x = fmaxf(__uint_as_float(v[j4 * 4 + 0]) + bv.x, 0.0f); o[j4].y = fmaxf(__uint_as_float(v[j4 * 4 + 1]) + bv.y, 0.0f);
        o[j4].z = fmaxf(__uint_as_float(v[j4 * 4 + 2]) + bv.z, 0.0f); o[j4].w = fmaxf(__uint_as_float(v[j4 * 4 + 3]) + bv.w, 0.0f);
        d0 = fmaf(o[j4].x, wa.x, d0); d0 = fmaf(o[j4].y, wa.y, d0); d0 = fmaf(o[j4].z, wa.z, d0); d0 = fmaf(o[j4].w, wa.w, d0);
        d1 = fmaf(o[j4].x, wb.x, d1); d1 = fmaf(o[j4].y, wb.y, d1); d1 = fmaf(o[j4].z, wb.z, d1); d1 = fmaf(o[j4].w, wb.w, d1);
      }
      if (store) {
        uint8_t* b = buf + (c & 3) * 4096;
        if (c >= 4) {   // the store of chunk c - 4 has read this buffer (at most the 3 newer ones still pending)
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 3;\n" ::: "memory");
          __syncwarp();
        }
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) *reinterpret_cast<float4*>(b + lane * 128 + ((j4 ^ (lane & 7)) << 4)) = o[j4];
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&maps.d[prob], b, nc, m0 + q * 32, learner);
          asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
      }
    }
    if (warp == 2 && lane == 0) FC_STAMP(74);
    if (hh == 1) { dpart[0][q * 32 + lane] = d0; dpart[1][q * 32 + lane] = d1; }
    asm volatile("bar.sync 1, 256;\n" ::: "memory");          // the 8 epilogue warps
    if (hh == 0) { d0 += dpart[0][q * 32 + lane]; d1 += dpart[1][q * 32 + lane]; fin = true; }
    if (store && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  }
  if (NS == 2) {   // the second CTA's share of the dot products -> the first CTA's shared memory; every thread of both CTAs meets at the cluster barrier
    if (fin && nh == 1) {
      uint32_t r0, r1;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r0) : "r"(smem_u32(&xpart[0][q * 32 + lane])), "r"(0));
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r1) : "r"(smem_u32(&xpart[1][q * 32 + lane])), "r"(0));
      asm volatile("st.shared::cluster.f32 [%0], %1;\n" ::"r"(r0), "f"(d0) : "memory");
      asm volatile("st.shared::cluster.f32 [%0], %1;\n" ::"r"(r1), "f"(d1) : "memory");
    }
    __syncwarp();
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
    if (fin && nh == 0) { d0 += xpart[0][q * 32 + lane]; d1 += xpart[1][q * 32 + lane]; }
  }
  if (fin && nh == 0 && erow < p.M) {
    const float* __restrict__ b3 = p.b3[prob] + lo;
    const float z0 = d0 + __ldg(b3);
    if (p.out_mode[prob] == TC_OUT_TANH) {
      float* o = p.out[prob] + lo + (long long)erow * p.ldo[prob];
      o[0] = tanhf(z0);
      if (J == 2) o[1] = tanhf(d1 + __ldg(b3 + 1));
    } else if (p.out_mode[prob] == TC_OUT_ID) {
      p.out[prob][lo + (long long)erow * p.ldo[prob]] = z0;
    } else {  // TC_OUT_TD: y = r + gamma (1 - done) q'; dq = 2 (q - y) / B   (DDPG.jl:133, d mse / d q)
      const float y = p.td_r[lo + erow] + (td_gamma * (1.0f - p.td_done[lo + erow])) * z0;
      p.out[prob][lo + (long long)erow * p.ldo[prob]] = y;
      p.td_dq[lo + erow] = 2.0f * (p.td_q[lo + erow] - y) * p.inv_batch;
    }
  }
  if (warp == 2 && lane == 0) FC_STAMP(76);
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(NCOL));
  }
}

// ---------------------------------------------------------------------------------------------------------------- backward chain
// The dX chain of a net for a 128-row tile in one CTA (see tc_gemm.h).  Per k-block of 32 layer-2 units: the h2 tile block arrives by TMA
// in the 128B-swizzled K-major operand layout, 8 warps turn it IN PLACE into dz2 = (sum_j dout[row][j] W3[n][j]) * (h2 > 0), the MMA warp
// (optionally) sends the finished block to HBM by a TMA store from the operand and issues tcgen05.mma 128 x 256 x 8 against the W2 block
// [256 layer-1 units][32 layer-2 units] (K-major as Flux stores W2; units beyond l1 are zero-filled by TMA).  The epilogue (8 warps: TMEM
// lane quarter x column half) masks with relu'(h1), stores dz1 through TMA from the then idle W2 ring, and folds the product with the two
// action rows of W1 into registers.  Replaces outer_mask_kernel + tc_gemm_kernel<0,0> (+ gemm_skinny_kernel).
constexpr int BC_THREADS = 320, BC_N = 256, BC_ASTAGES = 4, BC_BSTAGES = 4;   // BC_N: layer-1 units per row tile; a CTA takes all of them or (NS = 2) half
constexpr int BC_B_STAGE = BC_N * BLOCK_K * 4;                 // 32 KB: [256 rows][32 k]
constexpr int BC_SMEM = BC_ASTAGES * TILE_BYTES + BC_BSTAGES * BC_B_STAGE + 1024;
static_assert(BC_BSTAGES * BC_B_STAGE >= 8 * 4 * 4096, "the epilogue stages 4 chunks per warp in the W2 ring");

// NS = 2: two CTAs per row tile, each with 128 of the layer-1 units (half of the W2 stream; the h2 block and its dz2 are computed by both,
// stored by the first; the action-input gradient is the sum of the two CTAs' shares: two atomic adds onto zeros — commutative, hence
// deterministic).  For minibatches whose row tiles alone would leave more than half of the SMs idle.
template <int NS>
__global__ void __launch_bounds__(BC_THREADS, 1)
tc_bwd_chain_kernel(const __grid_constant__ TcMaps maps, const TcBwdChainArgs p) {
  constexpr int NC = BC_N / NS;                                // layer-1 units (accumulator columns) of this CTA
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + BC_ASTAGES * TILE_BYTES;
  __shared__ uint64_t h_full[BC_ASTAGES], a_full[BC_ASTAGES], a_empty[BC_ASTAGES], b_full[BC_BSTAGES], b_empty[BC_BSTAGES], acc_full;
  __shared__ uint32_t tmem_base_smem;
  __shared__ __align__(16) float w3s[2][2 * BC_N];            // W3[:, j] (zero beyond l2)
  __shared__ __align__(16) float w1a[2][BC_N];                // the two action rows of W1 (zero beyond l1)
  __shared__ float dpart[2][BLOCK_M];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = (blockIdx.x / NS) * BLOCK_M, nh = blockIdx.x % NS, learner = blockIdx.y, J = p.J;   // nh: which half of the layer-1 units
  const long long lo = (long long)learner * p.pop_stride;
  const int nkb = (p.L2 + BLOCK_K - 1) / BLOCK_K;              // k-blocks of 32 layer-2 units
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
  if (threadIdx.x == 0) {
    for (int k = 0; k < BC_ASTAGES; ++k) { mbar_init(&h_full[k], 1); mbar_init(&a_full[k], 8); mbar_init(&a_empty[k], 1); }
    for (int s = 0; s < BC_BSTAGES; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    mbar_init(&acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.a[0]) : "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.b[0]) : "memory");
    if (p.DZ2 && nh == 0) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.a[1]) : "memory");
    if (p.DZ1) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&maps.d[0]) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_smem)), "n"(NC));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;
  // everything this kernel reads may be its predecessor's output (the optimiser step, the forward pass): set-up above, data below
  asm volatile("griddepcontrol.wait;\n" ::: "memory");
  if (warp >= 2) {   // W3 and the action rows of W1 for the 8 producer / epilogue warps, while the TMA warp already streams the first blocks
    const int t = threadIdx.x - 64;
    for (int n = t; n < 2 * BC_N; n += BC_THREADS - 64) {
      const bool ok = n < p.L2;
      w3s[0][n] = ok ? __ldg(p.W3 + lo + (long long)n * J) : 0.0f;
      w3s[1][n] = (ok && J == 2) ? __ldg(p.W3 + lo + (long long)n * J + 1) : 0.0f;
    }
    if (p.dA) {
      for (int n = t; n < 2 * BC_N; n += BC_THREADS - 64) {
        const int j = n / BC_N, i = n - j * BC_N;
        w1a[j][i] = (i < NC && nh * NC + i < p.L1) ? __ldg(p.W1a + lo + (long long)j * p.L1 + nh * NC + i) : 0.0f;   // this CTA's units
      }
    }
    asm volatile("bar.sync 2, 256;\n" ::: "memory");
  }

  if (warp == 0) {
    // ===== TMA producer: the h2 block [128 rows][32 units] and the W2 block [256 layer-1 units][32 layer-2 units] of every k-block =====
    if (elect_one()) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int sa = kb % BC_ASTAGES, pa = (kb / BC_ASTAGES) & 1, sb = kb % BC_BSTAGES, pb = (kb / BC_BSTAGES) & 1;
        mbar_wait(&a_empty[sa], pa ^ 1);
        mbar_expect_tx(&h_full[sa], TILE_BYTES);
        tma_load_3d(sA + sa * TILE_BYTES, &maps.a[0], &h_full[sa], kb * BLOCK_K, m0, learner);
        mbar_wait(&b_empty[sb], pb ^ 1);
        mbar_expect_tx(&b_full[sb], BC_B_STAGE / NS);
        tma_load_3d(sB + sb * BC_B_STAGE, &maps.b[0], &b_full[sb], kb * BLOCK_K, nh * NC, learner);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (+ the dz2 stores from the operand) =====
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(NC >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
    if (elect_one()) {
      const bool store = p.DZ2 != nullptr && nh == 0;
      for (int kb = 0; kb < nkb; ++kb) {
        const int sa = kb % BC_ASTAGES, pa = (kb / BC_ASTAGES) & 1, sb = kb % BC_BSTAGES, pb = (kb / BC_BSTAGES) & 1;
        mbar_wait(&a_full[sa], pa);                         // the 8 warps have turned this block into dz2 (and fenced it)
        if (store) {
          tma_store_3d(&maps.a[1], sA + sa * TILE_BYTES, kb * BLOCK_K, m0, learner);
          asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
        mbar_wait(&b_full[sb], pb);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const uint32_t a0 = smem_u32(sA + sa * TILE_BYTES), b0 = smem_u32(sB + sb * BC_B_STAGE);
#pragma unroll
        for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
          const uint64_t ad = make_smem_desc(a0 + kk * 32, 16, 1024, 2);   // K-major, SWIZZLE_128B
          const uint64_t bd = make_smem_desc(b0 + kk * 32, 16, 1024, 2);   // K-major, SWIZZLE_128B: 256 rows of 128 bytes
          umma_tf32(tmem_base, ad, bd, idesc, (kb | kk) != 0 ? 1u : 0u);
        }
        umma_commit(&b_empty[sb]);
        if (kb > 0) {   // block kb - 1: its MMAs are covered by this commit; its store (all but the newest) has read the operand
          if (store) asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");
          umma_commit(&a_empty[(kb - 1) % BC_ASTAGES]);
        }
      }
      if (store) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
      umma_commit(&a_empty[(nkb - 1) % BC_ASTAGES]);
      umma_commit(&acc_full);
    }
  } else {
    // ===== dz2 producers (warps 2-9): thread = rows {lane, lane+32, lane+64, lane+96} x the 16-byte chunk cg = warp - 2 of every block =====
    const int cg = warp - 2;
    {
      float dz[4][2];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int row = m0 + lane + 32 * rr;
        dz[rr][0] = row < p.M ? __ldcg(p.dout + lo + (long long)row * J) : 0.0f;
        dz[rr][1] = (row < p.M && J == 2) ? __ldcg(p.dout + lo + (long long)row * J + 1) : 0.0f;
      }
      for (int kb = 0; kb < nkb; ++kb) {
        const int sa = kb % BC_ASTAGES, pa = (kb / BC_ASTAGES) & 1, n0 = kb * BLOCK_K + cg * 4;
        const float4 wa = *reinterpret_cast<const float4*>(&w3s[0][n0]);
        const float4 wb = *reinterpret_cast<const float4*>(&w3s[1][n0]);
        mbar_wait(&h_full[sa], pa);
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const int r = lane + 32 * rr;
          float4* q4 = reinterpret_cast<float4*>(sA + sa * TILE_BYTES + r * 128 + ((cg ^ (r & 7)) << 4));
          const float4 hv = *q4;
          float4 o;   // the same order as outer_mask_kernel: fma(dz[1], w[1], fma(dz[0], w[0], 0))
          o.x = hv.x > 0.0f ? fmaf(dz[rr][1], wb.x, fmaf(dz[rr][0], wa.x, 0.0f)) : 0.0f;
          o.y = hv.y > 0.0f ? fmaf(dz[rr][1], wb.y, fmaf(dz[rr][0], wa.y, 0.0f)) : 0.0f;
          o.z = hv.z > 0.0f ? fmaf(dz[rr][1], wb.z, fmaf(dz[rr][0], wa.z, 0.0f)) : 0.0f;
          o.w = hv.w > 0.0f ? fmaf(dz[rr][1], wb.w, fmaf(dz[rr][0], wa.w, 0.0f)) : 0.0f;
          *q4 = o;
        }
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[sa]);
      }
    }
    // ===== epilogue (the same 8 warps; TMEM lane quarter = warp % 4, column half hh of this CTA's layer-1 units) =====
    const int q = warp & 3, hh = cg >> 2;
    const int erow = m0 + q * 32 + lane;
    uint8_t* buf = sB + cg * (4 * 4096);
    const bool store = p.DZ1 != nullptr, want_da = p.dA != nullptr;
    const float* __restrict__ h1row = p.H1 + lo + (long long)(erow < p.M ? erow : 0) * p.ldh1;
    float d0 = 0.0f, d1 = 0.0f;
    mbar_wait(&acc_full, 0);
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
#pragma unroll 1
    for (int c = 0; c < NC / 64; ++c) {
      const int lc = hh * (NC / 2) + c * 32, nc = nh * NC + lc;   // column of this CTA's accumulator / layer-1 unit
      if (nc >= p.L1) break;
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)lc, v);
      float4 o[8];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {   // units beyond l1: W2 rows zero-filled -> accumulator 0
        const float4 hv = __ldcg(reinterpret_cast<const float4*>(h1row + nc + j4 * 4));
        o[j4].x = hv.x > 0.0f ? __uint_as_float(v[j4 * 4 + 0]) : 0.0f; o[j4].y = hv.y > 0.0f ? __uint_as_float(v[j4 * 4 + 1]) : 0.0f;
        o[j4].z = hv.z > 0.0f ? __uint_as_float(v[j4 * 4 + 2]) : 0.0f; o[j4].w = hv.w > 0.0f ? __uint_as_float(v[j4 * 4 + 3]) : 0.0f;
        if (want_da) {
          const float4 ua = *reinterpret_cast<const float4*>(&w1a[0][lc + j4 * 4]);
          const float4 ub = *reinterpret_cast<const float4*>(&w1a[1][lc + j4 * 4]);
          d0 = fmaf(o[j4].x, ua.x, d0); d0 = fmaf(o[j4].y, ua.y, d0); d0 = fmaf(o[j4].z, ua.z, d0); d0 = fmaf(o[j4].w, ua.w, d0);
          d1 = fmaf(o[j4].x, ub.x, d1); d1 = fmaf(o[j4].y, ub.y, d1); d1 = fmaf(o[j4].z, ub.z, d1); d1 = fmaf(o[j4].w, ub.w, d1);
        }
      }
      if (store) {
        uint8_t* b = buf + c * 4096;   // 4 chunks per warp: a buffer each
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) *reinterpret_cast<float4*>(b + lane * 128 + ((j4 ^ (lane & 7)) << 4)) = o[j4];
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&maps.d[0], b, nc, m0 + q * 32, learner);
          asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
      }
    }
    if (want_da) {
      if (hh == 1) { dpart[0][q * 32 + lane] = d0; dpart[1][q * 32 + lane] = d1; }
      asm volatile("bar.sync 1, 256;\n" ::: "memory");        // the 8 epilogue warps
      if (hh == 0 && erow < p.M) {   // times tanh'(z) = 1 - a^2 (the actor's output layer; EPI_TANH_GRAD of the layer-by-layer path)
        const float a0 = __ldcg(p.act + lo + (long long)erow * p.ld_act), a1 = __ldcg(p.act + lo + (long long)erow * p.ld_act + 1);
        const float g0 = (d0 + dpart[0][q * 32 + lane]) * (1.0f - a0 * a0), g1 = (d1 + dpart[1][q * 32 + lane]) * (1.0f - a1 * a1);
        if (NS == 1) { p.dA[lo + (long long)erow * 2] = g0; p.dA[lo + (long long)erow * 2 + 1] = g1; }
        else { atomicAdd(p.dA + lo + (long long)erow * 2, g0); atomicAdd(p.dA + lo + (long long)erow * 2 + 1, g1); }   // onto zeros (the host clears dA)
      }
    }
    if (store && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(NC));
  }
}

// deterministic second pass of a split-K GEMM: D[m][n] = sum_s W[s][m][n] (fixed order)
__global__ void __launch_bounds__(256)
tc_splitk_reduce_kernel(const float* __restrict__ ws, long long split_stride, int splits, float* __restrict__ D, long long n_elems) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_elems) return;
  float acc = ws[i];
  for (int s = 1; s < splits; ++s) acc += ws[(long long)s * split_stride + i];
  D[i] = acc;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// fp32 operand map: dim0 = contiguous dimension (n0 elements), dim1 = strided dimension (n1 rows, `ld` floats apart),
// dim2 = batch entries `bstride` floats apart (1 entry for a plain GEMM)
int make_tmap(CUtensorMap* tm, const float* ptr, long long n0, long long n1, long long ld, int box0, int box1, bool mn_major, int batch,
              long long bstride) {
  EncodeTiledFn enc = get_encode();
  REQUIRE(enc, SHEMS_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled is not available from this driver");
  REQUIRE(((uintptr_t)ptr & 15) == 0 && (ld * 4) % 16 == 0 && (bstride * 4) % 16 == 0, SHEMS_ERR_INVALID,
          "tc_gemm: operand needs a 16-byte aligned base, row stride and batch stride (ld=%lld, batch stride=%lld)", ld, bstride);
  cuuint64_t dims[3] = {(cuuint64_t)n0, (cuuint64_t)n1, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(batch > 1 ? bstride : ld * n1) * 4};
  cuuint32_t box[3] = {(cuuint32_t)box0, (cuuint32_t)box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  REQUIRE(r == CUDA_SUCCESS, SHEMS_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return SHEMS_OK;
}

template <bool A_MN, bool B_MN>
int set_smem_attr() {
  CUDA_TRY(cudaFuncSetAttribute(tc_gemm_kernel<A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  return SHEMS_OK;
}
// 3-D fp32 map of the output {N, M, splits} (rows ldd floats apart, splits split_stride floats apart), box 32 x 32 x 1, 128B swizzle
int make_tmap_out(CUtensorMap* tm, float* ptr, long long N, long long M, long long splits, long long ldd, long long split_stride) {
  EncodeTiledFn enc = get_encode();
  REQUIRE(enc, SHEMS_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)M, (cuuint64_t)splits};
  cuuint64_t strides[2] = {(cuuint64_t)ldd * 4, (cuuint64_t)(splits > 1 ? split_stride : ldd * M) * 4};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  REQUIRE(r == CUDA_SUCCESS, SHEMS_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled(D) failed (%d)", (int)r);
  return SHEMS_OK;
}

template <bool A_MN, bool B_MN>
int launch_variant(cudaStream_t st, const TcMaps& maps, const TcGemmArgs& a) {
  static bool attr_set = false;
  if (!attr_set) {
    if (int s = set_smem_attr<A_MN, B_MN>()) return s;
    attr_set = true;
  }
  const long long tiles = (long long)((a.M + BLOCK_M - 1) / BLOCK_M) * ((a.N + BLOCK_N - 1) / BLOCK_N) * (a.batch > 1 ? a.batch : a.splits) * a.nprob;
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  const unsigned grid = (unsigned)(tiles < n_sm ? tiles : n_sm);  // persistent: one CTA per SM, tiles dealt round-robin
  if (a.pdl) {   // a programmatic dependent of its predecessor in the stream
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(192); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<A_MN, B_MN>, maps, a));
  } else {
    tc_gemm_kernel<A_MN, B_MN><<<grid, 192, SMEM_BYTES, st>>>(maps, a);
  }
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

}  // namespace

// opt every variant into its dynamic shared memory on the current device (call once per device, outside stream capture)
int tc_gemm_prepare() {
  int s;
  if ((s = set_smem_attr<false, false>())) return s;
  if ((s = set_smem_attr<false, true>())) return s;
  if ((s = set_smem_attr<true, false>())) return s;
  if ((s = set_smem_attr<true, true>())) return s;
  REQUIRE(get_encode(), SHEMS_ERR_CUDA, "tc_gemm: cuTensorMapEncodeTiled is not available from this driver");
  CUDA_TRY(cudaFuncSetAttribute(tc_fwd_chain_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM));
  CUDA_TRY(cudaFuncSetAttribute(tc_fwd_chain_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM));
  CUDA_TRY(cudaFuncSetAttribute(tc_bwd_chain_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BC_SMEM));
  CUDA_TRY(cudaFuncSetAttribute(tc_bwd_chain_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, BC_SMEM));
  return SHEMS_OK;
}

// D_q = epi(A_q·B_q) for q < nprob same-shape products in ONE launch (own operands, outputs, bias / mask pointers; shared M, N, K,
// leading dimensions, major-ness, epilogue and batch strides).  With splits > 1 (single problem only) `workspace` must hold
// splits*M*N floats; the partial tiles are summed in a fixed order by a second kernel (deterministic, unlike atomics).
// bt.count > 1: that many independent products per problem (grid.z), entry i bt.s* floats behind entry i-1 (no split-K then).
int tc_gemm_multi(cudaStream_t st, int nprob, const TcOperand* A, const TcOperand* B, float* const* D, long long ldd, int M, int N, int K, int epi,
                  const float* const* bias, const float* const* aux, long long auxld, int splits, float* workspace, const TcBatch& bt) {
  REQUIRE(nprob >= 1 && nprob <= TC_MAX_PROBLEMS, SHEMS_ERR_INVALID, "tc_gemm: nprob=%d", nprob);
  REQUIRE(M >= 1 && N >= 1 && K >= 1 && splits >= 1 && bt.count >= 1, SHEMS_ERR_INVALID, "tc_gemm: M=%d N=%d K=%d splits=%d batch=%d", M, N, K, splits, bt.count);
  REQUIRE(splits == 1 || (workspace && epi == TC_EPI_NONE && ldd == N && bt.count == 1 && nprob == 1), SHEMS_ERR_INVALID,
          "tc_gemm: split-K needs a workspace, no epilogue, ldd == N and a single product");
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  TcGemmArgs a;
  memset(&a, 0, sizeof(a));
  a.M = M; a.N = N; a.K = K; a.splits = splits; a.epi = epi; a.auxld = auxld; a.nprob = nprob;
  a.batch = bt.count; a.bs_bias = bt.sBias; a.bs_aux = bt.sAux; a.pdl = bt.pdl ? 1 : 0;
  if (splits == 1) { a.ldd = ldd; a.split_stride = bt.count > 1 ? bt.sD : 0; }
  else { a.ldd = N; a.split_stride = (long long)M * N; }
  const int nz = bt.count > 1 ? bt.count : splits;
  a.tma_store = ((a.ldd % 4) == 0 && (a.split_stride % 4) == 0) ? 1 : 0;
  for (int q = 0; q < nprob; ++q) {
    REQUIRE(A[q].mn_major == A[0].mn_major && B[q].mn_major == B[0].mn_major && A[q].ld == A[0].ld && B[q].ld == B[0].ld, SHEMS_ERR_INVALID,
            "tc_gemm: the problems of one launch must share layout and leading dimensions");
    a.D[q] = splits == 1 ? D[q] : workspace;
    a.bias[q] = bias ? bias[q] : nullptr; a.aux[q] = aux ? aux[q] : nullptr;
    if (((uintptr_t)a.D[q] & 15) != 0) a.tma_store = 0;
  }
  for (int q = nprob; q < TC_MAX_PROBLEMS; ++q) { a.D[q] = a.D[0]; a.bias[q] = a.bias[0]; a.aux[q] = a.aux[0]; }
  int s;
  for (int q = 0; q < nprob; ++q) {
    // K-major: dim0 = K, dim1 = rows, box {32 k, 128 rows}; MN-major: dim0 = rows, dim1 = K, box {32 rows, 32 k}
    if ((s = A[q].mn_major ? make_tmap(&maps.a[q], A[q].ptr, M, K, A[q].ld, 32, BLOCK_K, true, bt.count, bt.sA)
                           : make_tmap(&maps.a[q], A[q].ptr, K, M, A[q].ld, BLOCK_K, BLOCK_M, false, bt.count, bt.sA))) return s;
    if ((s = B[q].mn_major ? make_tmap(&maps.b[q], B[q].ptr, N, K, B[q].ld, 32, BLOCK_K, true, bt.count, bt.sB)
                           : make_tmap(&maps.b[q], B[q].ptr, K, N, B[q].ld, BLOCK_K, BLOCK_N, false, bt.count, bt.sB))) return s;
    // TMA store of the output tile when D's rows are 16-byte aligned (activations with padded ld, gradients, the split-K workspace)
    if (a.tma_store && (s = make_tmap_out(&maps.d[q], a.D[q], N, M, nz, a.ldd, a.split_stride))) return s;
  }
  if (A[0].mn_major && B[0].mn_major) s = launch_variant<true, true>(st, maps, a);
  else if (A[0].mn_major) s = launch_variant<true, false>(st, maps, a);
  else if (B[0].mn_major) s = launch_variant<false, true>(st, maps, a);
  else s = launch_variant<false, false>(st, maps, a);
  if (s) return s;
  if (splits > 1) {
    const long long ne = (long long)M * N;
    tc_splitk_reduce_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(workspace, a.split_stride, splits, D[0], ne);
    CUDA_TRY(cudaGetLastError());
  }
  return SHEMS_OK;
}


// One launch = the forward pass of up to 3 nets (same widths) over the whole minibatch, 128 rows per CTA (see tc_fwd_chain_kernel)
#ifdef FC_TRACE
extern "C" __attribute__((visibility("default"))) int tc_fwd_chain_trace_read(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, fc_trace, sizeof(fc_trace));
}
#endif
int tc_fwd_chain(cudaStream_t st, const TcFwdChainArgs& a) {
  REQUIRE(a.nprob >= 1 && a.nprob <= TC_MAX_PROBLEMS && a.M >= 1, SHEMS_ERR_INVALID, "tc_fwd_chain: nprob=%d M=%d", a.nprob, a.M);
  REQUIRE(a.L1 >= 1 && a.L1 <= FC_KB * BLOCK_K && a.L2 >= 1 && a.L2 <= 2 * FC_N && a.L2 % 4 == 0, SHEMS_ERR_INVALID,
          "tc_fwd_chain: widths %d/%d outside the kernel's plan (l1 <= 256, l2 <= 512, l2 %% 4 == 0)", a.L1, a.L2);
  const int pop = a.pop > 1 ? a.pop : 1;
  REQUIRE(pop == 1 || a.pop_stride % 4 == 0, SHEMS_ERR_INVALID, "tc_fwd_chain: the learners' slabs must be a multiple of 16 bytes apart");
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  int s;
  for (int q = 0; q < a.nprob; ++q) {
    REQUIRE(a.K1[q] >= 1 && a.K1[q] <= 11 && (a.J[q] == 1 || a.J[q] == 2), SHEMS_ERR_INVALID, "tc_fwd_chain: K1=%d J=%d", a.K1[q], a.J[q]);
    REQUIRE(!a.H1[q] || (a.ldh1 % 4 == 0 && ((uintptr_t)a.H1[q] & 15) == 0 && a.ldh1 >= a.L1), SHEMS_ERR_INVALID,
            "tc_fwd_chain: h1 needs 16-byte aligned rows of at least l1 floats (a multiple of 4)");
    if ((s = make_tmap(&maps.b[q], a.W2[q], a.L2, a.L1, a.L2, 32, FC_BK, true, pop, a.pop_stride))) return s;   // MN-major: dim0 = columns, dim1 = k, dim2 = learner
    if (a.H1[q]) {   // h1 leaves through TMA stores from the swizzled A operand: box {32 columns, 128 rows}, SWIZZLE_128B
      EncodeTiledFn enc = get_encode();
      cuuint64_t dims[3] = {(cuuint64_t)a.ldh1, (cuuint64_t)a.M, (cuuint64_t)pop};
      cuuint64_t strides[2] = {(cuuint64_t)a.ldh1 * 4, (cuuint64_t)(pop > 1 ? a.pop_stride : a.ldh1 * (long long)a.M) * 4};
      cuuint32_t box[3] = {32, 128, 1};
      cuuint32_t estr[3] = {1, 1, 1};
      CUresult r = enc(&maps.a[q], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)a.H1[q], dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      REQUIRE(r == CUDA_SUCCESS, SHEMS_ERR_CUDA, "tc_fwd_chain: cuTensorMapEncodeTiled(h1) failed (%d)", (int)r);
    }
    if (a.H2[q] && (s = make_tmap_out(&maps.d[q], a.H2[q], a.L2, a.M, pop, a.ldh2, a.pop_stride))) return s;
  }
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_TRY(cudaFuncSetAttribute(tc_fwd_chain_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM));
    CUDA_TRY(cudaFuncSetAttribute(tc_fwd_chain_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC_SMEM));
    attr_set = true;
  }
  const int mt = (a.M + BLOCK_M - 1) / BLOCK_M, ns = a.nsplit == 2 ? 2 : 1;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(mt * a.nprob * ns), (unsigned)pop); cfg.blockDim = dim3(FC_THREADS); cfg.dynamicSmemBytes = FC_SMEM; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  if (ns == 2) {   // the two CTAs of a row tile form a cluster (distributed shared memory for the output layer's partial sums)
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  if (a.pdl) {     // a programmatic dependent of its predecessor in the stream (captured as such in the update's graph)
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  if (ns == 2) CUDA_TRY(cudaLaunchKernelEx(&cfg, tc_fwd_chain_kernel<2>, maps, a));
  else CUDA_TRY(cudaLaunchKernelEx(&cfg, tc_fwd_chain_kernel<1>, maps, a));
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

// One launch = the dX chain of a net over the whole minibatch, 128 rows per CTA (see tc_bwd_chain_kernel)
int tc_bwd_chain(cudaStream_t st, const TcBwdChainArgs& a) {
  REQUIRE(a.M >= 1 && a.L1 >= 1 && a.L1 <= BC_N && a.L2 >= 1 && a.L2 <= 2 * BC_N && a.L2 % 4 == 0 && (a.J == 1 || a.J == 2), SHEMS_ERR_INVALID,
          "tc_bwd_chain: M=%d widths %d/%d J=%d outside the kernel's plan (l1 <= 256, l2 <= 512, l2 %% 4 == 0)", a.M, a.L1, a.L2, a.J);
  REQUIRE(a.dout && a.W3 && a.W2 && a.H2 && a.H1 && a.ldh1 % 32 == 0 && a.ldh2 % 4 == 0 && (!a.dA || (a.W1a && a.act)), SHEMS_ERR_INVALID,
          "tc_bwd_chain: NULL operand, or activation rows that are not whole 128-byte lines");
  const int pop = a.pop > 1 ? a.pop : 1;
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  int s;
  if ((s = make_tmap(&maps.a[0], a.H2, a.L2, a.M, a.ldh2, BLOCK_K, BLOCK_M, false, pop, a.pop_stride))) return s;   // h2 blocks: K-major, SWIZZLE_128B
  if (a.DZ2 && (s = make_tmap(&maps.a[1], a.DZ2, a.L2, a.M, a.ldh2, BLOCK_K, BLOCK_M, false, pop, a.pop_stride))) return s;
  const int tiles = (a.M + BLOCK_M - 1) / BLOCK_M;
  const int ns = a.nsplit == 2 ? 2 : 1;
  if ((s = make_tmap(&maps.b[0], a.W2, a.L2, a.L1, a.L2, BLOCK_K, BC_N / ns, false, pop, a.pop_stride))) return s;   // W2 [l1][l2]: K-major B, rows beyond l1 zero
  if (a.DZ1 && (s = make_tmap_out(&maps.d[0], a.DZ1, a.L1, a.M, pop, a.ldh1, a.pop_stride))) return s;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_TRY(cudaFuncSetAttribute(tc_bwd_chain_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BC_SMEM));
    CUDA_TRY(cudaFuncSetAttribute(tc_bwd_chain_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, BC_SMEM));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(tiles * ns), (unsigned)pop); cfg.blockDim = dim3(BC_THREADS); cfg.dynamicSmemBytes = BC_SMEM; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = a.pdl ? 1 : 0;
  if (ns == 2) CUDA_TRY(cudaLaunchKernelEx(&cfg, tc_bwd_chain_kernel<2>, maps, a));
  else CUDA_TRY(cudaLaunchKernelEx(&cfg, tc_bwd_chain_kernel<1>, maps, a));
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

int tc_gemm(cudaStream_t st, const TcOperand& A, const TcOperand& B, float* D, long long ldd, int M, int N, int K, int epi,
            const float* bias, const float* aux, long long auxld, int splits, float* workspace, const TcBatch& bt) {
  float* Ds[1] = {D}; const float* bs[1] = {bias}; const float* as[1] = {aux};
  return tc_gemm_multi(st, 1, &A, &B, Ds, ldd, M, N, K, epi, bs, as, auxld, splits, workspace, bt);
}

// test / benchmark entry point (device pointers): D[M×N] = A·B with the stated major-ness
extern "C" int32_t shems_tc_gemm(const float* a_dev, int64_t lda, int32_t a_mn, const float* b_dev, int64_t ldb, int32_t b_mn, float* d_dev,
                                 int64_t ldd, int32_t M, int32_t N, int32_t K, int32_t epi, const float* bias_dev, const float* aux_dev,
                                 int64_t auxld, int32_t splits, float* workspace_dev, void* cuda_stream) {
  REQUIRE(a_dev && b_dev && d_dev, SHEMS_ERR_INVALID, "shems_tc_gemm: NULL argument");
  TcOperand A{a_dev, lda, a_mn != 0}, B{b_dev, ldb, b_mn != 0};
  return tc_gemm((cudaStream_t)cuda_stream, A, B, d_dev, ldd, M, N, K, epi, bias_dev, aux_dev, auxld, splits, workspace_dev, TcBatch());
}
