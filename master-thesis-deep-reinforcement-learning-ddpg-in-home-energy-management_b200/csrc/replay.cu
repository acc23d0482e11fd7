// replay.cu — device-resident replay memory: `memory = CircularBuffer{Any}(MEM_SIZE)` of
// [s, a, r, s', done] (RL-SHEMS/input.jl:140; src/memory_plotting_saving.jl:31-57) as a
// structure-of-arrays ring in HBM with on-device sampling.
//
// Layout: 23 float32 fields per slot in 32-slot tiles, see ring.cuh: a full record (s 9, a 2, r 1, s' 9, done 1 = 88 B) or a compact
// one (Soc_b, Soc_ev, a 2, r, Soc_b', Soc_ev', series tag: 32 B) whose other fields are rows of the ring's copy of an env series.
#include <new>
#include <vector>
#include <string.h>

#include "common.h"

#define TRY_PRIO(expr) do { const int _s = (expr); if (_s) return _s; } while (0)

extern "C" int32_t replay_create(int64_t capacity, int32_t device, ShemsReplay** out) {
  REQUIRE(out && capacity >= 1, SHEMS_ERR_INVALID, "replay_create: capacity=%lld", (long long)capacity);
  REQUIRE(shems_device_count() > 0, SHEMS_ERR_CUDA, "replay_create: no CUDA device (this library has no CPU fallback)");
  GUARD(device);
  ShemsReplay* rp = new (std::nothrow) ShemsReplay();
  REQUIRE(rp, SHEMS_ERR_INVALID, "replay_create: out of host memory");
  memset(rp, 0, sizeof(*rp));
  rp->device = device; rp->capacity = capacity;
  const size_t floats = ring_alloc_floats(capacity);
  cudaError_t st;
  if ((st = cudaMalloc(&rp->alloc, sizeof(float) * floats)) != cudaSuccess ||
      (st = cudaMemset(rp->alloc, 0, sizeof(float) * floats)) != cudaSuccess ||
      (st = cudaMalloc(&rp->minmax_scratch, sizeof(float) * 18)) != cudaSuccess) {
    shems_set_error("replay_create: %s", cudaGetErrorString(st));
    replay_destroy(rp);
    return SHEMS_ERR_CUDA;
  }
  rp->ring = ring_in_alloc(rp->alloc);
  *out = rp;
  return SHEMS_OK;
}
extern "C" int32_t replay_destroy(ShemsReplay* rp) {
  if (!rp) return SHEMS_OK;
  GUARD(rp->device);
  for (int i = 0; i < rp->n_src; ++i) cudaFree(rp->src[i].rows);
  cudaFree(rp->alloc); cudaFree(rp->prio_alloc); cudaFree(rp->idx_scratch); cudaFree(rp->minmax_scratch); cudaFree(rp->group_refs);
  delete rp;
  return SHEMS_OK;
}
extern "C" int32_t replay_set_stream(ShemsReplay* rp, void* s) {
  REQUIRE(rp, SHEMS_ERR_INVALID, "replay_set_stream: NULL handle");
  rp->stream = (cudaStream_t)s;
  return SHEMS_OK;
}
extern "C" int64_t replay_length(const ShemsReplay* rp) { return rp ? rp->length : 0; }
extern "C" int64_t replay_capacity(const ShemsReplay* rp) { return rp ? rp->capacity : 0; }
extern "C" int64_t replay_head(const ShemsReplay* rp) { return rp ? rp->head : 0; }
extern "C" int32_t replay_series_count(const ShemsReplay* rp) { return rp ? rp->n_src : 0; }

// ---- priorities (ring.cuh: the sum tree)
// One launch rebuilds the tree after leaves changed.  Block c owns the chunk of `sub` = min(P2, PRIO_SUB) slots from c * sub: with
// m >= 0 it gives the slots (s0 + i) mod cap, i < m, that fall in its chunk the leaf p_max and recomputes the chunk's subtree; with
// m < 0 it recomputes every chunk's subtree from the leaves as they are.  The last block to arrive recomputes the nodes above the
// chunk roots.
#define PRIO_SUB 1024
#define PRIO_THREADS 512
__global__ void __launch_bounds__(PRIO_THREADS)
replay_prio_refresh_kernel(float* __restrict__ tree, long long p2, long long cap, long long s0, long long m) {
  const long long sub = p2 < PRIO_SUB ? p2 : PRIO_SUB;
  const long long first = (long long)blockIdx.x * sub, last = first + sub < cap ? first + sub : cap;
  const long long end1 = s0 + m < cap ? s0 + m : cap;   // the written slots are [s0, end1) and, after a wrap, [0, s0 + m - cap)
  const bool touched = m < 0 || (first < end1 && s0 < last) || (s0 + m > cap && first < s0 + m - cap);
  if (touched) {
    if (m >= 0) {
      const float pmax = prio_header(tree)[PRIO_PMAX];
      for (long long s = first + threadIdx.x; s < last; s += blockDim.x) {
        long long d = s - s0;
        if (d < 0) d += cap;
        if (d < m) tree[p2 + s] = pmax;
      }
    }
    long long lo = p2 + first;
    for (long long width = sub >> 1; width >= 1; width >>= 1) {
      __syncthreads();
      lo >>= 1;
      for (long long t = threadIdx.x; t < width; t += blockDim.x) tree[lo + t] = __fadd_rn(tree[2 * (lo + t)], tree[2 * (lo + t) + 1]);
    }
  }
  __shared__ bool last_block;
  __syncthreads();
  unsigned* arrived = reinterpret_cast<unsigned*>(prio_header(tree) + PRIO_ARRIVED);
  if (threadIdx.x == 0) {
    __threadfence();
    last_block = atomicAdd(arrived, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last_block) return;
  __threadfence();
  long long lo = p2 / sub;   // the chunk roots are nodes p2/sub .. 2 p2/sub - 1
  for (long long width = lo >> 1; width >= 1; width >>= 1) {
    lo >>= 1;
    for (long long t = threadIdx.x; t < width; t += blockDim.x) tree[lo + t] = __fadd_rn(__ldcg(tree + 2 * (lo + t)), __ldcg(tree + 2 * (lo + t) + 1));
    __syncthreads();
  }
  if (threadIdx.x == 0) *arrived = 0u;
}

static int prio_refresh(ShemsReplay* rp, long long s0, long long m, cudaStream_t st) {
  const long long sub = rp->prio_p2 < PRIO_SUB ? rp->prio_p2 : PRIO_SUB;
  replay_prio_refresh_kernel<<<(unsigned)((rp->capacity + sub - 1) / sub), PRIO_THREADS, 0, st>>>(rp->prio, rp->prio_p2, rp->capacity, s0, m);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

int replay_after_rollout(ShemsReplay* rp, int64_t n_written, cudaStream_t st) {
  const int64_t m = n_written < rp->capacity ? n_written : rp->capacity;   // the slots that survive the push
  const int64_t s0 = (rp->head + n_written - m) % rp->capacity;
  rp->head = (rp->head + n_written) % rp->capacity;
  rp->length = rp->length + n_written > rp->capacity ? rp->capacity : rp->length + n_written;
  if (rp->prio && m > 0) return prio_refresh(rp, s0, m, st);
  return SHEMS_OK;
}

extern "C" int32_t replay_enable_priorities(ShemsReplay* rp) {
  REQUIRE(rp, SHEMS_ERR_INVALID, "replay_enable_priorities: NULL handle");
  if (rp->prio) return SHEMS_OK;
  GUARD(rp->device);
  const size_t floats = prio_alloc_floats(rp->capacity);
  CUDA_TRY(cudaStreamSynchronize(rp->stream));
  CUDA_TRY(cudaMalloc(&rp->prio_alloc, sizeof(float) * floats));
  rp->prio = rp->prio_alloc + PRIO_HEADER_FLOATS;
  rp->prio_p2 = prio_p2(rp->capacity);
  const float pmax = 1.0f;
  CUDA_TRY(cudaMemsetAsync(rp->prio_alloc, 0, sizeof(float) * floats, rp->stream));
  CUDA_TRY(cudaMemcpyAsync(rp->prio_alloc + PRIO_PMAX, &pmax, sizeof(float), cudaMemcpyHostToDevice, rp->stream));
  TRY_PRIO(prio_refresh(rp, ring_slot(0, rp->head, rp->length, rp->capacity), rp->length, rp->stream));   // every filled slot gets p_max
  CUDA_TRY(cudaStreamSynchronize(rp->stream));   // &pmax is on this stack frame
  return SHEMS_OK;
}

extern "C" int32_t replay_get_priorities(ShemsReplay* rp, float* prio_host, float* p_max) {
  REQUIRE(rp && prio_host && p_max, SHEMS_ERR_INVALID, "replay_get_priorities: NULL argument");
  REQUIRE(rp->prio, SHEMS_ERR_STATE, "replay_get_priorities: the memory has no priorities (replay_enable_priorities)");
  GUARD(rp->device);
  const int64_t cap = rp->capacity, len = rp->length;
  std::vector<float> leaves((size_t)cap);
  CUDA_TRY(cudaStreamSynchronize(rp->stream));
  CUDA_TRY(cudaMemcpy(leaves.data(), rp->prio + rp->prio_p2, sizeof(float) * (size_t)cap, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(p_max, rp->prio_alloc + PRIO_PMAX, sizeof(float), cudaMemcpyDeviceToHost));
  for (int64_t i = 0; i < len; ++i) prio_host[i] = leaves[(size_t)ring_slot(i, rp->head, len, cap)];
  return SHEMS_OK;
}

extern "C" int32_t replay_set_priorities(ShemsReplay* rp, const float* prio_host, float p_max) {
  REQUIRE(rp && prio_host, SHEMS_ERR_INVALID, "replay_set_priorities: NULL argument");
  REQUIRE(rp->prio, SHEMS_ERR_STATE, "replay_set_priorities: the memory has no priorities (replay_enable_priorities)");
  REQUIRE(isfinite(p_max) && p_max > 0.0f, SHEMS_ERR_INVALID, "replay_set_priorities: p_max=%g must be finite and > 0", (double)p_max);
  const int64_t cap = rp->capacity, len = rp->length;
  bool mass = false;
  for (int64_t i = 0; i < len; ++i) {
    REQUIRE(isfinite(prio_host[i]) && prio_host[i] >= 0.0f, SHEMS_ERR_INVALID, "replay_set_priorities: prio[%lld]=%g must be finite and >= 0",
            (long long)i, (double)prio_host[i]);
    mass = mass || prio_host[i] > 0.0f;
  }
  REQUIRE(mass || len == 0, SHEMS_ERR_INVALID, "replay_set_priorities: every priority is 0 (nothing could be drawn)");
  GUARD(rp->device);
  std::vector<float> leaves((size_t)rp->prio_p2, 0.0f);
  for (int64_t i = 0; i < len; ++i) leaves[(size_t)ring_slot(i, rp->head, len, cap)] = prio_host[i];
  CUDA_TRY(cudaMemcpyAsync(rp->prio + rp->prio_p2, leaves.data(), sizeof(float) * leaves.size(), cudaMemcpyHostToDevice, rp->stream));
  CUDA_TRY(cudaMemcpyAsync(rp->prio_alloc + PRIO_PMAX, &p_max, sizeof(float), cudaMemcpyHostToDevice, rp->stream));
  TRY_PRIO(prio_refresh(rp, 0, -1, rp->stream));
  CUDA_TRY(cudaStreamSynchronize(rp->stream));   // the host sources live on this stack frame
  return SHEMS_OK;
}

// the B draws and importance weights of update 0 of ddpg_update(seed) on this memory: one block (the weights are normalised by the
// largest of the B)
#define PRIO_SAMPLE_THREADS 1024
__global__ void __launch_bounds__(PRIO_SAMPLE_THREADS)
replay_sample_prioritized_kernel(const float* __restrict__ tree, long long p2, long long cap, long long head, long long len, unsigned long long seed,
                                 int B, float beta, int32_t* __restrict__ idx, float* __restrict__ w) {
  __shared__ double red[PRIO_SAMPLE_THREADS / 32];
  const float root = tree[1];
  double wmax = 0.0;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    float leaf;
    const long long slot = ring_draw_prioritized(tree, p2, seed, (uint64_t)j, 0u, B, &leaf);
    idx[j] = (int32_t)ring_logical(slot, head, len, cap);
    w[j] = leaf;   // the same thread turns it into the weight below
    wmax = fmax(wmax, ring_is_weight(leaf, len, root, beta));
  }
  for (int o = 16; o > 0; o >>= 1) wmax = fmax(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = wmax;
  __syncthreads();
  wmax = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) wmax = fmax(wmax, red[i]);
  for (int j = threadIdx.x; j < B; j += blockDim.x) w[j] = (float)(ring_is_weight(w[j], len, root, beta) / wmax);
}

extern "C" int32_t replay_sample_prioritized(ShemsReplay* rp, int32_t batch, uint64_t seed, float beta, int32_t* idx_dev, float* w_dev) {
  REQUIRE(rp && idx_dev && w_dev, SHEMS_ERR_INVALID, "replay_sample_prioritized: NULL argument");
  REQUIRE(batch >= 1, SHEMS_ERR_INVALID, "replay_sample_prioritized: batch=%d", batch);
  REQUIRE(isfinite(beta) && beta >= 0.0f && beta <= 1.0f, SHEMS_ERR_INVALID, "replay_sample_prioritized: beta=%g outside [0, 1]", (double)beta);
  REQUIRE(rp->prio, SHEMS_ERR_STATE, "replay_sample_prioritized: the memory has no priorities (replay_enable_priorities)");
  REQUIRE(rp->length > 0, SHEMS_ERR_STATE, "replay_sample_prioritized: memory is empty");
  GUARD(rp->device);
  replay_sample_prioritized_kernel<<<1, PRIO_SAMPLE_THREADS, 0, rp->stream>>>(rp->prio, rp->prio_p2, rp->capacity, rp->head, rp->length, seed, batch,
                                                                             beta, idx_dev, w_dev);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

int replay_series_entry(ShemsReplay* rp, unsigned long long serial, int series, const float4* rows_dev, int nrows, cudaStream_t user,
                        int* entry) {
  for (int i = 0; i < rp->n_src; ++i)
    if (rp->src[i].env_serial == serial && rp->src[i].series == series) { *entry = i; return SHEMS_OK; }
  *entry = -1;
  if (rp->n_src == RING_MAX_SERIES) return SHEMS_OK;
  const int i = rp->n_src;
  float* rows = nullptr;
  CUDA_TRY(cudaMalloc(&rows, sizeof(float) * 8 * (size_t)nrows));
  rp->src[i].env_serial = serial; rp->src[i].series = series; rp->src[i].nrows = nrows; rp->src[i].rows = rows;
  rp->src_ptrs[i] = rows;
  rp->n_src = i + 1;
  CUDA_TRY(cudaMemcpyAsync(rows, rows_dev, sizeof(float) * 8 * (size_t)nrows, cudaMemcpyDeviceToDevice, rp->stream));
  CUDA_TRY(cudaMemcpyAsync((void*)(ring_table(rp->ring) + i), &rp->src_ptrs[i], sizeof(float*), cudaMemcpyHostToDevice, rp->stream));
  if (user != rp->stream) {  // the records that will point at the copy are written on `user`: order them after it
    cudaEvent_t ev;
    CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t st = cudaEventRecord(ev, rp->stream);
    if (st == cudaSuccess) st = cudaStreamWaitEvent(user, ev, 0);
    cudaEventDestroy(ev);
    CUDA_TRY(st);
  }
  *entry = i;
  return SHEMS_OK;
}

// remember() for n transitions: slot = (head + i) mod cap.  When n > cap only the last cap survive.
__global__ void __launch_bounds__(256)
replay_push_kernel(float* __restrict__ ring, long long cap, long long head, const float* __restrict__ s, const float* __restrict__ a,
                   const float* __restrict__ r, const float* __restrict__ s2, const float* __restrict__ done, long long n, long long first) {
  const long long i = first + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float* q = ring + ring_base(ring_push_slot(head, i, cap));
  float si[9], s2i[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { si[k] = s[k * n + i]; s2i[k] = s2[k * n + i]; }
  ring_store_full(q, si, a[i], a[n + i], r[i], s2i, done ? done[i] : 0.0f);
}

extern "C" int32_t replay_push(ShemsReplay* rp, const float* s_dev, const float* a_dev, const float* r_dev, const float* s2_dev,
                               const float* done_dev, int64_t n) {
  REQUIRE(rp && s_dev && a_dev && r_dev && s2_dev, SHEMS_ERR_INVALID, "replay_push: NULL argument");
  REQUIRE(n >= 0, SHEMS_ERR_INVALID, "replay_push: n=%lld", (long long)n);
  if (n == 0) return SHEMS_OK;
  GUARD(rp->device);
  // only the newest `cap` of the n transitions can survive; skipping the rest also keeps slots single-writer
  const int64_t first = n > rp->capacity ? n - rp->capacity : 0;
  const int64_t cnt = n - first;
  replay_push_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, rp->stream>>>(rp->ring, rp->capacity, rp->head, s_dev, a_dev, r_dev, s2_dev,
                                                                           done_dev, n, first);
  CUDA_TRY(cudaGetLastError());
  return replay_after_rollout(rp, n, rp->stream);
}

// remember() for a population: arrays are SoA over all N = P*n_per instances, learner l = instances l*n_per .. l*n_per+n_per-1
// pushes its slice into its own ring (blockIdx.y = learner)
struct RingRef { float* ring; long long cap, head; };
__global__ void __launch_bounds__(256)
replay_push_groups_kernel(const RingRef* __restrict__ refs, const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ r,
                          const float* __restrict__ s2, const float* __restrict__ done, long long n_per, long long N) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_per) return;
  const RingRef ref = refs[blockIdx.y];
  const long long g = (long long)blockIdx.y * n_per + i;  // global instance
  float* q = ref.ring + ring_base(ring_push_slot(ref.head, i, ref.cap));
  float sg[9], s2g[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { sg[k] = s[k * N + g]; s2g[k] = s2[k * N + g]; }
  ring_store_full(q, sg, a[g], a[N + g], r[g], s2g, done ? done[g] : 0.0f);
}

extern "C" int32_t replay_push_groups(ShemsReplay* const* rps, int32_t n_groups, const float* s_dev, const float* a_dev, const float* r_dev,
                                      const float* s2_dev, const float* done_dev, int64_t n_per) {
  REQUIRE(rps && s_dev && a_dev && r_dev && s2_dev, SHEMS_ERR_INVALID, "replay_push_groups: NULL argument");
  REQUIRE(n_groups >= 1 && n_per >= 1, SHEMS_ERR_INVALID, "replay_push_groups: n_groups=%d n_per=%lld", n_groups, (long long)n_per);
  ShemsReplay* r0 = rps[0];
  REQUIRE(r0, SHEMS_ERR_INVALID, "replay_push_groups: rps[0] is NULL");
  GUARD(r0->device);
  std::vector<RingRef> refs((size_t)n_groups);
  for (int g = 0; g < n_groups; ++g) {
    ShemsReplay* rp = rps[g];
    REQUIRE(rp && rp->device == r0->device, SHEMS_ERR_INVALID, "replay_push_groups: rps[%d] missing or on another device", g);
    REQUIRE(n_per <= rp->capacity, SHEMS_ERR_INVALID, "replay_push_groups: n_per=%lld exceeds the capacity %lld of rps[%d]", (long long)n_per,
            (long long)rp->capacity, g);
    refs[g].ring = rp->ring; refs[g].cap = rp->capacity; refs[g].head = rp->head;
  }
  if (r0->group_refs_n < n_groups) {
    CUDA_TRY(cudaStreamSynchronize(r0->stream));
    cudaFree(r0->group_refs); r0->group_refs = nullptr; r0->group_refs_n = 0;
    CUDA_TRY(cudaMalloc(&r0->group_refs, sizeof(RingRef) * (size_t)n_groups));
    r0->group_refs_n = n_groups;
  }
  CUDA_TRY(cudaMemcpyAsync(r0->group_refs, refs.data(), sizeof(RingRef) * (size_t)n_groups, cudaMemcpyHostToDevice, r0->stream));
  replay_push_groups_kernel<<<dim3((unsigned)((n_per + 255) / 256), n_groups), 256, 0, r0->stream>>>((const RingRef*)r0->group_refs, s_dev, a_dev,
                                                                                                r_dev, s2_dev, done_dev, n_per,
                                                                                                n_per * n_groups);
  CUDA_TRY(cudaGetLastError());
  for (int g = 0; g < n_groups; ++g) TRY_PRIO(replay_after_rollout(rps[g], n_per, r0->stream));
  return SHEMS_OK;
}

// getData(): gather B sampled transitions into SoA minibatch arrays [k][B].
// idx != NULL: logical indices; else ring_draw(seed, j, update).
__global__ void __launch_bounds__(128)
replay_sample_kernel(const float* __restrict__ ring, long long cap, long long head, long long len, const int32_t* __restrict__ idx,
                     unsigned long long seed, unsigned update, int B, float* __restrict__ s, float* __restrict__ a, float* __restrict__ r,
                     float* __restrict__ s2, float* __restrict__ done) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= B) return;
  const long long li = idx ? idx[j] : ring_draw(seed, j, update, len);
  const float* q = ring + ring_base(ring_slot(li, head, len, cap));
  const float* row = ring_row(ring_table(ring), q);
#pragma unroll
  for (int k = 0; k < 9; ++k) { s[k * B + j] = ring_field(q, row, RING_S + k); s2[k * B + j] = ring_field(q, row, RING_S2 + k); }
  a[j] = ring_field(q, row, RING_A);
  a[B + j] = ring_field(q, row, RING_A + 1);
  r[j] = ring_field(q, row, RING_R);
  done[j] = ring_field(q, row, RING_DONE);
}

static int ensure_idx_scratch(ShemsReplay* rp, int64_t n) {
  if (rp->idx_scratch_n >= n) return SHEMS_OK;
  cudaFree(rp->idx_scratch);
  rp->idx_scratch = nullptr; rp->idx_scratch_n = 0;
  CUDA_TRY(cudaMalloc(&rp->idx_scratch, sizeof(int32_t) * (size_t)n));
  rp->idx_scratch_n = n;
  return SHEMS_OK;
}

extern "C" int32_t replay_sample(ShemsReplay* rp, int32_t batch, const int32_t* idx_host, uint64_t seed, float* s_dev, float* a_dev,
                                 float* r_dev, float* s2_dev, float* done_dev) {
  REQUIRE(rp && s_dev && a_dev && r_dev && s2_dev && done_dev, SHEMS_ERR_INVALID, "replay_sample: NULL argument");
  REQUIRE(batch >= 1, SHEMS_ERR_INVALID, "replay_sample: batch=%d", batch);
  REQUIRE(rp->length > 0, SHEMS_ERR_STATE, "replay_sample: memory is empty (sample from an empty collection)");
  GUARD(rp->device);
  const int32_t* didx = nullptr;
  if (idx_host) {
    for (int j = 0; j < batch; ++j)
      REQUIRE(idx_host[j] >= 0 && idx_host[j] < rp->length, SHEMS_ERR_INVALID, "replay_sample: idx[%d]=%d outside 0..%lld", j, idx_host[j],
              (long long)rp->length - 1);
    int st = ensure_idx_scratch(rp, batch);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(rp->idx_scratch, idx_host, sizeof(int32_t) * batch, cudaMemcpyHostToDevice, rp->stream));
    didx = rp->idx_scratch;
  }
  replay_sample_kernel<<<(batch + 127) / 128, 128, 0, rp->stream>>>(rp->ring, rp->capacity, rp->head, rp->length, didx, seed, 0u, batch,
                                                                   s_dev, a_dev, r_dev, s2_dev, done_dev);
  CUDA_TRY(cudaGetLastError());
  if (idx_host) CUDA_TRY(cudaStreamSynchronize(rp->stream));  // idx_host was staged asynchronously
  return SHEMS_OK;
}

// min_max_buffer(): min/max of the 9 state fields over a with-replacement sample of n draws.
// Float min/max are exact and order-independent -> atomics on the int-ordered bit pattern.
__device__ __forceinline__ void atomic_minf(float* addr, float v) {
  if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_maxf(float* addr, float v) {
  if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}
__global__ void __launch_bounds__(256)
replay_minmax_kernel(const float* __restrict__ ring, long long cap, long long head, long long len, const int32_t* __restrict__ idx,
                     unsigned long long seed, long long n, float* __restrict__ out /* [0..8]=min, [9..17]=max */) {
  float mn[9], mx[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { mn[k] = INFINITY; mx[k] = -INFINITY; }
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const long long li = idx ? idx[j] : ring_draw(seed, j, 0u, len);
    const float* q = ring + ring_base(ring_slot(li, head, len, cap));
    const float* row = ring_row(ring_table(ring), q);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const float v = ring_field(q, row, RING_S + k);
      mn[k] = fminf(mn[k], v); mx[k] = fmaxf(mx[k], v);
    }
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
      mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
    }
    if ((threadIdx.x & 31) == 0) { atomic_minf(out + k, mn[k]); atomic_maxf(out + 9 + k, mx[k]); }
  }
}

extern "C" int32_t replay_minmax(ShemsReplay* rp, int64_t n_samples, const int32_t* idx_host, uint64_t seed, float* s_min_host, float* s_max_host) {
  REQUIRE(rp && s_min_host && s_max_host, SHEMS_ERR_INVALID, "replay_minmax: NULL argument");
  REQUIRE(n_samples >= 1, SHEMS_ERR_INVALID, "replay_minmax: n_samples=%lld", (long long)n_samples);
  REQUIRE(rp->length > 0, SHEMS_ERR_STATE, "replay_minmax: memory is empty");
  GUARD(rp->device);
  const int32_t* didx = nullptr;
  if (idx_host) {
    for (int64_t j = 0; j < n_samples; ++j)
      REQUIRE(idx_host[j] >= 0 && idx_host[j] < rp->length, SHEMS_ERR_INVALID, "replay_minmax: idx[%lld]=%d outside 0..%lld", (long long)j,
              idx_host[j], (long long)rp->length - 1);
    int st = ensure_idx_scratch(rp, n_samples);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(rp->idx_scratch, idx_host, sizeof(int32_t) * (size_t)n_samples, cudaMemcpyHostToDevice, rp->stream));
    didx = rp->idx_scratch;
  }
  float init[18];
  for (int k = 0; k < 9; ++k) { init[k] = INFINITY; init[9 + k] = -INFINITY; }
  CUDA_TRY(cudaMemcpyAsync(rp->minmax_scratch, init, sizeof(init), cudaMemcpyHostToDevice, rp->stream));
  long long blocks = (n_samples + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  replay_minmax_kernel<<<(unsigned)blocks, 256, 0, rp->stream>>>(rp->ring, rp->capacity, rp->head, rp->length, didx, seed, n_samples, rp->minmax_scratch);
  CUDA_TRY(cudaGetLastError());
  float res[18];
  CUDA_TRY(cudaMemcpyAsync(res, rp->minmax_scratch, sizeof(res), cudaMemcpyDeviceToHost, rp->stream));
  CUDA_TRY(cudaStreamSynchronize(rp->stream));
  memcpy(s_min_host, res, sizeof(float) * 9);
  memcpy(s_max_host, res + 9, sizeof(float) * 9);
  return SHEMS_OK;
}

extern "C" int32_t replay_get(ShemsReplay* rp, float* s_host, float* a_host, float* r_host, float* s2_host, float* done_host) {
  REQUIRE(rp, SHEMS_ERR_INVALID, "replay_get: NULL handle");
  GUARD(rp->device);
  const int64_t len = rp->length, cap = rp->capacity;
  if (len == 0) return SHEMS_OK;
  CUDA_TRY(cudaStreamSynchronize(rp->stream));
  std::vector<float> host(ring_alloc_floats(cap));
  CUDA_TRY(cudaMemcpy(host.data(), rp->alloc, sizeof(float) * host.size(), cudaMemcpyDeviceToHost));
  const float* ring = ring_in_alloc(host.data());
  std::vector<std::vector<float>> rows((size_t)rp->n_src);  // host copies of the series table of the compact records
  std::vector<const float*> table((size_t)rp->n_src);
  for (int e = 0; e < rp->n_src; ++e) {
    rows[e].resize((size_t)8 * rp->src[e].nrows);
    CUDA_TRY(cudaMemcpy(rows[e].data(), rp->src[e].rows, sizeof(float) * rows[e].size(), cudaMemcpyDeviceToHost));
    table[e] = rows[e].data();
  }
  for (int64_t i = 0; i < len; ++i) {  // logical order, oldest first
    const float* q = ring + ring_base(ring_slot(i, rp->head, len, cap));
    const float* row = ring_row(table.data(), q);
    for (int k = 0; k < 9; ++k) {
      if (s_host) s_host[(size_t)k * len + i] = ring_field(q, row, RING_S + k);
      if (s2_host) s2_host[(size_t)k * len + i] = ring_field(q, row, RING_S2 + k);
    }
    if (a_host) { a_host[i] = ring_field(q, row, RING_A); a_host[(size_t)len + i] = ring_field(q, row, RING_A + 1); }
    if (r_host) r_host[i] = ring_field(q, row, RING_R);
    if (done_host) done_host[i] = ring_field(q, row, RING_DONE);
  }
  return SHEMS_OK;
}
