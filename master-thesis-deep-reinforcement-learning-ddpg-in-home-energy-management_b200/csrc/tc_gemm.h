// tc_gemm.h — TF32 tcgen05 GEMM used by the large-batch DDPG update (csrc/tc_gemm.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

enum { TC_EPI_NONE = 0, TC_EPI_BIAS_RELU = 1, TC_EPI_RELU_MASK = 2 };

struct TcOperand {
  const float* ptr;
  long long ld;      // floats between consecutive rows (K-major) or consecutive k (MN-major)
  bool mn_major;     // false: (row, k) at ptr[row*ld + k]; true: (row, k) at ptr[k*ld + row]
};
#define TC_MAX_PROBLEMS 3
struct TcGemmArgs {
  int M, N, K, splits, epi, tma_store, batch, nprob, pdl;
  float* D[TC_MAX_PROBLEMS]; long long ldd, split_stride;
  const float* bias[TC_MAX_PROBLEMS]; const float* aux[TC_MAX_PROBLEMS]; long long auxld, bs_bias, bs_aux;
};
// `count` independent products of one shape in a launch (a population of learners): strides in floats between entries
struct TcBatch {
  int count = 1;
  long long sA = 0, sB = 0, sD = 0, sBias = 0, sAux = 0;
  bool pdl = false;   // launch as a programmatic dependent of the predecessor in the stream (the kernel waits before touching its operands)
};
// D[M×N] (row-major, ldd) = epilogue(sum_k A(m,k) · B(n,k))
int tc_gemm(cudaStream_t st, const TcOperand& A, const TcOperand& B, float* D, long long ldd, int M, int N, int K, int epi,
            const float* bias, const float* aux, long long auxld, int splits, float* workspace, const TcBatch& batch = TcBatch());
// up to TC_MAX_PROBLEMS products of one shape in a single launch (e.g. the layer-2 forward passes of actor_target / critic / actor)
int tc_gemm_multi(cudaStream_t st, int nprob, const TcOperand* A, const TcOperand* B, float* const* D, long long ldd, int M, int N, int K, int epi,
                  const float* const* bias, const float* const* aux, long long auxld, int splits, float* workspace, const TcBatch& batch = TcBatch());
// sets the kernels' shared-memory attribute on the current device; call once per device before capturing launches in a graph
int tc_gemm_prepare();

// The whole forward pass of up to TC_MAX_PROBLEMS nets (same widths l1 <= 256, l2 <= 512) over a large minibatch in ONE launch:
// layer 1 (fp32 SIMT) -> layer 2 (tcgen05, TF32) -> output layer (1 or 2 units) in the epilogue; 128 rows per CTA.
enum { TC_OUT_TANH = 0, TC_OUT_ID = 1, TC_OUT_TD = 2 };
struct TcFwdChainArgs {
  int M, L1, L2, nprob, ldx, ldh1, ldh2;
  const float* X[TC_MAX_PROBLEMS]; int K1[TC_MAX_PROBLEMS];        // inputs [M][ldx] (K1 <= 12 columns used)
  const float *W1[TC_MAX_PROBLEMS], *b1[TC_MAX_PROBLEMS];          // Flux layout Wt[in][out]
  const float *W2[TC_MAX_PROBLEMS], *b2[TC_MAX_PROBLEMS];
  const float *W3[TC_MAX_PROBLEMS], *b3[TC_MAX_PROBLEMS]; int J[TC_MAX_PROBLEMS];
  float* H1[TC_MAX_PROBLEMS];                                      // [M][ldh1] layer-1 activations, or NULL (target nets: no backward pass)
  float* H2[TC_MAX_PROBLEMS];                                      // [M][ldh2] layer-2 activations, or NULL
  int out_mode[TC_MAX_PROBLEMS]; float* out[TC_MAX_PROBLEMS]; int ldo[TC_MAX_PROBLEMS];   // out[row*ldo + j]
  const float *td_r, *td_done, *td_q; float* td_dq; float inv_batch;                      // TC_OUT_TD
  const float* td_gamma; long long td_gamma_stride;   // TC_OUT_TD: γ of learner l at td_gamma[l * td_gamma_stride] (its DDPG control block)
  int nsplit;                      // 2: a cluster of two CTAs per row tile, half of the layer-2 units each (for launches with few row tiles)
  int pdl, early_weights;          // programmatic dependent launch; early_weights: the predecessor in the stream did not write the net's weights
  int pop; long long pop_stride;   // a population of learners (grid.y): every pointer above moves by pop_stride floats per learner
};
int tc_fwd_chain(cudaStream_t st, const TcFwdChainArgs& a);

// The backward pass of a net from its output layer down to layer 1 (the dX chain) for a large minibatch in ONE launch, 128 rows per CTA:
//   dz2 = (dout W3^T) masked by relu'(h2)        fp32 SIMT, in place on the TMA-loaded h2 tile = the tcgen05 A operand (optionally stored: DZ2)
//   dz1 = (dz2 W2^T) masked by relu'(h1)         tcgen05, TF32 (optionally stored: DZ1)
//   dA  = (dz1 W1[rows 9, 10]^T) (1 - a^2)       in the epilogue (critic inside the actor loss: the gradient w.r.t. the action inputs)
struct TcBwdChainArgs {
  int M, L1, L2, J, ldh1, ldh2, pdl;
  int nsplit;             // 2: two CTAs per row tile, half of the layer-1 units each (dA must be zero on entry: the halves add their shares)
  const float* dout;      // [M][J] gradient w.r.t. the net's output (J = 1 or 2)
  const float* W3;        // Flux layout [L2][J]
  const float* W2;        // Flux layout [L1][L2]
  const float* H2;        // [M][ldh2]
  const float* H1;        // [M][ldh1]
  float* DZ2;             // [M][ldh2] or NULL
  float* DZ1;             // [M][ldh1] or NULL
  const float* W1a;       // W1 rows of the two action inputs ([2][L1], row stride L1) or NULL
  const float* act;       // a = tanh output [M] rows, 2 columns, row stride ld_act
  float* dA;              // [M][2]
  int ld_act;
  int pop; long long pop_stride;
};
int tc_bwd_chain(cudaStream_t st, const TcBwdChainArgs& a);
