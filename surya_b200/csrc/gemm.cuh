// surya_b200 — tcgen05 GEMM interface (host side). See gemm_tcgen05.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sb {

enum Act : int { ACT_NONE = 0, ACT_GELU_ERF = 1, ACT_SILU = 2, ACT_HARDSWISH = 3, ACT_RELU = 4, ACT_GELU_TANH = 5 };
enum DType : int { DT_BF16 = 0, DT_F16 = 1 };

// C[M, Nout] = epilogue( A[M,K] @ W[N,K]^T ), 16-bit in / fp32 accumulate / 16-bit out.
//   epilogue: x = acc (+ bias[n]) -> round -> act -> round (+ residual[m,n]) -> round
//   swiglu=1: weight rows are interleaved (gate_0, up_0, gate_1, up_1, ...); Nout = N/2 and
//             out[m,j] = round(round(act(g)) * u).
struct GemmArgs {
  int dtype = DT_BF16;
  const void* A = nullptr; int lda = 0;   // [M, K], row stride lda (elements), lda*2 % 16 == 0
  const void* W = nullptr; int ldw = 0;   // [N, K], row stride ldw
  void* C = nullptr;       int ldc = 0;   // [M, Nout]
  int M = 0, N = 0, K = 0;
  const float* bias = nullptr;            // [N] fp32 or null
  const void* residual = nullptr; int ldr = 0;
  int act = ACT_NONE;
  int swiglu = 0;
  int out_f32 = 0;                        // C is float32 (no final rounding) when set
  int force_bn = 0;                       // 0 = heuristic, else 32/64/96/128/256; 1000 * pk + BN forces split-K
  int allow_splitk = 0;                   // the heuristic may pick the split-K cluster kernel (changes the fp32 summation
                                          // order, so only callers whose M never crosses the 256-row limit opt in: decode steps)
  // grouped 1x1 convolution (block-diagonal weights): n-block g reads A columns [g*group_k, g*group_k + K) and
  // W rows [g*group_n, (g+1)*group_n); W is [N, K] with K the zero-padded per-group depth; a_cols = A's width.
  int group_k = 0, group_n = 0, a_cols = 0;
  int w_constant = 0;                     // W is never written by a preceding kernel: its tiles may be prefetched
                                          // before the programmatic-dependency wait (engine weights)
  unsigned long long* dbg = nullptr;      // optional in-kernel timeline (see GemmKParams::dbg)
  // RMSNorm folded into the GEMM: C = epi(rs[m] * (A W^T) + bias), W already multiplied by the norm weight.
  //   rowscale  : rs given, fp32 [M] (row_rstd in ops.cu)
  //   ssq_inline: rs = rsqrt(sum_k A[m,k]^2 / ssq_k + ssq_eps) computed inside the kernel from the A tiles
  const float* rowscale = nullptr;
  int ssq_inline = 0;
  float ssq_eps = 0.f;
  int ssq_k = 0;                          // number of real columns in the mean (0 = K)
  // online argmax / softmax-denominator epilogue: per (row, n-tile) partials [M, am_ld]; C is only written when store_c
  float* am_val = nullptr;
  int* am_idx = nullptr;
  float* am_sum = nullptr;
  int am_ld = 0;
  int store_c = 1;
};
// M <= 16 rows: mma.sync kernel without the tcgen05 set-up costs (gemm_skinny.cu); gemm_launch routes to it when it applies.
bool gemm_skinny_ok(const GemmArgs& a);
int gemm_skinny_launch(const GemmArgs& a, cudaStream_t stream);
// Tile width gemm_launch will use for an argmax-epilogue launch of this shape (partials per row = ceil(N / width)).
int gemm_argmax_tile(int M, int N);

// Returns cudaSuccess or an error; sets a message retrievable through sb_last_error().
int gemm_launch(const GemmArgs& a, cudaStream_t stream);
// split-K over a thread-block cluster (gemm_splitk.cu): plan returns the split factor (0 = use the plain kernel)
int splitk_plan(const GemmArgs& a, int* bn_out);
int gemm_splitk_launch(const GemmArgs& a, int pk, int bn, cudaStream_t stream);

void set_error(const char* fmt, ...);
const char* last_error();
// Counts one kernel launch and converts cudaGetLastError() into a return code (+ error string).
int launch_ok();
long long launch_count();
void count_launches(long long n);  // kernels replayed through a CUDA graph
int num_sms();

// Launch with the programmatic-stream-serialization attribute (PDL) unless SB_PDL=0.
bool pdl_enabled();
template <typename... P, typename... A>
inline cudaError_t launch_pdl(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}

}  // namespace sb
