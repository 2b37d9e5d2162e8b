// surya_b200 — epilogue shared by the tcgen05 GEMM and implicit-GEMM convolution kernels.
// One call handles the 32 accumulator columns a thread just pulled from TMEM for its output row.
#pragma once
#include "gemm.cuh"
#include "sb_ptx.cuh"

namespace sb {

struct GemmKParams {
  int M, N, K;
  void* C;
  int ldc;
  const float* bias;
  const void* residual;
  int ldr;
  int act;
  int swiglu;
  int out_f32;
  int group_m;
  int group_k;  // grouped 1x1 conv: A column offset per n-block (0 = dense)
  int w_constant;  // W tiles may be fetched before the programmatic-dependency wait
  // RMSNorm folded into the GEMM (decoder layers, DESIGN.md §4): C = epi(rowscale[m] * (A W'^T) + bias) with W' = W * g and
  // rowscale = rsqrt(mean_k(A[m,k]^2) + eps), either read from global (prefill: row_rstd kernel) or computed by the epilogue
  // warps from the A stages while the main loop runs (ssq_inline: decode steps, no extra launch)
  const float* rowscale;
  int ssq_inline;
  float ssq_eps, ssq_inv_k;
  // lm_head with an online (max, argmax, sum exp) epilogue: per (row, n-tile) partials, logits never reach HBM unless
  // store_c is set (surya/recognition/__init__.py:294-324 needs argmax + max softmax only)
  float* am_val;
  int* am_idx;
  float* am_sum;
  int am_ld;
  int store_c;
  unsigned long long* dbg;  // optional timeline buffer (globaltimer ns) written by CTA 0: [0]=start [1]=setup done
                            // [2+kb]=k-block kb landed (first tile) [40]=accumulator ready [41]=epilogue done
};

__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case ACT_GELU_ERF: return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
    case ACT_SILU: return x / (1.0f + expf(-x));
    case ACT_HARDSWISH: return x * fminf(fmaxf(x + 3.0f, 0.0f), 6.0f) / 6.0f;
    case ACT_RELU: return fmaxf(x, 0.0f);
    case ACT_GELU_TANH: {
      const float k0 = 0.7978845608028654f, k1 = 0.044715f;
      float inner = k0 * (x + k1 * x * x * x);
      return 0.5f * x * (1.0f + tanhf(inner));
    }
    default: return x;
  }
}


// x = acc (+bias) -> round -> act -> round (+residual) -> round -> store; `row` is the global output row
// (already translated to an NHWC pixel index by the convolution kernel), `col0` the first of 32 columns.
template <typename T>
__device__ __noinline__ void epilogue_chunk(const uint32_t (&v)[32], const GemmKParams& p, int row, bool row_ok,
                                               int col0, bool vec_ok) {
  float x[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]);
  if (p.bias) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (col0 + j < p.N) x[j] += __ldg(p.bias + col0 + j);
    }
  }
  if (!row_ok) return;
  if (p.swiglu) {
    // columns (2i, 2i+1) = (gate_i, up_i)
    const int oc0 = col0 >> 1;
    const int n_out = p.N >> 1;
    T* crow = reinterpret_cast<T*>(p.C) + static_cast<size_t>(row) * p.ldc;
    T o[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float g = rnd<T>(x[2 * i]);
      float u = rnd<T>(x[2 * i + 1]);
      float sact = rnd<T>(apply_act(g, p.act));
      o[i] = from_f<T>(sact * u);
    }
    if (vec_ok && oc0 + 16 <= n_out) {
      uint4* dst = reinterpret_cast<uint4*>(crow + oc0);
      const uint4* src = reinterpret_cast<const uint4*>(o);
      dst[0] = src[0];
      dst[1] = src[1];
    } else {
      for (int i = 0; i < 16; ++i)
        if (oc0 + i < n_out) crow[oc0 + i] = o[i];
    }
  } else if (p.out_f32) {
    float* crow = reinterpret_cast<float*>(p.C) + static_cast<size_t>(row) * p.ldc;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float y = apply_act(x[j], p.act);
      if (col0 + j < p.N) crow[col0 + j] = y;
    }
  } else {
    T* crow = reinterpret_cast<T*>(p.C) + static_cast<size_t>(row) * p.ldc;
    const T* rrow = p.residual ? reinterpret_cast<const T*>(p.residual) + static_cast<size_t>(row) * p.ldr : nullptr;
    const bool full = (col0 + 32 <= p.N) && vec_ok;
    T r[32];
    if (rrow) {
      if (full) {
        const uint4* src = reinterpret_cast<const uint4*>(rrow + col0);
        uint4* dst = reinterpret_cast<uint4*>(r);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[i] = src[i];
      } else {
        for (int j = 0; j < 32; ++j) r[j] = (col0 + j < p.N) ? rrow[col0 + j] : from_f<T>(0.f);
      }
    }
    T o[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float y = rnd<T>(x[j]);
      if (p.act != ACT_NONE) y = rnd<T>(apply_act(y, p.act));
      if (rrow) y = y + to_f<T>(r[j]);
      o[j] = from_f<T>(y);
    }
    if (full) {
      uint4* dst = reinterpret_cast<uint4*>(crow + col0);
      const uint4* src = reinterpret_cast<const uint4*>(o);
#pragma unroll
      for (int i = 0; i < 4; ++i) dst[i] = src[i];
    } else {
      for (int j = 0; j < 32; ++j)
        if (col0 + j < p.N) crow[col0 + j] = o[j];
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Tile epilogue (8 warps): TMEM -> registers -> packed 16-bit math -> swizzled per-warp staging -> coalesced global.
//
// History (profiles/r01_gemm_prefill_ncu.md, tools/gemm_timeline.py): the first epilogue (epilogue_chunk above, kept as
// the generic fallback) was instruction-fetch bound and took 30-40 us per 128x256 tile; staging + compile-time
// activation brought it to 12.6 us, still longer than the 8.4 us main loop.  This version
//   * runs on 8 warps (two per TMEM lane quarter, alternating 64/32-column groups) so each SM sub-partition has two
//     epilogue warps to interleave;
//   * stages the tile's bias slice in shared memory once, before the accumulator is ready (overlaps the main loop);
//   * keeps the per-element instruction count minimal: packed cvt (cvt.rn.bf16x2.f32 / f16x2), one rounding per eager
//     op boundary, residual fetched with coalesced 16-byte loads issued before the TMEM load they overlap with;
//   * moves every global byte as part of a 64/128-byte row segment (XOR-swizzled staging, conflict-free).
// Requires ldc % 8 == 0, ldr % 8 == 0, N % 8 == 0 (N % 16 == 0 and act == silu with SwiGLU), 16-bit output.
constexpr int EPI_WARPS = 8;
constexpr int EPI_STAGE_BYTES = 32 * 128;                       // per warp: 32 rows x 128 B (swizzled, no padding)
constexpr int EPI_ROWSCALE_BYTES = 128 * 4;                     // per-row 1/rms of the tile's 128 rows (folded RMSNorm)
template <int BN> constexpr int epi_smem_bytes() { return EPI_WARPS * EPI_STAGE_BYTES + BN * 4 + EPI_ROWSCALE_BYTES; }

__device__ __forceinline__ bool epilogue_v2_ok(const GemmKParams& p) {
  if (p.out_f32 || (p.ldc & 7) || (p.residual && (p.ldr & 7))) return false;
  if (p.swiglu) return (p.act == ACT_SILU || p.act == ACT_GELU_TANH) && p.N % 16 == 0;
  return p.N % 8 == 0;
}

template <typename T> struct Pk;
template <> struct Pk<__nv_bfloat16> {
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float lo(uint32_t u) { return __uint_as_float(u << 16); }
  static __device__ __forceinline__ float hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
};
template <> struct Pk<__half> {
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float lo(uint32_t u) { return __half2float(__ushort_as_half(static_cast<unsigned short>(u & 0xffffu))); }
  static __device__ __forceinline__ float hi(uint32_t u) { return __half2float(__ushort_as_half(static_cast<unsigned short>(u >> 16))); }
};

template <int ACT>
__device__ __forceinline__ float act_ct(float x) {
  if constexpr (ACT == ACT_GELU_ERF) return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
  else if constexpr (ACT == ACT_SILU) return x / (1.0f + __expf(-x));
  else if constexpr (ACT == ACT_HARDSWISH) return x * fminf(fmaxf(x + 3.0f, 0.0f), 6.0f) * (1.0f / 6.0f);
  else if constexpr (ACT == ACT_RELU) return fmaxf(x, 0.0f);
  else if constexpr (ACT == ACT_GELU_TANH) {
    const float inner = 0.7978845608028654f * (x + 0.044715f * x * x * x);
    return 0.5f * x * (1.0f + tanhf(inner));
  } else return x;
}

// byte offset of 16-byte chunk `ch` of staged row `row` for rows of CPR chunks (XOR swizzle, bank-conflict free)
template <int CPR>
__device__ __forceinline__ int stage_off(int row, int ch) {
  if constexpr (CPR == 8) return row * 128 + ((ch ^ (row & 7)) << 4);
  else if constexpr (CPR == 4) return row * 64 + ((ch ^ ((row >> 1) & 3)) << 4);
  else if constexpr (CPR == 2) return row * 32 + ((ch ^ ((row >> 2) & 1)) << 4);
  else return row * 16;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const int n = valid ? 16 : 0;   // src-size 0 -> zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// One warp, one tile.  taddr: TMEM address (lane quarter, first accumulator column of the tile); row_fn(r): global output
// row of the warp's r-th row or -1; n_col0: first weight row (accumulator column) of the tile; half: 0/1 = which of the two
// warps sharing this lane quarter; sbias: the tile's bias slice (BN floats, already staged, zeros when absent).
// stage: 4 KB per warp = residual sub-tile (cp.async, prefetched one group ahead) + output sub-tile, both swizzled.
template <typename T, int ACT, bool SWIGLU, typename RowFn>
__device__ __forceinline__ void epilogue_tile_ct(uint32_t taddr, const GemmKParams& p, uint8_t* stage, const float* sbias,
                                                 int lane, int half, RowFn row_fn, int n_col0, float rs, const int NG) {
  constexpr int GW = 32;                            // accumulator columns per group (one tcgen05.ld .x32); NG groups per tile
  constexpr int GWO = SWIGLU ? GW / 2 : GW;         // output columns per group
  constexpr int CPR = GWO / 8;                      // 16-byte chunks per staged row
  constexpr int ITERS = CPR;                        // 32 rows x CPR chunks / 32 lanes
  uint8_t* rstage = stage;                          // residual sub-tile
  uint8_t* ostage = stage + 2048;                   // output sub-tile
  const int n_out = SWIGLU ? (p.N >> 1) : p.N;
  T* cbase = reinterpret_cast<T*>(p.C);
  const T* rbase = SWIGLU ? nullptr : reinterpret_cast<const T*>(p.residual);
  int grow[ITERS];
  const int pch = lane % CPR;                       // idx = it*32 + lane -> the chunk is the same for every `it`
  const int prow0 = lane / CPR;                     // row = it * (32 / CPR) + lane / CPR
#pragma unroll
  for (int it = 0; it < ITERS; ++it) grow[it] = row_fn(it * (32 / CPR) + prow0);

  auto prefetch_residual = [&](int g) {
    const int ocol0 = n_col0 + g * GW;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const bool ok = grow[it] >= 0 && ocol0 + pch * 8 < n_out;
      const T* src = ok ? rbase + static_cast<size_t>(grow[it]) * p.ldr + ocol0 + pch * 8 : rbase;
      cp_async16(rstage + stage_off<CPR>(it * (32 / CPR) + prow0, pch), src, ok);
    }
  };
  if (rbase && n_col0 + half * GW < p.N) prefetch_residual(half);

#pragma unroll 1
  for (int g = half; g < NG; g += 2) {
    const int acol0 = n_col0 + g * GW;
    if (acol0 >= p.N) break;
    const int ocol0 = SWIGLU ? (acol0 >> 1) : acol0;
    uint32_t o[GWO / 2];                            // this lane's packed output row segment
    {
      uint32_t v[32];
      tmem_ld_32x32(taddr + g * GW, v);
      tmem_ld_wait();
      const float* bs = sbias + g * GW;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(bs + j);
        // rs = 1 without a folded norm: fma(acc, 1, b) == acc + b exactly, so the other callers keep their bits
        const float x0 = fmaf(__uint_as_float(v[j]), rs, b4.x), x1 = fmaf(__uint_as_float(v[j + 1]), rs, b4.y);
        const float x2 = fmaf(__uint_as_float(v[j + 2]), rs, b4.z), x3 = fmaf(__uint_as_float(v[j + 3]), rs, b4.w);
        if constexpr (SWIGLU) {
          // (x0,x1) = (gate_i, up_i), (x2,x3) = (gate_i+1, up_i+1); every eager op boundary rounds once
          const uint32_t t0 = Pk<T>::pack(x0, x1), t1 = Pk<T>::pack(x2, x3);
          const uint32_t s = Pk<T>::pack(act_ct<ACT>(Pk<T>::lo(t0)), act_ct<ACT>(Pk<T>::lo(t1)));
          o[j / 4] = Pk<T>::pack(Pk<T>::lo(s) * Pk<T>::hi(t0), Pk<T>::hi(s) * Pk<T>::hi(t1));
        } else {
          uint32_t t0 = Pk<T>::pack(x0, x1), t1 = Pk<T>::pack(x2, x3);
          if constexpr (ACT != ACT_NONE) {
            t0 = Pk<T>::pack(act_ct<ACT>(Pk<T>::lo(t0)), act_ct<ACT>(Pk<T>::hi(t0)));
            t1 = Pk<T>::pack(act_ct<ACT>(Pk<T>::lo(t1)), act_ct<ACT>(Pk<T>::hi(t1)));
          }
          o[j / 2] = t0;
          o[j / 2 + 1] = t1;
        }
      }
    }
    if (rbase) {
      cp_async_wait_all();
      __syncwarp();                                 // every lane's residual pieces have landed
#pragma unroll
      for (int ch = 0; ch < CPR; ++ch) {
        const uint4 r4 = *reinterpret_cast<const uint4*>(rstage + stage_off<CPR>(lane, ch));
        const uint32_t rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t t = o[ch * 4 + k];
          o[ch * 4 + k] = Pk<T>::pack(Pk<T>::lo(t) + Pk<T>::lo(rr[k]), Pk<T>::hi(t) + Pk<T>::hi(rr[k]));
        }
      }
      __syncwarp();                                 // residual buffer free again
      if (g + 2 < NG && n_col0 + (g + 2) * GW < p.N) prefetch_residual(g + 2);
    }
    __syncwarp();                                   // previous group's output rows have been stored
#pragma unroll
    for (int ch = 0; ch < CPR; ++ch)
      *reinterpret_cast<uint4*>(ostage + stage_off<CPR>(lane, ch)) = make_uint4(o[ch * 4], o[ch * 4 + 1], o[ch * 4 + 2], o[ch * 4 + 3]);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      if (grow[it] >= 0 && ocol0 + pch * 8 < n_out)
        *reinterpret_cast<uint4*>(cbase + static_cast<size_t>(grow[it]) * p.ldc + ocol0 + pch * 8) =
            *reinterpret_cast<const uint4*>(ostage + stage_off<CPR>(it * (32 / CPR) + prow0, pch));
    }
  }
}

// Online (max, first argmax, sum exp(x - max)) over the tile's columns for this lane's row; logits are rounded to the storage
// type first (the reference takes argmax / softmax of the 16-bit lm_head output cast to fp32).  The two warps of a lane
// quarter cover alternating 32-column groups; their partials meet in shared memory (`xch` = base of the epilogue staging blocks) and warp half 0 writes
// the (row, n-tile) partial.  Columns beyond N are skipped.
struct AmPartial { float m; int i; float s; };
__device__ __forceinline__ void am_combine(AmPartial& a, const AmPartial& b) {
  if (b.m == -INFINITY) return;
  if (a.m == -INFINITY) { a = b; return; }
  if (b.m > a.m || (b.m == a.m && b.i < a.i)) {
    a.s = a.s * __expf(a.m - b.m) + b.s;
    a.m = b.m;
    a.i = b.i;
  } else {
    a.s += b.s * __expf(b.m - a.m);
  }
}

template <typename T, int BN>
__device__ __forceinline__ void epilogue_tile_argmax(uint32_t taddr, const GemmKParams& p, uint8_t* xch, const float* sbias,
                                                     int lane, int half, int q, int row, int n_col0, int nb, float rs) {
  constexpr int GW = 32, NG = BN / GW;
  AmPartial a{-INFINITY, 0x7fffffff, 0.f};
#pragma unroll 1
  for (int g = half; g < NG; g += 2) {
    const int acol0 = n_col0 + g * GW;
    if (acol0 >= p.N) break;
    uint32_t v[32];
    tmem_ld_32x32(taddr + g * GW, v);
    tmem_ld_wait();
    const float* bs = sbias + g * GW;
    float x[32];
    float cm = -INFINITY;
    int ci = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      x[j] = rnd<T>(fmaf(__uint_as_float(v[j]), rs, bs[j]));
      if (acol0 + j < p.N && x[j] > cm) { cm = x[j]; ci = acol0 + j; }     // ascending columns: the first maximum wins
    }
    if (cm == -INFINITY) continue;
    if (cm > a.m) { a.s *= __expf(a.m - cm); a.m = cm; a.i = ci; }
    float add = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (acol0 + j < p.N) add += __expf(x[j] - a.m);
    a.s += add;
  }
  // exchange through the half-1 warp's OWN staging block (nobody else touches it, also not a store_c epilogue still draining)
  float* mine = reinterpret_cast<float*>(xch + (4 + q) * EPI_STAGE_BYTES) + lane * 3;
  if (half == 1) {
    mine[0] = a.m;
    mine[1] = __int_as_float(a.i);
    mine[2] = a.s;
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");
  if (half == 0) {
    const float* other = mine;
    AmPartial b{other[0], __float_as_int(other[1]), other[2]};
    am_combine(a, b);
    if (row >= 0) {
      const size_t o = static_cast<size_t>(row) * p.am_ld + nb;
      p.am_val[o] = a.m;
      p.am_idx[o] = a.i;
      p.am_sum[o] = a.s;
    }
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");   // xch may be reused by the next tile
}

// Sum of squares of one 128 x 64 A stage (128-byte-swizzled, K-major) for the folded RMSNorm: thread t of the 256 epilogue
// threads owns half a row (row t/2, logical 16-byte chunks 4*(t&1) .. +3, i.e. elements [32*(t&1), +32) of the k-block, in
// order — row_rstd_kernel in ops.cu adds in exactly this order, so prefill and decode agree bit for bit).
template <typename T>
__device__ __forceinline__ float ssq_stage(const uint8_t* sa, int epi_tid, float acc) {
  const int r = epi_tid >> 1, hf = epi_tid & 1;
  const uint8_t* rowp = sa + r * 128;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int phys = (hf * 4 + j) ^ (r & 7);
    const uint4 u = *reinterpret_cast<const uint4*>(rowp + phys * 16);
    const T* e = reinterpret_cast<const T*>(&u);
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const float f = to_f<T>(e[x]);
      acc = fmaf(f, f, acc);
    }
  }
  return acc;
}

// Stage the tile's bias slice (zeros when the GEMM has none); called by all epilogue threads before the accumulator wait.
template <int BN>
__device__ __forceinline__ void epilogue_stage_bias(const GemmKParams& p, float* sbias, int epi_tid, int n_col0) {
  for (int j = epi_tid; j < BN; j += EPI_WARPS * 32)
    sbias[j] = (p.bias && n_col0 + j < p.N) ? __ldg(p.bias + n_col0 + j) : 0.f;
}

// Runtime -> compile-time dispatch on (act, swiglu); once per tile, outside every loop.  ng = 32-column groups in the tile.
template <typename T, typename RowFn>
__device__ __forceinline__ void epilogue_tile_rt(uint32_t taddr, const GemmKParams& p, uint8_t* stage, const float* sbias,
                                                 int lane, int half, RowFn row_fn, int n_col0, float rs, int ng) {
  if (p.swiglu) {   // SwiGLU (Qwen2 MLPs) or GeGLU (ADETR MLP, gelu_pytorch_tanh)
    if (p.act == ACT_SILU) epilogue_tile_ct<T, ACT_SILU, true>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng);
    else epilogue_tile_ct<T, ACT_GELU_TANH, true>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng);
    return;
  }
  switch (p.act) {
    case ACT_NONE: epilogue_tile_ct<T, ACT_NONE, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
    case ACT_GELU_ERF: epilogue_tile_ct<T, ACT_GELU_ERF, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
    case ACT_HARDSWISH: epilogue_tile_ct<T, ACT_HARDSWISH, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
    case ACT_RELU: epilogue_tile_ct<T, ACT_RELU, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
    case ACT_SILU: epilogue_tile_ct<T, ACT_SILU, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
    default: epilogue_tile_ct<T, ACT_GELU_TANH, false>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, ng); break;
  }
}

template <typename T, int BN, typename RowFn>
__device__ __forceinline__ void epilogue_tile_v2(uint32_t taddr, const GemmKParams& p, uint8_t* stage, const float* sbias,
                                                 int lane, int half, RowFn row_fn, int n_col0, float rs = 1.0f) {
  epilogue_tile_rt<T>(taddr, p, stage, sbias, lane, half, row_fn, n_col0, rs, BN / 32);
}

}  // namespace sb
