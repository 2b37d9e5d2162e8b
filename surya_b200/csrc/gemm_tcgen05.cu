// surya_b200 — persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M, Nout] = epilogue(A[M, K] @ W[N, K]^T)      (torch nn.Linear layout: both operands K-major)
//
// Replaces every cuBLAS call the reference makes through nn.Linear / 1x1 Conv2d on the hot path
// (SURVEY.md §2.2 K1, K3, K5-K7, K9-K11).  Design:
//   * one CTA per SM, persistent over a grouped tile raster (A/W tiles stay L2 resident);
//   * warp 0 = TMA producer (cp.async.bulk.tensor, 128B swizzle, BK = 64 elements per stage);
//   * warp 1 = MMA issuer: tcgen05.mma kind::f16, UMMA 128 x BN x 16, fp32 accumulators in TMEM,
//     two accumulator buffers so the epilogue of tile i overlaps the main loop of tile i+1;
//   * warp 2 = TMEM allocator; warps 4-7 = epilogue (tcgen05.ld -> bias/act/residual/SwiGLU -> global).
// Rounding to the storage type happens exactly where eager PyTorch has an op boundary (after the
// Linear, after the activation, after the residual add) so results track the reference path.
#include "gemm.cuh"

#include <mutex>
#include <string>
#include <unordered_map>
#include "gemm_epilogue.cuh"
#include "sb_ptx.cuh"

#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <atomic>
#include <mutex>

namespace sb {

__device__ __forceinline__ void tile_coords(int tile, int m_blocks, int n_blocks, int gm, int& mb, int& nb) {
  int per_group = gm * n_blocks;
  int g = tile / per_group;
  int first = g * gm;
  int gsz = min(m_blocks - first, gm);
  int r = tile - g * per_group;
  mb = first + r % gsz;
  nb = r / gsz;
}

template <typename T, int BN, int STAGES>
__global__ void __launch_bounds__(384, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
               const GemmKParams p) {
  constexpr int BM = 128, BK = 64;
  constexpr uint32_t A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN <= 32 ? 32 : 2 * BN <= 64 ? 64 : 2 * BN <= 128 ? 128 : 2 * BN <= 256 ? 256 : 512;
  static_assert(2 * BN <= 512, "two accumulator buffers must fit the 512 TMEM columns");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // array + offset keeps the shared address space (STS / LDS, not generic ST / LD)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  uint8_t* epi_smem = smem + STAGES * STAGE_BYTES + 256;   // 4 x EPI_WARP_BYTES staging for the epilogue warps

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  auto stamp = [&](int slot) {
    if (p.dbg && blockIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.dbg[slot] = t;
    }
  };
  if (threadIdx.x == 0) stamp(0);
  pdl_trigger();
  const int m_blocks = (p.M + BM - 1) / BM;
  const int n_blocks = (p.N + BN - 1) / BN;
  const int k_blocks = (p.K + BK - 1) / BK;
  const int num_tiles = m_blocks * n_blocks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      // folded RMSNorm: the epilogue warps read every A stage too, so a stage is free after the MMA commit AND their 8 arrivals
      mbar_init(&empty_bar[i], p.ssq_inline ? 1 + EPI_WARPS : 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) stamp(1);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      // Weight tiles of the first pipeline fill do not depend on the previous kernel: request them before the
      // programmatic-dependency wait so that the DRAM latency overlaps the predecessor's tail.
      int early = 0;
      if (p.w_constant && static_cast<int>(blockIdx.x) < num_tiles) {
        int mb, nb;
        tile_coords(blockIdx.x, m_blocks, n_blocks, p.group_m, mb, nb);
        early = k_blocks < STAGES ? k_blocks : STAGES;
        for (int kb = 0; kb < early; ++kb) {
          uint8_t* sa = smem + kb * STAGE_BYTES;
          mbar_expect_tx(&full_bar[kb], STAGE_BYTES);
          tma_load_2d(sa + A_BYTES, &tma_b, &full_bar[kb], kb * BK, nb * BN);
        }
      }
      pdl_wait();
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int mb, nb;
        tile_coords(tile, m_blocks, n_blocks, p.group_m, mb, nb);
        for (int kb = 0; kb < k_blocks; ++kb) {
          uint8_t* sa = smem + s * STAGE_BYTES;
          uint8_t* sbp = sa + A_BYTES;
          if (tile == static_cast<int>(blockIdx.x) && kb < early) {
            tma_load_2d(sa, &tma_a, &full_bar[s], kb * BK + nb * p.group_k, mb * BM);   // B already in flight
          } else {
            mbar_wait(&empty_bar[s], ph ^ 1);
            mbar_expect_tx(&full_bar[s], STAGE_BYTES);
            tma_load_2d(sa, &tma_a, &full_bar[s], kb * BK + nb * p.group_k, mb * BM);
            tma_load_2d(sbp, &tma_b, &full_bar[s], kb * BK, nb * BN);
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (one thread)
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(TypeInfo<T>::umma_fmt, BM, BN);
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (tile == static_cast<int>(blockIdx.x) && kb < 38) stamp(2 + kb);
          const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
          const uint64_t da = umma_desc_k128(sa);
          const uint64_t db = umma_desc_k128(sa + A_BYTES);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // +32 bytes (= 2 x 16B units) per UMMA_K step inside the 128B swizzle atom
            umma_f16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit(&tfull_bar[as]);
        as ^= 1;
        if (as == 0) aph ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue warps
    pdl_wait();
    const int q = warp & 3;             // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;   // two warps share a quarter and alternate column groups
    const int epi_tid = threadIdx.x - 128;
    uint8_t* stage = epi_smem + (warp - 4) * EPI_STAGE_BYTES;
    float* sbias = reinterpret_cast<float*>(epi_smem + EPI_WARPS * EPI_STAGE_BYTES);
    float* srs = sbias + BN;                              // 128 per-row scales of the current tile (folded RMSNorm)
    int as = 0;
    uint32_t aph = 0;
    int es = 0;                                           // pipeline stage / phase as seen by the sum-of-squares pass
    uint32_t eph = 0;
    const bool vec_ok = (p.ldc % 8 == 0) && (!p.residual || p.ldr % 8 == 0);
    const bool v2 = epilogue_v2_ok(p);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      int mb, nb;
      tile_coords(tile, m_blocks, n_blocks, p.group_m, mb, nb);
      if (v2) {
        asm volatile("bar.sync 1, 256;" ::: "memory");   // all epilogue warps are done with the previous tile's bias
        epilogue_stage_bias<BN>(p, sbias, epi_tid, nb * BN);
        if (p.rowscale && epi_tid < BM) srs[epi_tid] = mb * BM + epi_tid < p.M ? __ldg(p.rowscale + mb * BM + epi_tid) : 0.f;
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      if (p.ssq_inline) {
        // sum of squares of the tile's 128 A rows, taken from the pipeline stages while the MMA warp consumes them
        float acc = 0.f;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[es], eph);
          acc = ssq_stage<T>(smem + es * STAGE_BYTES, epi_tid, acc);
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty_bar[es]);
          if (++es == STAGES) { es = 0; eph ^= 1; }
        }
        const float tot = acc + __shfl_xor_sync(0xffffffffu, acc, 1);
        if ((epi_tid & 1) == 0) srs[epi_tid >> 1] = rsqrtf(tot * p.ssq_inv_k + p.ssq_eps);
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after();
      if (warp == 4 && lane == 0 && tile == static_cast<int>(blockIdx.x)) stamp(40);
      const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
      if (v2) {
        const int row0 = mb * BM + q * 32;
        const float rs = (p.ssq_inline || p.rowscale) ? srs[q * 32 + lane] : 1.0f;
        if (!p.am_val || p.store_c)
          epilogue_tile_v2<T, BN>(tacc, p, stage, sbias, lane, half,
                                  [&](int r) { return row0 + r < p.M ? row0 + r : -1; }, nb * BN, rs);
        if (p.am_val)
          epilogue_tile_argmax<T, BN>(tacc, p, epi_smem, sbias, lane, half, q,
                                      row0 + lane < p.M ? row0 + lane : -1, nb * BN, nb, rs);
      } else if (half == 0) {
        const int row = mb * BM + q * 32 + lane;
        const bool row_ok = row < p.M;
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t v[32];
          __syncwarp();  // tcgen05.ld is .sync.aligned: reconverge lanes that skipped the previous chunk
          tmem_ld_32x32(tacc + c * 32, v);
          tmem_ld_wait();
          const int col0 = nb * BN + c * 32;
          if (col0 >= p.N) continue;
          epilogue_chunk<T>(v, p, row, row_ok, col0, vec_ok);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      if (warp == 4 && lane == 0 && tile == static_cast<int>(blockIdx.x)) stamp(41);
      as ^= 1;
      if (as == 0) aph ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
  if (threadIdx.x == 0) stamp(42);
}

// ----------------------------------------------------------------------------------- host side
static thread_local char g_err[512] = {0};
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* last_error() { return g_err; }

static std::atomic<long long> g_launches{0};
long long launch_count() { return g_launches.load(); }
bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SB_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
bool splitk_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SB_SPLITK"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
void count_launches(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int launch_ok() {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("kernel launch failed: %s", cudaGetErrorString(e));
    return -2;
  }
  return 0;
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// cuTensorMapEncodeTiled costs 1-2 us of host time per operand; engines issue the same few hundred (pointer, shape, box)
// combinations every forward / step, so encoded maps are memoised (key = every argument of the encode call).
static CUresult encode_tiled_cached(CUtensorMap* map, CUtensorMapDataType dt, int rank, const void* base, const cuuint64_t* dims,
                                    const cuuint64_t* strides, const cuuint32_t* box, const cuuint32_t* estr,
                                    CUtensorMapSwizzle swz) {
  struct Key { uint64_t v[18]; };
  Key k{};
  k.v[0] = reinterpret_cast<uint64_t>(base);
  k.v[1] = (static_cast<uint64_t>(dt) << 40) | (static_cast<uint64_t>(rank) << 32) | static_cast<uint64_t>(swz);
  for (int i = 0; i < rank; ++i) { k.v[2 + i] = dims[i]; k.v[10 + i] = (static_cast<uint64_t>(box[i]) << 32) | estr[i]; }
  for (int i = 0; i + 1 < rank; ++i) k.v[6 + i] = strides[i];
  const std::string key(reinterpret_cast<const char*>(&k), sizeof(k));
  static std::mutex mu;
  static std::unordered_map<std::string, CUtensorMap> cache;
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *map = it->second; return CUDA_SUCCESS; }
  }
  CUresult r = get_encode_fn()(map, dt, rank, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) {
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > 16384) cache.clear();
    cache.emplace(key, *map);
  }
  return r;
}

// 2-D K-major operand map: global [rows, K] with row stride ld (elements); box = 64 x box_rows; 128B swizzle.
int make_tma_2d(CUtensorMap* map, int dtype, const void* base, int rows, int K, int ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return -1;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (static_cast<size_t>(ld) * 2) % 16 != 0) {
    set_error("TMA operand must be 16B aligned with a 16B-multiple row pitch (ptr=%p ld=%d)", base, ld);
    return -2;
  }
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled_cached(map, dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base,
                                   dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: %d (rows=%d K=%d ld=%d box_rows=%d)", (int)r, rows, K, ld, box_rows);
    return -3;
  }
  return 0;
}

int make_tma_2d_sw(CUtensorMap* map, int dtype, const void* base, int rows, int K, int ld, int box_k, int box_rows,
                   int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return -1; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (static_cast<size_t>(ld) * 2) % 16 != 0) {
    set_error("TMA operand must be 16B aligned with a 16B-multiple row pitch (ptr=%p ld=%d)", base, ld);
    return -2;
  }
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_k), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled_cached(map, dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base,
                                   dims, strides, box, estr,
                                   swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                                        : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE));
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(2d) failed: %d", (int)r); return -3; }
  return 0;
}

// NHWC activation map for the implicit-GEMM convolution: dims {C, W, H, N}; box {box_c, box_w, box_h, 1} OUTPUT
// pixels, traversed with `stride` in W and H (boxDim = pixels * stride, elementStrides = stride).
int make_tma_nhwc(CUtensorMap* map, int dtype, const void* base, int N, int H, int W, int C, int box_c, int box_w,
                  int box_h, int stride, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)"); return -1; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (static_cast<size_t>(C) * 2) % 16 != 0) {
    set_error("NHWC TMA operand must be 16B aligned with C %% 8 == 0 (ptr=%p C=%d)", base, C);
    return -2;
  }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)(box_w * stride), (cuuint32_t)(box_h * stride), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = encode_tiled_cached(map, dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base,
                                   dims, strides, box, estr,
                                   swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                                        : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE));
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(nhwc) failed: %d (N=%d H=%d W=%d C=%d box=%d,%d,%d stride=%d)", (int)r, N, H, W, C,
              box_c, box_w, box_h, stride);
    return -3;
  }
  return 0;
}

template <typename T, int BN, int STAGES>
static int launch_cfg(const GemmArgs& a, cudaStream_t stream) {
  constexpr uint32_t STAGE_BYTES = 128 * 64 * 2 + BN * 64 * 2;
  constexpr size_t SMEM = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + epi_smem_bytes<BN>();
  static bool attr_set = false;
  auto kern = gemm_tn_kernel<T, BN, STAGES>;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute(smem=%zu) failed: %s", SMEM, cudaGetErrorString(e));
      return -10;
    }
    attr_set = true;
  }
  CUtensorMap ma, mb;
  int rc = make_tma_2d(&ma, a.dtype, a.A, a.M, a.group_k ? a.a_cols : a.K, a.lda, 128);
  if (rc) return rc;
  rc = make_tma_2d(&mb, a.dtype, a.W, a.N, a.K, a.ldw, BN);  // grouped: W is [N, K] with K = padded per-group depth
  if (rc) return rc;
  GemmKParams p{};
  p.M = a.M; p.N = a.N; p.K = a.K;
  p.C = a.C; p.ldc = a.ldc;
  p.bias = a.bias;
  p.residual = a.residual; p.ldr = a.ldr;
  p.act = a.act; p.swiglu = a.swiglu; p.out_f32 = a.out_f32;
  p.group_m = 8;
  p.group_k = a.group_k;
  p.dbg = a.dbg;
  p.w_constant = a.w_constant;
  p.rowscale = a.rowscale;
  p.ssq_inline = a.ssq_inline;
  p.ssq_eps = a.ssq_eps;
  p.ssq_inv_k = 1.0f / static_cast<float>(a.ssq_k > 0 ? a.ssq_k : a.K);
  p.am_val = a.am_val; p.am_idx = a.am_idx; p.am_sum = a.am_sum; p.am_ld = a.am_ld; p.store_c = a.store_c;
  int m_blocks = (a.M + 127) / 128, n_blocks = (a.N + BN - 1) / BN;
  int tiles = m_blocks * n_blocks;
  int grid = tiles < num_sms() ? tiles : num_sms();
  if (launch_pdl(kern, dim3(grid), dim3(384), SMEM, stream, ma, mb, p) != cudaSuccess) { /* reported by launch_ok */ }
  return launch_ok();
}

template <typename T>
static int launch_typed(const GemmArgs& a, cudaStream_t stream) {
  int bn = a.force_bn;
  if (bn >= 1000) return gemm_splitk_launch(a, bn / 1000, bn % 1000, stream);   // forced split-K: 1000 * pk + BN
  if (bn == 0 && a.allow_splitk && splitk_enabled() && !a.rowscale && !a.ssq_inline && !a.am_val) {
    int sbn = 0;
    const int pk = splitk_plan(a, &sbn);
    if (pk >= 2) return gemm_splitk_launch(a, pk, sbn, stream);
  }
  if (bn == 0) {
    // Big problems: 128x256 tiles (highest flop per byte of smem fill).  Otherwise the main loop is bound by DRAM latency x
    // bytes in flight per SM, so prefer a single wave of many small tiles: cost = waves * bytes per k-block, with a penalty
    // when fewer than ~60 % of the SMs would be streaming the weight matrix.
    const int sms = num_sms();
    const int m_blocks = (a.M + 127) / 128;
    if (a.N <= 128 && m_blocks >= sms) {
      // narrow outputs over many rows (1x1 "project" convs): the launch streams A; a tile wider than N only adds zero-filled W
      // loads and MMA / epilogue work (profiles/r01c_det_launch_summary.md: N = 64 ran on 256-wide tiles at 43 % of HBM peak)
      bn = a.N <= 32 ? 32 : a.N <= 64 ? 64 : a.N <= 96 ? 96 : 128;
    } else if (m_blocks * ((a.N + 255) / 256) >= (sms * 3) / 4) {
      bn = 256;
    } else {
      const int cands[5] = {256, 128, 96, 64, 32};
      double best = 1e30;
      for (int i = 0; i < 5; ++i) {
        const int c = cands[i];
        if (a.swiglu && (c % 32)) continue;
        const int tiles = m_blocks * ((a.N + c - 1) / c);
        const int waves = (tiles + sms - 1) / sms;
        double cost = static_cast<double>(waves) * (128 + c);
        const double occ = 0.6 * sms / tiles;
        if (occ > 1.0) cost *= occ;
        if (cost < best) { best = cost; bn = c; }
      }
    }
  }
  if (a.am_val && a.force_bn == 0) bn = gemm_argmax_tile(a.M, a.N);   // the caller sized its partial buffers with this
  if (a.group_k) bn = a.group_n;  // one n-block per channel group
  switch (bn) {
    case 256: return launch_cfg<T, 256, 4>(a, stream);
    case 128: return launch_cfg<T, 128, 6>(a, stream);
    case 96: return launch_cfg<T, 96, 6>(a, stream);
    case 64: return launch_cfg<T, 64, 8>(a, stream);
    case 32: return launch_cfg<T, 32, 8>(a, stream);
    default: set_error("unsupported BN %d", bn); return -12;
  }
}

int gemm_argmax_tile(int M, int N) {
  (void)M;
  return N >= 4096 ? 256 : (N >= 1024 ? 128 : 64);
}

int gemm_launch(const GemmArgs& a, cudaStream_t stream) {
  if (a.M <= 0 || a.N <= 0 || a.K <= 0) return 0;
  if (a.rowscale || a.ssq_inline || a.am_val) {
    // these ride on the staged 16-bit epilogue only (and on the plain kernel: split-K would change who owns a row's columns)
    const bool v2 = !a.out_f32 && a.ldc % 8 == 0 && (!a.residual || a.ldr % 8 == 0) &&
                    (a.swiglu ? ((a.act == ACT_SILU || a.act == ACT_GELU_TANH) && a.N % 16 == 0) : a.N % 8 == 0);
    if (!v2 || a.group_k || a.force_bn >= 1000) {
      set_error("gemm: rowscale / ssq_inline / argmax epilogues need the 16-bit staged epilogue (N %% 8 == 0, 16-byte pitches), "
                "no grouped or split-K mode");
      return -15;
    }
    if (a.rowscale && a.ssq_inline) { set_error("gemm: rowscale and ssq_inline are exclusive"); return -15; }
    if (a.am_val && (!a.am_idx || !a.am_sum || a.am_ld <= 0)) { set_error("gemm: incomplete argmax partial buffers"); return -15; }
  }
  if (a.swiglu && (a.N % 2 != 0)) {
    set_error("swiglu epilogue needs an even N");
    return -13;
  }
  if (a.dtype != DT_BF16 && a.dtype != DT_F16) { set_error("unsupported dtype %d", a.dtype); return -14; }
  if (gemm_skinny_ok(a)) return gemm_skinny_launch(a, stream);
  if (a.dtype == DT_BF16) return launch_typed<__nv_bfloat16>(a, stream);
  return launch_typed<__half>(a, stream);
}

}  // namespace sb
