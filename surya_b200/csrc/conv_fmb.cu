// surya_b200 — FusedMBConv in one kernel: 3x3 conv (expand, + folded BN, Hardswish) -> 1x1 project (+ folded BN, + identity
// shortcut), the expanded tensor never leaves the SM.
//
// Stands in for FusedMBConv.forward (surya/detection/model/encoderdecoder.py:228-270) of the EfficientViT stages 0 and 1 and
// replaces the op pair conv_igemm -> gemm of det_engine.cu.  At BASELINE config 3 the four blocks write and re-read
// 2.1 + 1.0 + 1.0 + 0.5 GB of expanded activations per 32-page forward (profiles/r02_det_launch_summary.md).
//
// Back-to-back GEMM per 128-pixel tile (8 rows x 16 px):
//   for each chunk j of 128 mid channels:
//     GEMM1  acc1[j & 1] (TMEM, 128 cols) = sum over 9 taps x Cin/BKC channel chunks of  A1 (tap box, TMA)  x  W1[j] (TMA)
//     epi1   8 warps: acc1 + shift -> round -> Hardswish -> round -> 128B-swizzled A2 tile in shared memory (2 k-blocks of 64)
//     GEMM2  acc2 (TMEM, Cout cols) += A2 x W2[:, chunk j] (TMA)          [issued after GEMM1(j+1): epi1(j) hides under it]
//   epi2     4 warps: acc2 + shift (+ block input) -> round -> NHWC store
// Rounding points are those of the two separate kernels (expand output in T after the shift, after Hardswish; project output
// in T after the shift, after the residual add); the fp32 sum over the mid channels runs in the same k order as gemm_tn_kernel.
#include "gemm.cuh"
#include "gemm_epilogue.cuh"
#include "ops.cuh"
#include "sb_ptx.cuh"

#include <cstdlib>

namespace sb {

int make_tma_2d(CUtensorMap* map, int dtype, const void* base, int rows, int K, int ld, int box_rows);
int make_tma_2d_sw(CUtensorMap* map, int dtype, const void* base, int rows, int K, int ld, int box_k, int box_rows,
                   int swizzle_bytes);
int make_tma_nhwc(CUtensorMap* map, int dtype, const void* base, int N, int H, int W, int C, int box_c, int box_w,
                  int box_h, int stride, int swizzle_bytes);

struct FmbParams {
  int n_img, H, W, Ho, Wo, Cin, Cmid, Cout, stride;
  int tiles_x, tiles_y;
  const float* bias1;     // [Cmid]
  const float* bias2;     // [Cout]
  const void* residual;   // NHWC [n_img, Ho, Wo, Cout] or null
  void* out;              // NHWC [n_img, Ho, Wo, Cout]
};

template <typename T, int COUT, int STAGES, int NW2>
__global__ void __launch_bounds__(512, 1)
fmb_fused_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w1,
                 const __grid_constant__ CUtensorMap tma_w2, const FmbParams fp) {
  constexpr int BM = 128, TW = 16, TH = 8, CH = 128;                 // mid-channel chunk
  constexpr int BKC = 64;                                            // input channels per GEMM1 k-block
  constexpr uint32_t A1_BYTES = BM * BKC * 2;
  constexpr uint32_t W1_BYTES = CH * BKC * 2;
  constexpr uint32_t S1_BYTES = A1_BYTES + W1_BYTES;
  constexpr uint32_t A2_KB_BYTES = BM * 64 * 2;                      // one 64-channel k-block of the A2 tile (16 KB)
  constexpr uint32_t A2_BYTES = 2 * A2_KB_BYTES;                     // 128 mid channels
  constexpr uint32_t W2_KB_BYTES = COUT * 64 * 2, W2_BYTES = 2 * W2_KB_BYTES;
  constexpr uint32_t TMEM_COLS = 512;                                // acc1: 2 x 128, acc2: COUT at column 256

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // array + offset keeps the shared address space (STS / LDS, not generic ST / LD)
  uint8_t* s_1 = smem;
  uint8_t* s_a2 = s_1 + STAGES * S1_BYTES;
  uint8_t* s_w2 = s_a2 + 2 * A2_BYTES;
  float* s_b1 = reinterpret_cast<float*>(s_w2 + NW2 * W2_BYTES);
  float* s_b2 = s_b1 + fp.Cmid;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_b2 + COUT);
  uint64_t* s1_full = bars;
  uint64_t* s1_empty = s1_full + STAGES;
  uint64_t* t1_full = s1_empty + STAGES;
  uint64_t* t1_empty = t1_full + 2;
  uint64_t* a2_full = t1_empty + 2;
  uint64_t* a2_empty = a2_full + 2;
  uint64_t* w2_full = a2_empty + 2;
  uint64_t* w2_empty = w2_full + NW2;
  uint64_t* t2_full = w2_empty + NW2;
  uint64_t* t2_empty = t2_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t2_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_img = fp.tiles_x * fp.tiles_y;
  const int num_tiles = fp.n_img * tiles_per_img;
  const int nch = fp.Cmid / CH;
  const int cpb = fp.Cin / BKC;                                      // channel chunks per tap
  const int kb1 = 9 * cpb;                                           // GEMM1 k-blocks per mid chunk

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tma_a); tma_prefetch_desc(&tma_w1); tma_prefetch_desc(&tma_w2); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&s1_full[i], 1); mbar_init(&s1_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&t1_full[i], 1); mbar_init(&t1_empty[i], 8);
      mbar_init(&a2_full[i], 8); mbar_init(&a2_empty[i], 1);
    }
    for (int i = 0; i < NW2; ++i) { mbar_init(&w2_full[i], 1); mbar_init(&w2_empty[i], 1); }
    mbar_init(t2_full, 1); mbar_init(t2_empty, 4);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < fp.Cmid; i += blockDim.x) s_b1[i] = fp.bias1 ? fp.bias1[i] : 0.f;
  for (int i = threadIdx.x; i < COUT; i += blockDim.x) s_b2[i] = fp.bias2 ? fp.bias2[i] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto coords = [&](int tile, int& img, int& oy0, int& ox0) {
    img = tile / tiles_per_img;
    const int t = tile - img * tiles_per_img;
    oy0 = (t / fp.tiles_x) * TH;
    ox0 = (t % fp.tiles_x) * TW;
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0; uint32_t ph = 0; int wb = 0; uint32_t wph = 0;
      auto load_w2 = [&](int j) {
        mbar_wait(&w2_empty[wb], wph ^ 1);
        mbar_expect_tx(&w2_full[wb], W2_BYTES);
        tma_load_2d(s_w2 + wb * W2_BYTES, &tma_w2, &w2_full[wb], j * CH, 0);
        tma_load_2d(s_w2 + wb * W2_BYTES + W2_KB_BYTES, &tma_w2, &w2_full[wb], j * CH + 64, 0);
        if (++wb == NW2) { wb = 0; wph ^= 1; }
      };
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int img, oy0, ox0;
        coords(tile, img, oy0, ox0);
        const int x0 = ox0 * fp.stride - 1, y0 = oy0 * fp.stride - 1;
        for (int j = 0; j < nch; ++j) {
          int kcol = 0;
          for (int r = 0; r < 3; ++r)
            for (int sx = 0; sx < 3; ++sx)
              for (int cc = 0; cc < cpb; ++cc, kcol += BKC) {
                mbar_wait(&s1_empty[s], ph ^ 1);
                uint8_t* sa = s_1 + s * S1_BYTES;
                mbar_expect_tx(&s1_full[s], S1_BYTES);
                tma_load_4d(sa, &tma_a, &s1_full[s], cc * BKC, x0 + sx, y0 + r, img);
                tma_load_2d(sa + A1_BYTES, &tma_w1, &s1_full[s], kcol, j * CH);
                if (++s == STAGES) { s = 0; ph ^= 1; }
              }
          if (j >= 1) load_w2(j - 1);
        }
        load_w2(nch - 1);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc1 = umma_idesc_f16(TypeInfo<T>::umma_fmt, BM, CH);
      constexpr uint32_t idesc2 = umma_idesc_f16(TypeInfo<T>::umma_fmt, BM, COUT);
      int s = 0; uint32_t ph = 0; int wb = 0; uint32_t wph = 0;
      uint32_t t1ph[2] = {0, 0}, a2ph[2] = {0, 0}, t2ph = 0;
      auto gemm2 = [&](int j) {
        const int b = j & 1;
        mbar_wait(&a2_full[b], a2ph[b]);
        a2ph[b] ^= 1;
        mbar_wait(&w2_full[wb], wph);
        if (j == 0) { mbar_wait(t2_empty, t2ph ^ 1); }
        tc_fence_after();
        const uint32_t d2 = tmem_base + 256;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const uint64_t da = umma_desc_k128(smem_u32(s_a2 + b * A2_BYTES + kk * A2_KB_BYTES));
          const uint64_t db = umma_desc_k128(smem_u32(s_w2 + wb * W2_BYTES + kk * W2_KB_BYTES));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(d2, da + 2 * k, db + 2 * k, idesc2, (j | kk | k) != 0 ? 1u : 0u);
        }
        umma_commit(&a2_empty[b]);
        umma_commit(&w2_empty[wb]);
        if (++wb == NW2) { wb = 0; wph ^= 1; }
      };
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int j = 0; j < nch; ++j) {
          const int b = j & 1;
          mbar_wait(&t1_empty[b], t1ph[b] ^ 1);
          t1ph[b] ^= 1;
          tc_fence_after();
          const uint32_t d1 = tmem_base + b * CH;
          for (int kb = 0; kb < kb1; ++kb) {
            mbar_wait(&s1_full[s], ph);
            tc_fence_after();
            const uint32_t sa = smem_u32(s_1 + s * S1_BYTES);
            const uint64_t da = umma_desc_k128(sa);
            const uint64_t db = umma_desc_k128(sa + A1_BYTES);
#pragma unroll
            for (int k = 0; k < BKC / 16; ++k) umma_f16(d1, da + 2 * k, db + 2 * k, idesc1, (kb | k) != 0 ? 1u : 0u);
            umma_commit(&s1_empty[s]);
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
          umma_commit(&t1_full[b]);
          if (j >= 1) gemm2(j - 1);
        }
        gemm2(nch - 1);
        umma_commit(t2_full);
        t2ph ^= 1;
      }
    }
  } else if (warp >= 12) {
    // ------------------------------------------------------------------ epilogue 2: project output
    const int q = warp & 3;
    const int row = q * 32 + lane;
    uint32_t t2ph = 0;
    T* out = reinterpret_cast<T*>(fp.out);
    const T* res = reinterpret_cast<const T*>(fp.residual);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      int img, oy0, ox0;
      coords(tile, img, oy0, ox0);
      const int oy = oy0 + (row >> 4), ox = ox0 + (row & 15);
      const bool ok = oy < fp.Ho && ox < fp.Wo;
      const size_t pix = (static_cast<size_t>(img) * fp.Ho + (ok ? oy : 0)) * fp.Wo + (ok ? ox : 0);
      mbar_wait(t2_full, t2ph);
      t2ph ^= 1;
      tc_fence_after();
      const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + 256;
#pragma unroll 1
      for (int g = 0; g < COUT / 32; ++g) {
        uint32_t v[32];
        tmem_ld_32x32(tacc + g * 32, v);
        tmem_ld_wait();
        uint32_t o[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2)
          o[j >> 1] = Pk<T>::pack(__uint_as_float(v[j]) + s_b2[g * 32 + j], __uint_as_float(v[j + 1]) + s_b2[g * 32 + j + 1]);
        if (res && ok) {
          const uint4* rp = reinterpret_cast<const uint4*>(res + pix * COUT + g * 32);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint4 r4 = __ldg(rp + c);
            const uint32_t rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t t = o[c * 4 + k];
              o[c * 4 + k] = Pk<T>::pack(Pk<T>::lo(t) + Pk<T>::lo(rr[k]), Pk<T>::hi(t) + Pk<T>::hi(rr[k]));
            }
          }
        }
        if (ok) {
          uint4* op = reinterpret_cast<uint4*>(out + pix * COUT + g * 32);
#pragma unroll
          for (int c = 0; c < 4; ++c) op[c] = make_uint4(o[c * 4], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t2_empty);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue 1: expanded chunk -> A2 tile in shared memory
    const int q = warp & 3, hh = (warp - 4) >> 2;          // lane quarter; 64-channel k-block of the chunk
    const int row = q * 32 + lane;
    uint32_t t1ph[2] = {0, 0}, a2ph[2] = {0, 0};
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int j = 0; j < nch; ++j) {
        const int b = j & 1;
        mbar_wait(&t1_full[b], t1ph[b]);
        t1ph[b] ^= 1;
        tc_fence_after();
        mbar_wait(&a2_empty[b], a2ph[b] ^ 1);              // GEMM2 of two chunks ago has read this A2 buffer
        a2ph[b] ^= 1;
        const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + b * CH + hh * 64;
        uint8_t* dst = s_a2 + b * A2_BYTES + hh * A2_KB_BYTES + row * 128;
        const float* bs = s_b1 + j * CH + hh * 64;
#pragma unroll 1
        for (int g = 0; g < 2; ++g) {
          uint32_t v[32];
          tmem_ld_32x32(tacc + g * 32, v);
          tmem_ld_wait();
          uint32_t o[16];
#pragma unroll
          for (int jj = 0; jj < 32; jj += 2) {
            const uint32_t t = Pk<T>::pack(__uint_as_float(v[jj]) + bs[g * 32 + jj], __uint_as_float(v[jj + 1]) + bs[g * 32 + jj + 1]);
            o[jj >> 1] = Pk<T>::pack(act_ct<ACT_HARDSWISH>(Pk<T>::lo(t)), act_ct<ACT_HARDSWISH>(Pk<T>::hi(t)));
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int ch = g * 4 + c;                       // 16-byte chunk inside the 128-byte row
            *reinterpret_cast<uint4*>(dst + ((ch ^ (row & 7)) << 4)) = make_uint4(o[c * 4], o[c * 4 + 1], o[c * 4 + 2], o[c * 4 + 3]);
          }
        }
        tc_fence_before();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) { mbar_arrive(&t1_empty[b]); mbar_arrive(&a2_full[b]); }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

bool fmb_fused_ok(int Cin, int Cmid, int Cout, int ksize, int stride, int pad, int act1, int act2) {
  static int en = -1;
  if (en < 0) { const char* e = getenv("SB_FMB_FUSED"); en = e ? (e[0] - '0') : 1; }
  if (!en) return false;
  if (ksize != 3 || pad != 1 || (stride != 1 && stride != 2) || act1 != ACT_HARDSWISH || act2 != ACT_NONE) return false;
  // Cin = 32 (stage 0, block 0) stays on the two separate kernels: fused, it measured slower (1.38 vs 1.33 ms at B = 32)
  if (Cin != 64 && Cin != 128) return false;
  if (Cmid % 128 || Cmid < 128 || Cmid > 1024) return false;
  return Cout == 64 || Cout == 128;
}

template <typename T, int COUT, int STAGES, int NW2>
static int launch_fmb(int dtype, const void* in, const void* w1, const void* w2, const FmbParams& fp, cudaStream_t st) {
  constexpr int BKC = 64;
  constexpr size_t S1 = static_cast<size_t>(128 * BKC * 2) * 2;
  const size_t SMEM = STAGES * S1 + 2 * 32768 + NW2 * (COUT * 256) + (fp.Cmid + COUT) * 4 + 512 + 1024;
  auto kern = fmb_fused_kernel<T, COUT, STAGES, NW2>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM) != cudaSuccess) {
    cudaGetLastError();
    set_error("fmb_fused: cudaFuncSetAttribute(smem=%zu) failed", SMEM);
    return -10;
  }
  CUtensorMap ma, m1, m2;
  int rc = make_tma_nhwc(&ma, dtype, in, fp.n_img, fp.H, fp.W, fp.Cin, BKC, 16, 8, fp.stride, BKC * 2);
  if (rc) return rc;
  rc = make_tma_2d_sw(&m1, dtype, w1, fp.Cmid, 9 * fp.Cin, 9 * fp.Cin, BKC, 128, BKC * 2);
  if (rc) return rc;
  rc = make_tma_2d(&m2, dtype, w2, COUT, fp.Cmid, fp.Cmid, COUT);
  if (rc) return rc;
  const int tiles = fp.n_img * fp.tiles_x * fp.tiles_y;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, 512, SMEM, st>>>(ma, m1, m2, fp);
  return launch_ok();
}

// in NHWC [n_img, H, W, Cin]; w1 T [Cmid][9*Cin] (tap-major, BN folded), bias1 fp32 [Cmid]; w2 T [Cout][Cmid], bias2 fp32 [Cout];
// residual NHWC [n_img, Ho, Wo, Cout] or null; out NHWC [n_img, Ho, Wo, Cout].
int fmb_fused(int dtype, const void* in, const void* w1, const float* bias1, const void* w2, const float* bias2,
              const void* residual, void* out, int n_img, int H, int W, int Cin, int Cmid, int Cout, int stride, cudaStream_t st) {
  if (n_img <= 0) return 0;
  if (!fmb_fused_ok(Cin, Cmid, Cout, 3, stride, 1, ACT_HARDSWISH, ACT_NONE)) { set_error("fmb_fused: unsupported shape"); return -1; }
  FmbParams fp{};
  fp.n_img = n_img; fp.H = H; fp.W = W; fp.Ho = (H + 2 - 3) / stride + 1; fp.Wo = (W + 2 - 3) / stride + 1;
  fp.Cin = Cin; fp.Cmid = Cmid; fp.Cout = Cout; fp.stride = stride;
  fp.tiles_x = (fp.Wo + 15) / 16; fp.tiles_y = (fp.Ho + 7) / 8;
  fp.bias1 = bias1; fp.bias2 = bias2; fp.residual = residual; fp.out = out;
#define FMB(T_) \
  do { \
    if (Cout == 64) return launch_fmb<T_, 64, 3, 2>(dtype, in, w1, w2, fp, st); \
    return launch_fmb<T_, 128, 3, 1>(dtype, in, w1, w2, fp, st); \
  } while (0)
  if (dtype == DT_BF16) FMB(__nv_bfloat16); else FMB(__half);
#undef FMB
}

}  // namespace sb
