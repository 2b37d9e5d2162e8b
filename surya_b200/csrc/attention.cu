// surya_b200 — attention kernels.
//
//  attn_varlen  : block-diagonal (per-sequence) flash attention over packed tokens, optional causal mask and GQA.
//                 Replaces flash_attn_varlen_func / SDPA in the recognition vision tower
//                 (surya/common/surya/encoder/__init__.py:136-178, 202-263, 266-411) and in decoder prefill
//                 (surya/common/surya/decoder/__init__.py:101-128, flash_attn_utils.py:106-154).
//                 Tensor-core path: mma.sync m16n8k16 (fp32 accumulate), online softmax in fp32 registers,
//                 P rounded to the storage type before the PV product (flash-attention semantics).
//                 Attention is < 1 % of the recognition FLOPs (SURVEY.md §8a a10), the tcgen05 budget goes to the GEMMs.
//  decode_attn  : q_len = 1 attention over the slot KV cache fused with RoPE(q,k) and the in-place cache append
//                 (decoder/__init__.py:161-238 with DynamicCache.update -> no torch.cat, SURVEY.md §2.2 K10/K20).
//                 HBM-bound: streams K and V once, CUDA-core FMA.
#include "ops.cuh"
#include "sb_ptx.cuh"

namespace sb {

template <typename T> struct Mma;
template <> struct Mma<__nv_bfloat16> {
  static __device__ __forceinline__ void run(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  static __device__ __forceinline__ uint32_t pack(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
};
template <> struct Mma<__half> {
  static __device__ __forceinline__ void run(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  static __device__ __forceinline__ uint32_t pack(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
};

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t smem_addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_addr));
}

struct AttnKParams {
  const void* q; int ldq;
  const void* k; int ldk;
  const void* v; int ldv;
  void* out; int ldo;
  const int* seq_start;
  const int* seq_len;
  int q_tiles;      // q tiles per sequence (ceil(max_len / 64))
  int n_heads, group;  // group = n_heads / n_kv_heads
  int causal;
  float scale_log2;  // scale * log2(e)
};

template <typename T, int HD>
__global__ void __launch_bounds__(128) attn_varlen_kernel(const AttnKParams p) {
  constexpr int BQ = 64, BKV = 64, LDS = HD + 8, KS = HD / 16, DN = HD / 8;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  T* sQ = reinterpret_cast<T*>(smem_attn);
  T* sK = sQ + BQ * LDS;
  T* sV = sK + BKV * LDS;

  const int seq = blockIdx.x / p.q_tiles;
  const int qt = blockIdx.x % p.q_tiles;
  const int h = blockIdx.y;
  const int kvh = h / p.group;
  const int len = p.seq_len[seq];
  const int q0 = qt * BQ;
  if (q0 >= len) return;
  const int start = p.seq_start[seq];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;

  const T* qbase = reinterpret_cast<const T*>(p.q) + static_cast<size_t>(h) * HD;
  const T* kbase = reinterpret_cast<const T*>(p.k) + static_cast<size_t>(kvh) * HD;
  const T* vbase = reinterpret_cast<const T*>(p.v) + static_cast<size_t>(kvh) * HD;

  constexpr int VPR = HD / 8;  // uint4 per row
  // ---- load Q tile
  for (int i = tid; i < BQ * VPR; i += 128) {
    int r = i / VPR, c = i % VPR;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (q0 + r < len) val = *reinterpret_cast<const uint4*>(qbase + static_cast<size_t>(start + q0 + r) * p.ldq + c * 8);
    *reinterpret_cast<uint4*>(sQ + r * LDS + c * 8) = val;
  }
  __syncthreads();

  const int rbase = warp * 16;
  uint32_t aQ[KS][4];
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
    aQ[ks][0] = *reinterpret_cast<const uint32_t*>(sQ + (rbase + g) * LDS + ks * 16 + 2 * t);
    aQ[ks][1] = *reinterpret_cast<const uint32_t*>(sQ + (rbase + g + 8) * LDS + ks * 16 + 2 * t);
    aQ[ks][2] = *reinterpret_cast<const uint32_t*>(sQ + (rbase + g) * LDS + ks * 16 + 8 + 2 * t);
    aQ[ks][3] = *reinterpret_cast<const uint32_t*>(sQ + (rbase + g + 8) * LDS + ks * 16 + 8 + 2 * t);
  }

  float O[DN][4];
#pragma unroll
  for (int i = 0; i < DN; ++i) { O[i][0] = O[i][1] = O[i][2] = O[i][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

  const int kv_end = p.causal ? min(len, q0 + BQ) : len;
  const int n_kt = (kv_end + BKV - 1) / BKV;
  for (int kt = 0; kt < n_kt; ++kt) {
    const int k0 = kt * BKV;
    __syncthreads();  // previous tile fully consumed
    for (int i = tid; i < BKV * VPR; i += 128) {
      int r = i / VPR, c = i % VPR;
      uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
      if (k0 + r < len) {
        size_t tok = static_cast<size_t>(start + k0 + r);
        kv = *reinterpret_cast<const uint4*>(kbase + tok * p.ldk + c * 8);
        vv = *reinterpret_cast<const uint4*>(vbase + tok * p.ldv + c * 8);
      }
      *reinterpret_cast<uint4*>(sK + r * LDS + c * 8) = kv;
      *reinterpret_cast<uint4*>(sV + r * LDS + c * 8) = vv;
    }
    __syncthreads();

    float S[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      S[nt][0] = S[nt][1] = S[nt][2] = S[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t b0 = *reinterpret_cast<const uint32_t*>(sK + (nt * 8 + g) * LDS + ks * 16 + 2 * t);
        uint32_t b1 = *reinterpret_cast<const uint32_t*>(sK + (nt * 8 + g) * LDS + ks * 16 + 8 + 2 * t);
        Mma<T>::run(S[nt], aQ[ks], b0, b1);
      }
    }
    // ---- mask, scale (log2 domain), online softmax
    const int qi0 = q0 + rbase + g, qi1 = qi0 + 8;
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        int key = k0 + nt * 8 + 2 * t + (e & 1);
        int qi = (e < 2) ? qi0 : qi1;
        bool ok = key < len && (!p.causal || key <= qi);
        float sv = ok ? S[nt][e] * p.scale_log2 : -INFINITY;
        S[nt][e] = sv;
        if (e < 2) mx0 = fmaxf(mx0, sv); else mx1 = fmaxf(mx1, sv);
      }
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
    // rows with no visible key yet keep m = -inf; guard the subtraction against inf - inf
    const float ms0 = (mn0 == -INFINITY) ? 0.f : mn0, ms1 = (mn1 == -INFINITY) ? 0.f : mn1;
    const float c0 = exp2f(m0 - ms0), c1 = exp2f(m1 - ms1);
    m0 = mn0; m1 = mn1;
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      S[nt][0] = exp2f(S[nt][0] - ms0);
      S[nt][1] = exp2f(S[nt][1] - ms0);
      S[nt][2] = exp2f(S[nt][2] - ms1);
      S[nt][3] = exp2f(S[nt][3] - ms1);
      rs0 += S[nt][0] + S[nt][1];
      rs1 += S[nt][2] + S[nt][3];
    }
    l0 = l0 * c0 + rs0;
    l1 = l1 * c1 + rs1;
#pragma unroll
    for (int dn = 0; dn < DN; ++dn) {
      O[dn][0] *= c0; O[dn][1] *= c0; O[dn][2] *= c1; O[dn][3] *= c1;
    }
    // ---- O += P V
#pragma unroll
    for (int kc = 0; kc < 4; ++kc) {
      uint32_t aP[4];
      aP[0] = Mma<T>::pack(S[2 * kc][0], S[2 * kc][1]);
      aP[1] = Mma<T>::pack(S[2 * kc][2], S[2 * kc][3]);
      aP[2] = Mma<T>::pack(S[2 * kc + 1][0], S[2 * kc + 1][1]);
      aP[3] = Mma<T>::pack(S[2 * kc + 1][2], S[2 * kc + 1][3]);
      const int mid = lane >> 3, r = lane & 7;
#pragma unroll
      for (int dn = 0; dn < DN; dn += 2) {
        uint32_t bv[4];
        const T* addr = sV + (kc * 16 + (mid & 1) * 8 + r) * LDS + (dn + (mid >> 1)) * 8;
        ldmatrix_x4_trans(bv, smem_u32(addr));
        Mma<T>::run(O[dn], aP, bv[0], bv[1]);
        Mma<T>::run(O[dn + 1], aP, bv[2], bv[3]);
      }
    }
  }
  // ---- finalize
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = l0 > 0.f ? 1.f / l0 : 0.f, i1 = l1 > 0.f ? 1.f / l1 : 0.f;
  T* obase = reinterpret_cast<T*>(p.out) + static_cast<size_t>(h) * HD;
  const int r0 = q0 + rbase + g, r1 = r0 + 8;
#pragma unroll
  for (int dn = 0; dn < DN; ++dn) {
    int col = dn * 8 + 2 * t;
    if (r0 < len)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(start + r0) * p.ldo + col) =
          Mma<T>::pack(O[dn][0] * i0, O[dn][1] * i0);
    if (r1 < len)
      *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(start + r1) * p.ldo + col) =
          Mma<T>::pack(O[dn][2] * i1, O[dn][3] * i1);
  }
}

template <typename T, int HD>
static int launch_varlen(const AttnArgs& a, cudaStream_t st) {
  constexpr size_t SMEM = 3 * 64 * (HD + 8) * sizeof(T);
  auto kern = attn_varlen_kernel<T, HD>;
  static bool attr_set = false;
  if (!attr_set) {
    if (SMEM > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    attr_set = true;
  }
  AttnKParams p;
  p.q = a.q; p.ldq = a.ldq; p.k = a.k; p.ldk = a.ldk; p.v = a.v; p.ldv = a.ldv; p.out = a.out; p.ldo = a.ldo;
  p.seq_start = a.seq_start; p.seq_len = a.seq_len;
  p.q_tiles = (a.max_len + 63) / 64;
  p.n_heads = a.n_heads; p.group = a.n_heads / a.n_kv_heads;
  p.causal = a.causal;
  p.scale_log2 = a.scale * 1.4426950408889634f;
  dim3 grid(a.n_seq * p.q_tiles, a.n_heads), block(128);
  kern<<<grid, block, SMEM, st>>>(p);
  return launch_ok();
}

template <typename T>
static int dispatch_varlen(const AttnArgs& a, cudaStream_t st) {
  switch (a.head_dim) {
    case 32: return launch_varlen<T, 32>(a, st);
    case 64: return launch_varlen<T, 64>(a, st);
    case 80: return launch_varlen<T, 80>(a, st);
    case 96: return launch_varlen<T, 96>(a, st);
    case 128: return launch_varlen<T, 128>(a, st);
    default: set_error("attn_varlen: unsupported head_dim %d (32/64/80/96/128)", a.head_dim); return -1;
  }
}

int attn_varlen(const AttnArgs& a, cudaStream_t st) {
  if (a.n_seq <= 0 || a.max_len <= 0) return 0;
  if (a.n_heads % a.n_kv_heads) { set_error("attn_varlen: n_heads must be a multiple of n_kv_heads"); return -1; }
  if (a.ldq % 8 || a.ldk % 8 || a.ldv % 8 || a.ldo % 2) { set_error("attn_varlen: pitches must be 16B multiples"); return -1; }
  return a.dtype == DT_BF16 ? dispatch_varlen<__nv_bfloat16>(a, st) : dispatch_varlen<__half>(a, st);
}

// =========================================================================================== decode attention
struct DecodeKParams {
  const void* qkv; int ld;
  void* kcache; void* vcache;
  const int* slot; const int* pos;
  const float* inv_freq;
  void* out; int ldo;
  int n_heads, n_kv_heads, s_max;
  float scale;
};

template <typename T, int HD, int G>
__global__ void __launch_bounds__(128) decode_attn_kernel(const DecodeKParams p) {
  constexpr int HALF = HD / 2, VPR = HD / 8, NKG = 128 / VPR;
  extern __shared__ __align__(16) uint8_t smem_dec[];
  T* q_t = reinterpret_cast<T*>(smem_dec);                  // [G][HD] rotated queries (in T; the first G*HD floats' worth of space)
  float* red = reinterpret_cast<float*>(smem_dec) + G * HD;  // [NKG][G][HD]
  float* sc = red + NKG * G * HD;                           // [G][s_max]
  __shared__ float s_red[4][G];
  __shared__ float s_max_g[G], s_sum_g[G];

  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x, kvh = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int slot = p.slot[b];
  const int pos = p.pos[b];
  const int n_keys = pos + 1;
  if (pos < 0 || pos >= p.s_max) {
    // the cache row is full (host-side callers reject this before launching, recognition.py / layout.py): never write past
    // the slot — emit zeros so a caller that ignored the bound sees an obviously dead row instead of corrupting a neighbour
    T* orow0 = reinterpret_cast<T*>(p.out) + static_cast<size_t>(b) * p.ldo + (blockIdx.y * G) * HD;
    for (int i = threadIdx.x; i < G * HD; i += 128) orow0[i] = from_f<T>(0.f);
    return;
  }
  const T* row = reinterpret_cast<const T*>(p.qkv) + static_cast<size_t>(b) * p.ld;
  T* kc = reinterpret_cast<T*>(p.kcache) + (static_cast<size_t>(slot) * p.n_kv_heads + kvh) * p.s_max * HD;
  T* vc = reinterpret_cast<T*>(p.vcache) + (static_cast<size_t>(slot) * p.n_kv_heads + kvh) * p.s_max * HD;

  // ---- RoPE on the G query heads and the new key; append k, v
  for (int idx = tid; idx < (G + 1) * HALF; idx += 128) {
    int hh = idx / HALF, i = idx % HALF;
    const T* src = (hh < G) ? row + (kvh * G + hh) * HD : row + (p.n_heads + kvh) * HD;
    float f = static_cast<float>(pos) * p.inv_freq[i];
    float c = rnd<T>(cosf(f)), s = rnd<T>(sinf(f));
    float x1 = to_f<T>(src[i]), x2 = to_f<T>(src[i + HALF]);
    float o1 = rnd<T>(rnd<T>(x1 * c) + rnd<T>(-x2 * s));
    float o2 = rnd<T>(rnd<T>(x2 * c) + rnd<T>(x1 * s));
    if (hh < G) {
      q_t[hh * HD + i] = from_f<T>(o1);          // exactly representable: o1 / o2 are already rounded to T
      q_t[hh * HD + i + HALF] = from_f<T>(o2);
    } else {
      kc[static_cast<size_t>(pos) * HD + i] = from_f<T>(o1);
      kc[static_cast<size_t>(pos) * HD + i + HALF] = from_f<T>(o2);
    }
  }
  {
    const T* vsrc = row + (p.n_heads + p.n_kv_heads + kvh) * HD;
    for (int i = tid; i < HD; i += 128) vc[static_cast<size_t>(pos) * HD + i] = vsrc[i];
  }
  __syncthreads();

  // ---- scores: one key per thread
  float tmax[G];
#pragma unroll
  for (int gq = 0; gq < G; ++gq) tmax[gq] = -INFINITY;
#pragma unroll 2
  for (int j = tid; j < n_keys; j += 128) {
    const uint4* kr = reinterpret_cast<const uint4*>(kc + static_cast<size_t>(j) * HD);
    float acc[G];
#pragma unroll
    for (int gq = 0; gq < G; ++gq) acc[gq] = 0.f;
#pragma unroll
    for (int c = 0; c < VPR; ++c) {
      uint4 u = kr[c];
      const T* e = reinterpret_cast<const T*>(&u);
      const unsigned short* kb = reinterpret_cast<const unsigned short*>(e);
#pragma unroll
      for (int gq = 0; gq < G; ++gq) {
        // one 16-byte broadcast read of 8 q values (kept in T: they are rounded to T anyway) and 8 mixed-precision FMAs
        // (FHFMA: 16-bit operands, fp32 accumulate, no conversion instructions) — bit-identical to fmaf(float(q), float(k), acc)
        const uint4 qv = *reinterpret_cast<const uint4*>(q_t + gq * HD + c * 8);
        const unsigned short* qb = reinterpret_cast<const unsigned short*>(&qv);
#pragma unroll
        for (int x = 0; x < 8; ++x) acc[gq] = fma16<T>(qb[x], kb[x], acc[gq]);
      }
    }
#pragma unroll
    for (int gq = 0; gq < G; ++gq) {
      float sv = acc[gq] * p.scale;
      sc[gq * p.s_max + j] = sv;
      tmax[gq] = fmaxf(tmax[gq], sv);
    }
  }
#pragma unroll
  for (int gq = 0; gq < G; ++gq) {
    float m = warp_max(tmax[gq]);
    if (lane == 0) s_red[warp][gq] = m;
  }
  __syncthreads();
  if (tid < G) s_max_g[tid] = fmaxf(fmaxf(s_red[0][tid], s_red[1][tid]), fmaxf(s_red[2][tid], s_red[3][tid]));
  __syncthreads();
  float tsum[G];
#pragma unroll
  for (int gq = 0; gq < G; ++gq) tsum[gq] = 0.f;
  for (int j = tid; j < n_keys; j += 128) {
#pragma unroll
    for (int gq = 0; gq < G; ++gq) {
      float pv = __expf(sc[gq * p.s_max + j] - s_max_g[gq]);
      tsum[gq] += pv;
      sc[gq * p.s_max + j] = rnd<T>(pv);
    }
  }
#pragma unroll
  for (int gq = 0; gq < G; ++gq) {
    float s = warp_sum(tsum[gq]);
    if (lane == 0) s_red[warp][gq] = s;
  }
  __syncthreads();
  if (tid < G) s_sum_g[tid] = s_red[0][tid] + s_red[1][tid] + s_red[2][tid] + s_red[3][tid];
  __syncthreads();

  // ---- O = P V : thread = (key group, 8-wide dim chunk)
  const int chunk = tid % VPR, kg = tid / VPR;
  if (kg < NKG) {
    float acc[G][8];
#pragma unroll
    for (int gq = 0; gq < G; ++gq)
#pragma unroll
      for (int x = 0; x < 8; ++x) acc[gq][x] = 0.f;
    // keys in batches of PVU with every V load of the batch issued before the first use: the loop is a DRAM-latency chain
    // otherwise (one dependent 16-byte load per iteration).  (A 256-thread variant that prefetched all K / V rows into
    // registers up front was 18 % slower end to end: it halves the number of resident CTAs.)
    constexpr int PVU = 4;
    for (int j0 = kg; j0 < n_keys; j0 += NKG * PVU) {
      uint4 u[PVU];
#pragma unroll
      for (int t = 0; t < PVU; ++t) {
        const int j = j0 + t * NKG;
        u[t] = j < n_keys ? *reinterpret_cast<const uint4*>(vc + static_cast<size_t>(j) * HD + chunk * 8) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int t = 0; t < PVU; ++t) {
        const int j = j0 + t * NKG;
        if (j >= n_keys) break;
        const unsigned short* vb = reinterpret_cast<const unsigned short*>(&u[t]);
#pragma unroll
        for (int gq = 0; gq < G; ++gq) {
          const unsigned short pb = bits_of<T>(from_f<T>(sc[gq * p.s_max + j]));     // p was rounded to T after the softmax
#pragma unroll
          for (int x = 0; x < 8; ++x) acc[gq][x] = fma16<T>(pb, vb[x], acc[gq][x]);
        }
      }
    }
#pragma unroll
    for (int gq = 0; gq < G; ++gq)
#pragma unroll
      for (int x = 0; x < 8; ++x) red[(kg * G + gq) * HD + chunk * 8 + x] = acc[gq][x];
  }
  __syncthreads();
  T* orow = reinterpret_cast<T*>(p.out) + static_cast<size_t>(b) * p.ldo + (kvh * G) * HD;
  for (int i = tid; i < G * HD; i += 128) {
    float s = 0.f;
#pragma unroll
    for (int k2 = 0; k2 < NKG; ++k2) s += red[k2 * G * HD + i];
    orow[i] = from_f<T>(s / s_sum_g[i / HD]);
  }
}

template <typename T, int HD, int G>
static int launch_decode(const DecodeAttnArgs& a, cudaStream_t st) {
  constexpr int NKG = 128 / (HD / 8);
  size_t smem = (static_cast<size_t>(G) * HD + static_cast<size_t>(NKG) * G * HD + static_cast<size_t>(G) * a.s_max) *
                sizeof(float);
  auto kern = decode_attn_kernel<T, HD, G>;
  static size_t attr = 0;
  if (smem > 48 * 1024 && smem > attr) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      set_error("decode_attn: %zu bytes of shared memory exceed the device limit (s_max too large)", smem);
      return -3;
    }
    attr = smem;
  }
  DecodeKParams p;
  p.qkv = a.qkv; p.ld = a.ld; p.kcache = a.kcache; p.vcache = a.vcache; p.slot = a.slot; p.pos = a.pos;
  p.inv_freq = a.inv_freq; p.out = a.out; p.ldo = a.ldo;
  p.n_heads = a.n_heads; p.n_kv_heads = a.n_kv_heads; p.s_max = a.s_max; p.scale = a.scale;
  dim3 grid(a.batch, a.n_kv_heads), block(128);
  launch_pdl(kern, grid, block, smem, st, p);
  return launch_ok();
}

template <typename T, int HD>
static int dispatch_decode_g(const DecodeAttnArgs& a, cudaStream_t st) {
  int G = a.n_heads / a.n_kv_heads;
  switch (G) {
    case 1: return launch_decode<T, HD, 1>(a, st);
    case 2: return launch_decode<T, HD, 2>(a, st);
    case 4: return launch_decode<T, HD, 4>(a, st);
    case 8: return launch_decode<T, HD, 8>(a, st);
    default: set_error("decode_attn: unsupported GQA group %d (1/2/4/8)", G); return -1;
  }
}

template <typename T>
static int dispatch_decode(const DecodeAttnArgs& a, cudaStream_t st) {
  switch (a.head_dim) {
    case 64: return dispatch_decode_g<T, 64>(a, st);
    case 80: return dispatch_decode_g<T, 80>(a, st);
    case 128: return dispatch_decode_g<T, 128>(a, st);
    default: set_error("decode_attn: unsupported head_dim %d (64/80/128)", a.head_dim); return -1;
  }
}

int decode_attn(const DecodeAttnArgs& a, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  if (a.n_heads % a.n_kv_heads) { set_error("decode_attn: n_heads must be a multiple of n_kv_heads"); return -1; }
  return a.dtype == DT_BF16 ? dispatch_decode<__nv_bfloat16>(a, st) : dispatch_decode<__half>(a, st);
}

}  // namespace sb
