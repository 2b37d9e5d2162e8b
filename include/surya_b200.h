/* surya_b200 — C ABI of libsurya_b200.so (sm_100a).
 *
 * The reference (VikParuchuri/surya v0.14.6) has no FFI: its seam is Python attribute access on
 * `predictor.model` (surya/common/predictor.py:20-29).  Every entry point below replaces one group of
 * library calls (cuBLAS / cuDNN / flash-attn / torch eager) that the reference's nn.Modules make on the
 * hot path; the comment on each cites the reference code it stands in for.  The Python mirrors in
 * surya_b200/*.py bind these through ctypes (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; `*_dev` / unnamed tensor pointers are DEVICE pointers owned by
 * the caller, row-major; `stream` is a cudaStream_t passed as void*; dtype: 0 = bf16, 1 = fp16.
 * Return 0 on success, negative on error (message via sb_last_error()).  No hidden global state besides the
 * per-thread error string; one engine per GPU/thread.
 */
#ifndef SURYA_B200_H
#define SURYA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_DT_BF16 0
#define SB_DT_F16 1

#define SB_ACT_NONE 0
#define SB_ACT_GELU_ERF 1
#define SB_ACT_SILU 2
#define SB_ACT_HARDSWISH 3
#define SB_ACT_RELU 4
#define SB_ACT_GELU_TANH 5

const char* sb_last_error(void);
int sb_version(void);
/* Number of kernels this library has launched in the calling process (all entry points). */
long long sb_launch_count(void);

/* ------------------------------------------------------------------------------------------------ ops
 * nn.Linear (+bias, activation, residual, SwiGLU) : torch.nn.functional.linear -> cuBLAS in the reference,
 * e.g. surya/common/surya/decoder/__init__.py:37-50,147-158; encoder/__init__.py:22-35,140-141,115-119.
 * C[M,Nout] = epi(A[M,K] @ W[N,K]^T).  bias is fp32 [N] or NULL; residual [M,Nout] or NULL.
 * swiglu=1: W rows interleaved (gate_i, up_i), Nout = N/2, out = act(gate)*up.  out_f32: C is float32.
 * force_bn: 0 = tile heuristic; 32/64/96/128/256 = fixed tile width; -1 = heuristic that may also pick the split-K cluster
 * kernel (fp32 partials summed in a fixed order over <= 3 K slices; for decode-sized M <= 256 callers); 1000*pk + BN forces it. */
int sb_gemm(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
            const float* bias, const void* residual, int ldr, int act, int swiglu, int out_f32, int force_bn,
            void* stream);

/* nn.Linear applied to Qwen2RMSNorm(x) with the norm folded into the GEMM (decoder/__init__.py:241-258 followed by
 * :147-158 / :37-50, and the final norm + lm_head / bbox_head of surya/common/surya/__init__.py:323-330):
 *   C = epi(rs[m] * (A W^T) + bias),  W = nn.Linear weight x norm weight per column (packed by the caller),
 *   rs[m] = rsqrt(mean_k A[m,k]^2 + eps): read from `rowscale` (fp32 [M], see sb_row_rstd) or, when rowscale is NULL, computed
 *   inside the kernel from the A tiles with rms_eps (no separate pass over A; used by the decode steps).
 * Optional online argmax epilogue (am_val != NULL): per (row, n-tile) partials (max logit, first argmax, sum exp(l - max)) of
 * the 16-bit-rounded outputs into [M, am_ld] arrays, tile width = sb_gemm_argmax_tile(M, N); C is written only if store_c —
 * RecognitionPredictor.process_outputs (surya/recognition/__init__.py:294-324) needs argmax and max-softmax only. */
int sb_gemm_rmsnorm(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                    const float* bias, const void* residual, int ldr, int act, int swiglu, const float* rowscale, float rms_eps,
                    float* am_val, int* am_idx, float* am_sum, int am_ld, int store_c, int force_bn, void* stream);
int sb_gemm_argmax_tile(int M, int N);
/* rs[row] = rsqrt(mean(x[row]^2) + eps) in the summation order sb_gemm_rmsnorm's in-kernel pass uses (bit-identical). */
int sb_row_rstd(int dtype, const void* x, int ldx, float* rs, int rows, int H, float eps, const int* src_rows, void* stream);

/* sb_gemm with an in-kernel timeline of CTA 0 (globaltimer ns into timeline_dev[0..42]); profiling aid. */
int sb_gemm_timeline(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                     const float* bias, const void* residual, int ldr, int act, int swiglu, int force_bn,
                     unsigned long long* timeline_dev, void* stream);

/* Qwen2RMSNorm (decoder/__init__.py:241-258, encoder/__init__.py:90-104); src_rows optional gather. */
int sb_rmsnorm(int dtype, const void* x, int ldx, const void* w, void* y, int ldy, int rows, int H, float eps,
               const int* src_rows, void* stream);

/* Row gather + zero pad (+ fp32 -> 16-bit conversion): window re-ordering of patch rows
 * (encoder/__init__.py:622-627) fused with the K-padding the TMA pitch rule needs (588 -> 592). */
int sb_gather_pad_rows(int dtype, const void* src, int src_is_f32, int lds, const int* perm, void* dst, int ldd,
                       int rows, int K, int Kp, void* stream);

/* apply_rotary_pos_emb_vision on a fused qkv buffer (encoder/__init__.py:188-199, 523-550). pos_rc = int2 (row,col). */
int sb_rope_vision(int dtype, void* qkv, int ld, const int* pos_rc, const float* inv_freq, int n_tok, int nh, int d,
                   void* stream);

/* apply_rotary_pos_emb (decoder/__init__.py:60-84, 346-361) + DynamicCache.update without the torch.cat
 * (decoder/__init__.py:190-195): rotates q,k in place and writes k,v into cache[slot][kv_head][pos][:]. */
int sb_rope_kv_append(int dtype, void* qkv, int ld, const int* tok_pos, const int* tok_slot, const float* inv_freq,
                      void* kcache, void* vcache, int n_tok, int nh, int nkv, int d, int s_max, void* stream);

/* flash_attn_varlen_func / SDPA over packed sequences (encoder/__init__.py:174-176, 400-406;
 * flash_attn_utils.py:106-154).  Head h of q at column q_col0 + h*d of a row-major matrix with pitch ldq. */
int sb_attn_varlen(int dtype, const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* out,
                   int ldo, const int* seq_start, const int* seq_len, int n_seq, int max_len, int n_heads,
                   int n_kv_heads, int head_dim, int causal, float scale, void* stream);

/* flash_attn_with_kvcache / SDPA decode step (flash_attn_utils.py:157-188) fused with RoPE and cache append. */
int sb_decode_attn(int dtype, const void* qkv, int ld, void* kcache, void* vcache, const int* slot, const int* pos,
                   const float* inv_freq, void* out, int ldo, int batch, int n_heads, int n_kv_heads, int head_dim,
                   int s_max, float scale, void* stream);

/* embed_ids_boxes_images: token embedding + 2-D learned image position embedding + masked_scatter
 * (surya/common/surya/__init__.py:197-272). feat_row[t] < 0 -> plain token embedding. */
int sb_embed_splice(int dtype, const long long* ids, const int* feat_row, const int* hidx, const int* widx,
                    const void* embed, const void* feat, int ldf, const void* h_embed, const void* w_embed,
                    void* out, int ldo, int n_tok, int H, void* stream);
int sb_embed_rows(int dtype, const long long* ids, const void* embed, void* out, int ldo, int n, int H, void* stream);

/* RecognitionPredictor.process_outputs (surya/recognition/__init__.py:294-324): argmax, max-softmax score,
 * done mask, next input id. */
int sb_argmax_score(int dtype, const void* logits, int ld, int rows, int V, long long* tok, float* score,
                    unsigned char* done, long long* next_ids, int eos, int pad, void* stream);

/* bbox_head + sigmoid (+ trunc(sig * bbox_size)) (surya/common/surya/__init__.py:329; recognition/__init__.py:315-316). */
int sb_small_head(int dtype, const void* x, int ldx, const void* w, const void* b, int rows, int H, int n_out,
                  int sigmoid, float* out_f, long long* out_box, float box_scale, void* stream);


/* ------------------------------------------------------------------------------------------------ recognition engine
 * Replaces SuryaModel.forward (surya/common/surya/__init__.py:274-338) as driven by RecognitionPredictor.prefill /
 * decode (surya/recognition/__init__.py:326-352, 354-471) and the ContinuousBatchingCache
 * (surya/recognition/cache.py:7-105): the engine owns a slot-indexed KV cache [layer][slot][kv_head][s_max][d];
 * sequences are processed ragged (no left padding), which is observationally equivalent because RoPE uses
 * per-row position_ids (SURVEY.md §9.5).  All tensor/array pointers are DEVICE pointers unless named *_host. */
typedef struct sb_rec_engine sb_rec_engine;

typedef struct {
  int dtype;                 /* SB_DT_BF16 / SB_DT_F16 */
  /* vision tower (surya/common/surya/encoder/config.py:16-34) */
  int enc_depth, enc_hidden, enc_heads, enc_inter, enc_inter_pad;
  int patch_dim, patch_dim_pad, merge_unit /* spatial_merge_size^2 */, enc_out_hidden;
  unsigned int fullatt_mask; /* bit i set -> block i attends per image, else per window */
  /* decoder (surya/common/surya/decoder/config.py:30-49) */
  int dec_layers, dec_hidden, dec_heads, dec_kv_heads, dec_head_dim, dec_inter, dec_inter_pad;
  float rms_eps;
  int vocab, eos_id, pad_id;
  float bbox_size;
  /* capacities */
  int max_slots, s_max, max_patches, max_tokens, max_seqs;
} sb_rec_config;

/* Weight table: device pointers in the order given by the SB_RW_* indices (16-bit weights in cfg.dtype unless
 * noted fp32).  Per-layer entries are strided: index = base + layer * stride + k. */
enum {
  SB_RW_PATCH_W = 0,      /* [enc_hidden, patch_dim_pad] */
  SB_RW_MERGER_LN,        /* [enc_hidden] */
  SB_RW_MERGER_W0, SB_RW_MERGER_B0 /* fp32 */, SB_RW_MERGER_W2, SB_RW_MERGER_B2 /* fp32 */,
  SB_RW_ENC_INV_FREQ,     /* fp32 [head_dim/4] */
  SB_RW_LM_W,             /* [vocab, dec_hidden] lm_head weight (= token embedding, tied) x decoder.norm.weight per column */
  SB_RW_EMBED,            /* [vocab, dec_hidden] token embedding (input lookups) */
  SB_RW_LM_BIAS,          /* fp32 [vocab] */
  SB_RW_BBOX_W, SB_RW_BBOX_B, /* [6, dec_hidden] x decoder.norm.weight per column, [6] */
  SB_RW_H_EMBED, SB_RW_W_EMBED, /* [enc_size, dec_hidden] */
  SB_RW_DEC_INV_FREQ,     /* fp32 [head_dim/2] */
  SB_RW_ENC_BASE,         /* first per-block entry of the vision tower */
  SB_RW_COUNT_FIXED = SB_RW_ENC_BASE
};
enum { /* per vision block */
  SB_RWE_NORM1 = 0, SB_RWE_QKV_W, SB_RWE_QKV_B /* fp32 */, SB_RWE_PROJ_W, SB_RWE_PROJ_B /* fp32 */, SB_RWE_NORM2,
  SB_RWE_GU_W /* [2*inter_pad, hidden] gate/up interleaved */, SB_RWE_GU_B /* fp32 */, SB_RWE_DOWN_W /* [hidden, inter_pad] */,
  SB_RWE_DOWN_B /* fp32 */, SB_RWE_STRIDE
};
enum { /* per decoder layer (base = SB_RW_ENC_BASE + enc_depth * SB_RWE_STRIDE).  The decoder's RMSNorm weights are folded
        * into the GEMM that consumes the normalised activations: W'[n,k] = W[n,k] * g[k] (rounded once to cfg.dtype); the
        * kernels apply the per-row 1/rms in the GEMM epilogue (decoder/__init__.py:241-258, 288-310). */
  SB_RWD_QKV_W = 0 /* [(nh+2nkv)*d, hidden] x input_layernorm.weight */, SB_RWD_QKV_B /* fp32 */, SB_RWD_O_W,
  SB_RWD_GU_W /* gate/up interleaved, x post_attention_layernorm.weight */, SB_RWD_DOWN_W, SB_RWD_STRIDE
};

int sb_rec_create(const sb_rec_config* cfg, const void* const* weights, int n_weights, sb_rec_engine** out);
void sb_rec_destroy(sb_rec_engine* eng);
size_t sb_rec_workspace_bytes(const sb_rec_engine* eng);

/* Vision tower + decoder prefill for n_seq new sequences (= RecognitionPredictor.prefill's model call).
 *   tiles [n_patches, patch_dim] (cfg.dtype, or fp32 when tiles_f32), patch_perm = window order source rows,
 *   patch_pos_rc = int2 (row, col) per permuted patch; windows / images given as (start, len) in permuted rows;
 *   input_ids: the n_tok REAL tokens of all sequences back to back; tok_feat_row[t] = merged-feature row for an
 *   image token (in permuted/merged order) or -1; tok_hidx/tok_widx = learned 2-D embedding rows;
 *   tok_pos = position id, tok_slot = KV slot; seqs as (start, len); last_tok[s] = index of the last token.
 * Outputs per sequence (any may be NULL): logits [n_seq, vocab] cfg.dtype, token i64, score f32,
 *   bbox i64 [n_seq,6] = trunc(sigmoid * bbox_size), bbox_sig f32 [n_seq,6], done u8, next_ids i64. */
int sb_rec_prefill(sb_rec_engine* eng, const void* tiles, int tiles_f32, int n_patches, const int* patch_perm,
                   const int* patch_pos_rc, const int* win_start, const int* win_len, int n_win, int max_win_len,
                   const int* img_start, const int* img_len, int n_img, int max_img_len, const long long* input_ids,
                   int n_tok, const int* tok_feat_row, const int* tok_hidx, const int* tok_widx, const int* tok_pos,
                   const int* tok_slot, const int* seq_start, const int* seq_len, int n_seq, int max_seq_len,
                   const int* last_tok, void* logits, long long* tok, float* score, long long* bbox, float* bbox_sig,
                   unsigned char* done, long long* next_ids, void* stream);

/* One decode step for `batch` rows (= RecognitionPredictor.decode's model call + process_outputs):
 * row b feeds input_ids[b] at position pos[b] of KV slot slot[b]. */
int sb_rec_decode(sb_rec_engine* eng, const long long* input_ids, const int* slot, const int* pos, int batch,
                  void* logits, long long* tok, float* score, long long* bbox, float* bbox_sig, unsigned char* done,
                  long long* next_ids, void* stream);

/* n_steps greedy steps kept on the device (CUDA-graph replay): ids_io/pos_io are updated in place
 * (ids <- next input id, pos += 1); outputs are step-major [n_steps, batch(,6)]. */
int sb_rec_decode_steps(sb_rec_engine* eng, long long* ids_io, const int* slot, int* pos_io, int batch, int n_steps,
                        long long* tok_hist, float* score_hist, long long* bbox_hist, unsigned char* done_hist,
                        int use_graph, void* stream);

/* Recognition crop preprocessing on the device (SURVEY §8 f2): SuryaOCRProcessor.scale_to_fit (cv2 INTER_LANCZOS4 when the pixel
 * count is outside [168*168, 1024*256], surya/common/surya/processor/__init__.py:140-178) + _process_and_tile (cv2 INTER_CUBIC to the
 * next multiple of patch*merge, x*(1/255) in double, (x - mean)/std in float, merge-block-major tiles, :180-230) for n_crops uint8 HWC
 * crops packed in `crops_u8` (device).  desc: n_crops x 9 int32 (device) = {byte offset of the crop, h, w, nh, nw (size after
 * scale_to_fit, = h, w when it does not apply), hb, wb (multiples of patch*merge), float offset of the crop's [nh, nw, 3] intermediate
 * in `scratch`, first tile row}; the host computes the sizes with the reference's own Python arithmetic.  tiles: fp32
 * [rows, ld_tiles >= 3*patch*patch] (device), exactly the `image_tiles` sb_rec_prefill takes with tiles_f32 = 1.  mean3 / std3: host. */
int sb_rec_preprocess(const unsigned char* crops_u8, const int* desc, int n_crops, int max_nh, int max_nw, int max_hb, int max_wb,
                      int any_scale_to_fit, float* scratch, float* tiles, int ld_tiles, int patch, int merge, const float* mean3,
                      const float* std3, void* stream);

/* Device-side scheduler state of the continuous-batching loop (SURVEY §8 f3): the stop rules of
 * RecognitionPredictor.prediction_loop (surya/recognition/__init__.py:568-601 — EOS / PAD, len >= max_tokens,
 * detect_repeat_token of surya/recognition/util.py:59-69) evaluated by a kernel after every step of sb_rec_decode_steps instead of
 * a per-token loop on the host.  All arrays are caller-owned DEVICE memory of `batch` rows (ring: batch x max_repeats):
 *   gen_count  tokens generated so far per row (seed 1 after prefill: the prefill token counts);
 *   ring       the row's last max_repeats tokens, token i at slot i % max_repeats (seed slot 0 with the prefill token);
 *   row_done   sticky stop flag (seed 1 for idle rows, 0 for running rows);
 *   n_valid    out: per row, how many steps of the current sb_rec_decode_steps call belong to it (1 + index of its stopping step);
 *   n_active   out (may be NULL): rows still running after the last step.
 * gen_count == NULL switches the rules off again.  Changing the state invalidates the captured decode graph. */
int sb_rec_set_sched(sb_rec_engine* eng, int* gen_count, long long* ring, unsigned char* row_done, int* n_valid, int* n_active,
                     int max_tokens, int max_repeats);
/* One evaluation of the same rules on explicit histories ([T, batch] layouts of sb_rec_decode_steps) for host step `step`. */
int sb_rec_stop_rules(const long long* tok_hist, const unsigned char* done_hist, int step, int batch, int* gen_count, long long* ring,
                      unsigned char* row_done, int* n_valid, int* n_active, int max_tokens, int max_repeats, void* stream);
/* Parity taps: copy `bytes` of a named workspace ("feat" = merged image features in window order before the
 * 2-D position embedding, "x", "xl", "logits", "qkv") into dst (device). */
int sb_rec_debug_copy(sb_rec_engine* eng, const char* name, void* dst, size_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------------ detection engine
 * Replaces EfficientViTForSemanticSegmentation.forward (surya/detection/model/encoderdecoder.py:725-753) as called by
 * DetectionPredictor.batch_detection (surya/detection/__init__.py:111-120), plus the predictor's x4 bilinear upsample
 * (:120-129).  The network is handed over as a flat op program (built by surya_b200/detection.py from the config the
 * way the reference assembles its modules) over NHWC activations; BatchNorm is folded into weights at pack time. */
typedef struct sb_det_engine sb_det_engine;

enum { SB_DOP_STEM = 0, SB_DOP_CONV = 1, SB_DOP_PW = 2, SB_DOP_DW = 3, SB_DOP_GPW = 4, SB_DOP_MLA = 5, SB_DOP_UPCAT = 6,
       SB_DOP_CLS = 7 };

typedef struct {
  int op;                 /* SB_DOP_* */
  int src[4];             /* input buffer ids (src[0] = main input; -2 = external pixel_values) */
  int n_src;
  int src_off[4];         /* UPCAT: channel offset of each source in the concatenated output */
  int dst;                /* output buffer id (-3 = external logits) */
  int res;                /* residual buffer id or -1 */
  int w, b;               /* weight-table indices (-1 = none) */
  int cin, cout, k, stride, pad, act, groups;
  int heads, dim;         /* MLA */
  float eps;              /* MLA */
} sb_det_op;

/* weights: device pointers (see surya_b200/detection.py:pack_det_weights for the per-op layouts);
 * buf_elems[i]: capacity of workspace buffer i in elements PER IMAGE at the maximum resolution. */
int sb_det_create(int dtype, const sb_det_op* ops, int n_ops, const void* const* weights, int n_weights,
                  const long long* buf_elems, int n_bufs, int max_batch, sb_det_engine** out);
void sb_det_destroy(sb_det_engine* eng);
size_t sb_det_workspace_bytes(const sb_det_engine* eng);
/* pixel_values: NCHW [B,3,H,W] (engine dtype, or fp32 when in_f32); logits: NCHW [B, num_labels, H/4, W/4] engine dtype. */
int sb_det_forward(sb_det_engine* eng, const void* pixel_values, int in_f32, int B, int H, int W, void* logits,
                   void* stream);
/* F.interpolate(logits, size=(HO, WO), mode="bilinear").float() : NCHW fp32 out (surya/detection/__init__.py:120-132). */
int sb_det_upsample(int dtype, const void* logits, float* out, int planes, int hs, int ws, int HO, int WO, void* stream);
/* SegformerImageProcessor's rescale + normalise on the device (surya/detection/processor.py:94-95, 126-146):
 * uint8 NHWC [B,H,W,3] -> NCHW engine dtype, x = (u8 / 255 - mean) / std in fp32 with the ImageNet default mean / std. */
int sb_det_normalize_u8(int dtype, const unsigned char* pages_nhwc, void* out_nchw, int B, int H, int W, void* stream);
/* Front half of the detection post-processing on the device, TEXT channel only (surya/detection/__init__.py:120-132 upsample +
 * .float(); surya/detection/heatmap.py:14-24 get_dynamic_thresholds; :33 `linemap > low_text`):
 *   map16      [B, HO, WO] engine-dtype image of F.interpolate(logits[:, 0]) — exactly the values the reference casts to fp32
 *   mask       [B, HO, WO] uint8 = map > low_text(page)          (input of cv2.connectedComponentsWithStats)
 *   thresholds [B, 4] fp32 = text_threshold, low_text, top-10 % mean, scaling factor (per page)
 *   hist_scratch [B, 16384] uint32, zero on entry, zero on exit
 * 3 bytes per pixel leave the device instead of 8 and the host no longer partitions a megapixel per page. */
int sb_det_text_front(int dtype, const void* logits, int n_labels, int B, int hs, int ws, int HO, int WO, void* map16,
                      unsigned char* mask, float* thresholds, unsigned int* hist_scratch, float text_threshold, float low_text,
                      void* stream);
/* parity tap: copy workspace buffer `buf` (NHWC) into dst. */
int sb_det_debug_copy(sb_det_engine* eng, int buf, void* dst, size_t bytes, void* stream);

/* k x k dense convolution, NHWC, implicit GEMM on tcgen05 (op-level entry point used by the kernel tests). */
int sb_conv2d_nhwc(int dtype, const void* in, const void* weight, const float* bias, const void* residual, void* out,
                   int n_img, int H, int W, int Cin, int Cout, int ksize, int stride, int pad, int act, void* stream);
int sb_dwconv_nhwc(int dtype, const void* in, const void* w, const float* bias, void* out, int B, int H, int W, int C,
                   int ks, int stride, int pad, int act, void* stream);
int sb_gemm_grouped(int dtype, const void* A, int lda, int a_cols, const void* W, int ldw, void* C, int ldc, int M, int N,
                    int Kpad, int group_k, int group_n, void* stream);
int sb_lite_mla(int dtype, const void* qkv_a, const void* qkv_b, void* out, int B, int HW, int heads, int dim, float eps,
                void* stream);

/* ------------------------------------------------------------------------------------------------ layout / table_rec ops
 * Donut-Swin encoder (surya/common/donut/encoder.py) and ADETR decoder (surya/common/adetr/decoder.py) pieces that the
 * recognition / detection entry points above do not already cover; the layer loops are driven from
 * surya_b200/layout.py (round 1: correctness first, C++ engine-isation is the next step). */
/* SuryaADETRDecoderRMSNorm (adetr/decoder.py:29-47): T(clamp(x * rsqrt(max(mean(x^2), eps)) * (1 + w))). */
int sb_rmsnorm_adetr(int dtype, const void* x, int ldx, const void* w, void* y, int ldy, int rows, int H, float eps,
                     void* stream);
/* nn.LayerNorm (donut/encoder.py:117,163,544-548; layout/model/decoder.py:73). */
int sb_layernorm(int dtype, const void* x, const void* w, const void* b, void* y, int rows, int C, float eps, void* stream);
/* ocr_error (SURVEY §8 f4) — Embeddings.forward of DistilBertForSequenceClassification (surya/ocr_error/model/encoder.py:60-91):
 * y[r] = LayerNorm(T(word[ids[r]] + ptab[pos[r]])) for the PACKED real tokens of a right-padded batch; ids / pos are int32 device
 * arrays of `rows` entries (the host plan drops the pad positions, which the reference computes and then masks, :171-175).  The
 * rest of the model runs on sb_gemm (q/k/v fused, out_lin + residual, lin1 + GELU, lin2 + residual, pre_classifier + ReLU),
 * sb_attn_varlen (non-causal, one segment per text), sb_layernorm and sb_small_head (classifier): surya_b200/ocr_error.py. */
int sb_embed_pos_layernorm(int dtype, const int* ids, const int* pos, const void* word, const void* ptab, const void* w,
                           const void* b, void* y, int rows, int C, float eps, void* stream);
/* im2col of the patch-embedding Conv2d(k = stride = P) (donut/encoder.py:228-230): NCHW -> [B*gh*gw, Kp], col = c*P*P+ky*P+kx;
 * gh = ceil(H/P), gw = ceil(W/P), a partial last patch is zero filled (DonutSwinPatchEmbeddings.maybe_pad, :232-239). */
int sb_patch_gather(int dtype, const void* in, int in_f32, void* out, int B, int Cin, int H, int W, int P, int Kp, void* stream);
/* x[b, t, :] += tab[t, :] (stage sin-cos table donut/encoder.py:773-776; position_embeddings layout/model/encoder.py:76-77). */
int sb_add_bcast_rows(int dtype, void* x, const void* tab, long long rows, int rows_per_batch, int C, void* stream);
/* DonutSwinPatchMerging's 2x2 gather (donut/encoder.py:301-312): [B,H,W,C] -> [B,ceil(H/2),ceil(W/2),4C]; an odd H / W is zero
 * padded (maybe_pad, :281-287). */
int sb_patch_merge_gather(int dtype, const void* x, void* y, int B, int H, int W, int C, void* stream);
/* DonutSwinLayer attention core (donut/encoder.py:383-442, 562-590, 598-664): 8x8 windows, cyclic shift, relative-position
 * bias table [225, nh], -100 shift mask; qkv [B*H*W, 3C] and out [B*H*W, C] in natural token order.  H / W that are not multiples
 * of 8 are zero padded to the window like maybe_pad (:591-596, crop :657-659): a pad token's q/k/v is the fp32 QKV bias
 * `qkv_bias` [3C] (required then, may be NULL otherwise).  H, W < 8 is an error (the reference's own bias table breaks there). */
int sb_swin_window_attn(int dtype, const void* qkv, const float* qkv_bias, const void* bias_table, void* out, int B, int H, int W,
                        int C, int nh, int shift, void* stream);
/* BboxEmbedding (layout/model/decoder.py:36-57): tables = 15 device pointers (w,h,cx,cy,xskew,yskew,x1,y1,...,y4,label). */
int sb_bbox_embed_sum(int dtype, const long long* boxes, const void* const* tables, void* out, int n, int Hd, int bbox_size,
                      void* stream);
/* q_len = 1 attention over a fixed K/V set with explicit strides (ADETR cross-attention, adetr/decoder.py:150-194). */
int sb_attn_single_query(int dtype, const void* q, int ldq, const void* K, const void* V, long long batch_stride,
                         long long head_stride, long long token_stride, void* out, int ldo, int B, int nh, int nkv, int head_dim,
                         int n_keys, float scale, void* stream);
/* LabelEmbedding (table_rec/model/decoder.py:46-73): boxes int64 [n,10]; tables = 13 device pointers (w,h,cx,cy,xskew,yskew,
 * x1,y1,x3,y3 of width box_w; category, merge, colspan of width prop_w); out [n, box_w + prop_w]. */
int sb_label_embed(int dtype, const long long* boxes, const void* const* tables, void* out, int n, int box_w, int prop_w,
                   int bbox_size, int vocab, void* stream);
/* Per-step token formation of LayoutPredictor / TableRecPredictor (layout/__init__.py:125-137; table_rec/__init__.py:76-97 +
 * shaper.py:12-52): out int64 [B, 6 + n_heads] = trunc(clamp(bbox * bbox_size)) x6, then per head argmax (mode 0) or
 * round(max(v, 1)) (mode 1, colspan); done[b] = head `done_head`'s token is eos or pad (may be NULL).
 * Optional loop state (all may be NULL) so a whole decode step can be replayed as a CUDA graph: cache_pos[b] += 1
 * (decoder_position_ids + 1, layout/__init__.py:124, table_rec/__init__.py:71) after the step's tokens [hist_T][B][6+n_heads],
 * bbox [hist_T][B][6], raw head outputs [hist_T][B][n_k] and done flags were appended at row cache_pos[b] - hist_base[0]. */
int sb_box_next_token(const float* bbox, const float* const* heads, const int* head_n, const int* head_mode, int n_heads,
                      float bbox_size, long long* out, unsigned char* done, int done_head, int eos, int pad, int B, int* cache_pos,
                      const int* hist_base, int hist_T, long long* hist_tok, float* hist_bbox, float* const* hist_heads,
                      unsigned char* hist_done, void* stream);

/* ------------------------------------------------------------------------------------------------ layout / table_rec engine
 * Donut-Swin encoder + ADETR box decoder with the layer loops, workspaces, K/V caches and the greedy loop in C++
 * (DonutSwinLayoutModel / DonutSwinModel.forward, surya/layout/model/encoder.py:33-81, surya/table_rec/model/encoder.py:35-87;
 * SuryaLayoutDecoder / SuryaTableRecDecoder.forward, surya/layout/model/decoder.py:95-126, surya/table_rec/model/decoder.py:121-155;
 * the predictors' step loops, surya/layout/__init__.py:106-137, surya/table_rec/__init__.py:33-131).
 * Weight table (device pointers; 16-bit tensors in the engine dtype unless marked f32):
 *   [SB_LW_PE_W] patch-embed weight [embed_dim, Kp] (K = in_ch*patch^2 zero-padded to a multiple of 64), [SB_LW_PE_B] bias f32,
 *   [SB_LW_PE_LN_W/B] embeddings.norm, [SB_LW_ENC_POS] position_embeddings [enc_len, hidden];
 *   per stage: sin-cos table [H*W, C]; per layer SB_LW_ENC_LAYER tensors in SB_LWE_* order (fused qkv [3C, C] + f32 bias,
 *   relative_position_bias_table [225, nh], ...); per non-final stage: downsample.norm w, b, reduction [2C, 4C];
 *   decoder: embedding tables (layout 15: w,h,cx,cy,xskew,yskew,x1..y4,label; table 13: w,h,cx,cy,xskew,yskew,x1,y1,x3,y3,
 *   category,merge,colspan); per layer SB_LW_DEC_LAYER tensors in SB_LWD_* order (cross K|V fused [2*n_kv*64, enc_hidden],
 *   self q|k|v fused, gate/up rows interleaved); tail in SB_LWX_* order (inv_freq f32);
 *   heads: layout bbox_w, bbox_b, class_w; table bbox, category, merges, colspan, is_header. */
enum { SB_LW_PE_W = 0, SB_LW_PE_B, SB_LW_PE_LN_W, SB_LW_PE_LN_B, SB_LW_ENC_POS, SB_LW_ENC_FIXED };
enum { SB_LWE_LN1_W = 0, SB_LWE_LN1_B, SB_LWE_QKV_W, SB_LWE_QKV_B, SB_LWE_RPB, SB_LWE_O_W, SB_LWE_O_B, SB_LWE_LN2_W, SB_LWE_LN2_B,
       SB_LWE_FC1_W, SB_LWE_FC1_B, SB_LWE_FC2_W, SB_LWE_FC2_B, SB_LW_ENC_LAYER };
enum { SB_LW_ENC_MERGE = 3 };
enum { SB_LWD_CROSS_NORM = 0, SB_LWD_SELF_NORM, SB_LWD_MLP_NORM, SB_LWD_CQ_W, SB_LWD_CKV_W, SB_LWD_CO_W, SB_LWD_CO_B, SB_LWD_SQKV_W,
       SB_LWD_SO_W, SB_LWD_SO_B, SB_LWD_GU_W, SB_LWD_DOWN_W, SB_LW_DEC_LAYER };
enum { SB_LWX_FINAL_NORM = 0, SB_LWX_OUT_LN_W, SB_LWX_OUT_LN_B, SB_LWX_INV_FREQ, SB_LW_DEC_TAIL };

typedef struct sb_layout_config {
  int dtype;                                   /* SB_DT_* */
  int img_h, img_w, patch, in_ch, embed_dim, n_stages, depths[4], heads[4], window;
  float enc_ln_eps;
  int kind;                                    /* 0 = layout (BboxEmbedding, double residual flow), 1 = table_rec (LabelEmbedding) */
  int dec_layers, hidden, inter, enc_hidden, n_heads, n_kv, head_dim;
  float rms_eps, dec_ln_eps;
  int double_residual, bbox_size, vocab, box_w, prop_w;
  int n_out_heads, head_n[4];                  /* layout: {label_count}; table: {category, merges, 1 (colspan), is_header} */
  int eos, pad;
  int max_batch, s_max;
} sb_layout_config;
typedef struct sb_layout_engine sb_layout_engine;

int sb_layout_create(const sb_layout_config* cfg, const void* const* weights, int n_weights, sb_layout_engine** out);
void sb_layout_destroy(sb_layout_engine* e);
size_t sb_layout_workspace_bytes(const sb_layout_engine* e);
/* pixels NCHW [batch, in_ch, img_h, img_w] (engine dtype, or float32 when pixels_f32) -> enc_out [batch, Lk, hidden]. */
int sb_layout_encode(sb_layout_engine* e, const void* pixels, int pixels_f32, int batch, void* enc_out, void* stream);
/* One whole greedy pass on the device: cross K/V of `enc`, prompt [batch, q_len, 6 + n_out_heads] int64 fed position by
 * position, then n_steps tokens (token formation, position advance and history append in sb_box_next_token's kernel; steps
 * replayed as CUDA graphs of 8).  Histories (device): tok [n_steps, batch, ncol] i64, bbox [n_steps, batch, 6] f32,
 * heads[k] [n_steps, batch, head_n[k]] f32, done [n_steps, batch] u8 (may be NULL for layout). */
int sb_layout_decode(sb_layout_engine* e, const void* enc, int batch, const long long* prompt, int q_len, int n_steps,
                     long long* hist_tok, float* hist_bbox, float* const* hist_heads, unsigned char* hist_done, int use_graph,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SURYA_B200_H */
