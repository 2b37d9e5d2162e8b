// surya_b200 — extern "C" surface (op level). Engine-level entry points live in rec_engine.cu / det_engine.cu.
#include "../../include/surya_b200.h"
#include "ops.cuh"

using namespace sb;

extern "C" {

const char* sb_last_error(void) { return last_error(); }
int sb_version(void) { return 1; }
long long sb_launch_count(void) { return launch_count(); }

int sb_gemm(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
            const float* bias, const void* residual, int ldr, int act, int swiglu, int out_f32, int force_bn,
            void* stream) {
  GemmArgs a;
  a.dtype = dtype; a.A = A; a.lda = lda; a.W = W; a.ldw = ldw; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K; a.bias = bias; a.residual = residual; a.ldr = ldr;
  a.act = act; a.swiglu = swiglu; a.out_f32 = out_f32;
  a.force_bn = force_bn < 0 ? 0 : force_bn;
  a.allow_splitk = force_bn < 0 ? 1 : 0;
  return gemm_launch(a, static_cast<cudaStream_t>(stream));
}

int sb_gemm_rmsnorm(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                    const float* bias, const void* residual, int ldr, int act, int swiglu, const float* rowscale, float rms_eps,
                    float* am_val, int* am_idx, float* am_sum, int am_ld, int store_c, int force_bn, void* stream) {
  GemmArgs a;
  a.dtype = dtype; a.A = A; a.lda = lda; a.W = W; a.ldw = ldw; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K; a.bias = bias; a.residual = residual; a.ldr = ldr;
  a.act = act; a.swiglu = swiglu;
  a.force_bn = force_bn;
  a.rowscale = rowscale;
  if (!rowscale) { a.ssq_inline = 1; a.ssq_eps = rms_eps; a.ssq_k = K; }
  a.am_val = am_val; a.am_idx = am_idx; a.am_sum = am_sum; a.am_ld = am_ld;
  a.store_c = am_val ? store_c : 1;
  return gemm_launch(a, static_cast<cudaStream_t>(stream));
}

int sb_gemm_argmax_tile(int M, int N) { return gemm_argmax_tile(M, N); }

int sb_row_rstd(int dtype, const void* x, int ldx, float* rs, int rows, int H, float eps, const int* src_rows, void* stream) {
  return row_rstd(dtype, x, ldx, rs, rows, H, eps, src_rows, static_cast<cudaStream_t>(stream));
}

int sb_gemm_timeline(int dtype, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                     const float* bias, const void* residual, int ldr, int act, int swiglu, int force_bn,
                     unsigned long long* timeline_dev, void* stream) {
  GemmArgs a;
  a.dtype = dtype; a.A = A; a.lda = lda; a.W = W; a.ldw = ldw; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K; a.bias = bias; a.residual = residual; a.ldr = ldr;
  a.act = act; a.swiglu = swiglu; a.force_bn = force_bn; a.dbg = timeline_dev;
  return gemm_launch(a, static_cast<cudaStream_t>(stream));
}

int sb_rmsnorm(int dtype, const void* x, int ldx, const void* w, void* y, int ldy, int rows, int H, float eps,
               const int* src_rows, void* stream) {
  return rmsnorm(dtype, x, ldx, w, y, ldy, rows, H, eps, src_rows, static_cast<cudaStream_t>(stream));
}

int sb_gather_pad_rows(int dtype, const void* src, int src_is_f32, int lds, const int* perm, void* dst, int ldd,
                       int rows, int K, int Kp, void* stream) {
  return gather_pad_rows(dtype, src, src_is_f32, lds, perm, dst, ldd, rows, K, Kp, static_cast<cudaStream_t>(stream));
}

int sb_rope_vision(int dtype, void* qkv, int ld, const int* pos_rc, const float* inv_freq, int n_tok, int nh, int d,
                   void* stream) {
  return rope_vision(dtype, qkv, ld, pos_rc, inv_freq, n_tok, nh, d, static_cast<cudaStream_t>(stream));
}

int sb_rope_kv_append(int dtype, void* qkv, int ld, const int* tok_pos, const int* tok_slot, const float* inv_freq,
                      void* kcache, void* vcache, int n_tok, int nh, int nkv, int d, int s_max, void* stream) {
  return rope_kv_append(dtype, qkv, ld, tok_pos, tok_slot, inv_freq, kcache, vcache, n_tok, nh, nkv, d, s_max,
                        static_cast<cudaStream_t>(stream));
}

int sb_attn_varlen(int dtype, const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* out,
                   int ldo, const int* seq_start, const int* seq_len, int n_seq, int max_len, int n_heads,
                   int n_kv_heads, int head_dim, int causal, float scale, void* stream) {
  AttnArgs a;
  a.dtype = dtype; a.q = q; a.ldq = ldq; a.k = k; a.ldk = ldk; a.v = v; a.ldv = ldv; a.out = out; a.ldo = ldo;
  a.seq_start = seq_start; a.seq_len = seq_len; a.n_seq = n_seq; a.max_len = max_len;
  a.n_heads = n_heads; a.n_kv_heads = n_kv_heads; a.head_dim = head_dim; a.causal = causal; a.scale = scale;
  return attn_varlen(a, static_cast<cudaStream_t>(stream));
}

int sb_decode_attn(int dtype, const void* qkv, int ld, void* kcache, void* vcache, const int* slot, const int* pos,
                   const float* inv_freq, void* out, int ldo, int batch, int n_heads, int n_kv_heads, int head_dim,
                   int s_max, float scale, void* stream) {
  DecodeAttnArgs a;
  a.dtype = dtype; a.qkv = qkv; a.ld = ld; a.kcache = kcache; a.vcache = vcache; a.slot = slot; a.pos = pos;
  a.inv_freq = inv_freq; a.out = out; a.ldo = ldo; a.batch = batch; a.n_heads = n_heads; a.n_kv_heads = n_kv_heads;
  a.head_dim = head_dim; a.s_max = s_max; a.scale = scale;
  return decode_attn(a, static_cast<cudaStream_t>(stream));
}

int sb_embed_splice(int dtype, const long long* ids, const int* feat_row, const int* hidx, const int* widx,
                    const void* embed, const void* feat, int ldf, const void* h_embed, const void* w_embed,
                    void* out, int ldo, int n_tok, int H, void* stream) {
  return embed_splice(dtype, ids, feat_row, hidx, widx, embed, feat, ldf, h_embed, w_embed, out, ldo, n_tok, H,
                      static_cast<cudaStream_t>(stream));
}

int sb_embed_rows(int dtype, const long long* ids, const void* embed, void* out, int ldo, int n, int H, void* stream) {
  return embed_rows(dtype, ids, embed, out, ldo, n, H, static_cast<cudaStream_t>(stream));
}

int sb_argmax_score(int dtype, const void* logits, int ld, int rows, int V, long long* tok, float* score,
                    unsigned char* done, long long* next_ids, int eos, int pad, void* stream) {
  return argmax_score(dtype, logits, ld, rows, V, tok, score, done, next_ids, eos, pad,
                      static_cast<cudaStream_t>(stream));
}

int sb_small_head(int dtype, const void* x, int ldx, const void* w, const void* b, int rows, int H, int n_out,
                  int sigmoid, float* out_f, long long* out_box, float box_scale, void* stream) {
  return small_head(dtype, x, ldx, w, b, rows, H, n_out, sigmoid, out_f, out_box, box_scale,
                    static_cast<cudaStream_t>(stream));
}

int sb_rec_preprocess(const unsigned char* crops_u8, const int* desc, int n_crops, int max_nh, int max_nw, int max_hb, int max_wb,
                      int any_scale_to_fit, float* scratch, float* tiles, int ld_tiles, int patch, int merge, const float* mean3,
                      const float* std3, void* stream) {
  return rec_preprocess(crops_u8, desc, n_crops, max_nh, max_nw, max_hb, max_wb, any_scale_to_fit, scratch, tiles, ld_tiles, patch, merge,
                        mean3, std3, static_cast<cudaStream_t>(stream));
}

int sb_rec_stop_rules(const long long* tok_hist, const unsigned char* done_hist, int step, int batch, int* gen_count, long long* ring,
                      unsigned char* row_done, int* n_valid, int* n_active, int max_tokens, int max_repeats, void* stream) {
  return stop_rules(tok_hist, done_hist, nullptr, step, batch, gen_count, ring, row_done, n_valid, n_active, max_tokens, max_repeats,
                    static_cast<cudaStream_t>(stream));
}

int sb_rmsnorm_adetr(int dtype, const void* x, int ldx, const void* w, void* y, int ldy, int rows, int H, float eps,
                     void* stream) {
  return rmsnorm(dtype, x, ldx, w, y, ldy, rows, H, eps, nullptr, static_cast<cudaStream_t>(stream), 1);
}
int sb_layernorm(int dtype, const void* x, const void* w, const void* b, void* y, int rows, int C, float eps, void* stream) {
  return layernorm(dtype, x, w, b, y, rows, C, eps, static_cast<cudaStream_t>(stream));
}
int sb_embed_pos_layernorm(int dtype, const int* ids, const int* pos, const void* word, const void* ptab, const void* w,
                           const void* b, void* y, int rows, int C, float eps, void* stream) {
  return embed_pos_layernorm(dtype, ids, pos, word, ptab, w, b, y, rows, C, eps, static_cast<cudaStream_t>(stream));
}
int sb_patch_gather(int dtype, const void* in, int in_f32, void* out, int B, int Cin, int H, int W, int P, int Kp, void* stream) {
  return patch_gather(dtype, in, in_f32, out, B, Cin, H, W, P, Kp, static_cast<cudaStream_t>(stream));
}
int sb_add_bcast_rows(int dtype, void* x, const void* tab, long long rows, int rows_per_batch, int C, void* stream) {
  return add_bcast_rows(dtype, x, tab, rows, rows_per_batch, C, static_cast<cudaStream_t>(stream));
}
int sb_patch_merge_gather(int dtype, const void* x, void* y, int B, int H, int W, int C, void* stream) {
  return patch_merge_gather(dtype, x, y, B, H, W, C, static_cast<cudaStream_t>(stream));
}
int sb_swin_window_attn(int dtype, const void* qkv, const float* qkv_bias, const void* bias_table, void* out, int B, int H, int W,
                        int C, int nh, int shift, void* stream) {
  return swin_window_attn(dtype, qkv, qkv_bias, bias_table, out, B, H, W, C, nh, shift, static_cast<cudaStream_t>(stream));
}
int sb_bbox_embed_sum(int dtype, const long long* boxes, const void* const* tables, void* out, int n, int Hd, int bbox_size,
                      void* stream) {
  return bbox_embed_sum(dtype, boxes, tables, out, n, Hd, bbox_size, static_cast<cudaStream_t>(stream));
}
int sb_attn_single_query(int dtype, const void* q, int ldq, const void* K, const void* V, long long batch_stride,
                         long long head_stride, long long token_stride, void* out, int ldo, int B, int nh, int nkv, int head_dim,
                         int n_keys, float scale, void* stream) {
  return attn_single_query(dtype, q, ldq, K, V, batch_stride, head_stride, token_stride, out, ldo, B, nh, nkv, head_dim, n_keys,
                           scale, static_cast<cudaStream_t>(stream));
}
int sb_label_embed(int dtype, const long long* boxes, const void* const* tables, void* out, int n, int box_w, int prop_w,
                   int bbox_size, int vocab, void* stream) {
  return label_embed(dtype, boxes, tables, out, n, box_w, prop_w, bbox_size, vocab, static_cast<cudaStream_t>(stream));
}
int sb_box_next_token(const float* bbox, const float* const* heads, const int* head_n, const int* head_mode, int n_heads,
                      float bbox_size, long long* out, unsigned char* done, int done_head, int eos, int pad, int B, int* cache_pos,
                      const int* hist_base, int hist_T, long long* hist_tok, float* hist_bbox, float* const* hist_heads,
                      unsigned char* hist_done, void* stream) {
  return box_next_token(bbox, heads, head_n, head_mode, n_heads, bbox_size, out, done, done_head, eos, pad, B, cache_pos,
                        hist_base, hist_T, hist_tok, hist_bbox, hist_heads, hist_done, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
