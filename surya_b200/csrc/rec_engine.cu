// surya_b200 — recognition engine: vision tower + decoder prefill + decode steps as one C++ object.
//
// Stands in for SuryaModel.forward (surya/common/surya/__init__.py:274-338) under RecognitionPredictor.prefill /
// decode (surya/recognition/__init__.py:326-352, 354-471).  The layer loops live here (not in Python) so that a
// decode step is 62 back-to-back kernel launches on one stream (5 per decoder layer + lm_head + tail), capturable into a
// CUDA graph and replayed with token feedback / position increment / history done on the device (sb_rec_decode_steps).
#include "../../include/surya_b200.h"
#include "ops.cuh"
#include "sb_ptx.cuh"

#include <cstring>
#include <string>
#include <vector>

using namespace sb;

#define CK(x)                    \
  do {                           \
    int rc_ = (x);               \
    if (rc_) return rc_;         \
  } while (0)

struct sb_rec_engine {
  sb_rec_config c;
  std::vector<const void*> w;
  size_t esz = 2;
  // workspaces (device)
  uint8_t* arena = nullptr;
  size_t arena_bytes = 0;
  void *x = nullptr, *nbuf = nullptr, *qkv = nullptr, *ao = nullptr, *act = nullptr, *x0 = nullptr, *m1 = nullptr,
       *feat = nullptr, *xl = nullptr, *logits = nullptr;
  void* kcache = nullptr;  // [layer][slot][kvh][s_max][d]
  void* vcache = nullptr;
  // staging for the device-side decode loop
  long long* st_tok = nullptr; float* st_score = nullptr; long long* st_bbox = nullptr; unsigned char* st_done = nullptr;
  long long* st_next = nullptr; int* st_step = nullptr; unsigned int* st_counter = nullptr;
  // folded RMSNorm: per-row 1/rms of the residual stream (prefill; decode steps compute it inside the GEMM)
  float* rs = nullptr;
  // lm_head argmax partials [rows, am_ld]: (max, argmax, sum exp) per 128 x am_bn logit tile
  float* am_val = nullptr; int* am_idx = nullptr; float* am_sum = nullptr;
  int am_ld = 0, am_bn = 0;
  int qkv_w_enc = 0, qkv_w_dec = 0;
  // CUDA graph cache for decode_steps
  cudaGraphExec_t graph_exec = nullptr;
  int graph_batch = 0;
  long long graph_nodes = 0;
  // the legacy default stream cannot be captured: decode_steps hops onto an engine-owned stream, ordered by events
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  const void* graph_key[8] = {nullptr};
  // device-side stop rules (sb_rec_set_sched): caller-owned per-row state, evaluated by stop_rules_kernel after every loop step
  int* sc_gen = nullptr; long long* sc_ring = nullptr; unsigned char* sc_done = nullptr; int* sc_valid = nullptr; int* sc_active = nullptr;
  int sc_max_tokens = 0, sc_max_repeats = 0;

  const void* W(int idx) const { return w[idx]; }
  const void* WE(int layer, int k) const { return w[SB_RW_ENC_BASE + layer * SB_RWE_STRIDE + k]; }
  const void* WD(int layer, int k) const {
    return w[SB_RW_ENC_BASE + c.enc_depth * SB_RWE_STRIDE + layer * SB_RWD_STRIDE + k];
  }
  void* kc(int layer) const {
    return static_cast<uint8_t*>(kcache) + static_cast<size_t>(layer) * c.max_slots * c.dec_kv_heads * c.s_max * c.dec_head_dim * esz;
  }
  void* vc(int layer) const {
    return static_cast<uint8_t*>(vcache) + static_cast<size_t>(layer) * c.max_slots * c.dec_kv_heads * c.s_max * c.dec_head_dim * esz;
  }
};

static size_t al256(size_t v) { return (v + 255) & ~size_t(255); }

// norm: 0 = plain, 1 = folded RMSNorm with the per-row scale in e->rs (prefill), 2 = folded RMSNorm with the scale computed
// inside the GEMM from the A tiles (decode steps, lm_head)
static int linear(const sb_rec_engine* e, const void* A, int lda, const void* Wt, int ldw, void* C, int ldc, int M, int N,
                  int K, const void* bias_f32, const void* residual, int ldr, int act, int swiglu, cudaStream_t st,
                  int allow_splitk = 0, int norm = 0) {
  GemmArgs a;
  if (norm == 1) a.rowscale = e->rs;
  if (norm == 2) { a.ssq_inline = 1; a.ssq_eps = e->c.rms_eps; a.ssq_k = K; }
  a.dtype = e->c.dtype;
  a.A = A; a.lda = lda; a.W = Wt; a.ldw = ldw; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K;
  a.bias = static_cast<const float*>(bias_f32);
  a.residual = residual; a.ldr = ldr; a.act = act; a.swiglu = swiglu;
  a.w_constant = 1;   // engine weights are never written after packing
  a.allow_splitk = allow_splitk;
  return gemm_launch(a, st);
}

// ------------------------------------------------------------------------------------------------ vision tower
static int run_vision(sb_rec_engine* e, const void* tiles, int tiles_f32, int n, const int* perm, const int* pos_rc,
                      const int* win_start, const int* win_len, int n_win, int max_win, const int* img_start,
                      const int* img_len, int n_img, int max_img, cudaStream_t st) {
  const sb_rec_config& c = e->c;
  const int H = c.enc_hidden, nh = c.enc_heads, hd = H / nh;
  const int dt = c.dtype;
  CK(gather_pad_rows(dt, tiles, tiles_f32, c.patch_dim, perm, e->x0, c.patch_dim_pad, n, c.patch_dim, c.patch_dim_pad, st));
  CK(linear(e, e->x0, c.patch_dim_pad, e->W(SB_RW_PATCH_W), c.patch_dim_pad, e->x, H, n, H, c.patch_dim_pad, nullptr,
            nullptr, 0, ACT_NONE, 0, st));
  const int ldq = 3 * H;
  uint8_t* qkv8 = static_cast<uint8_t*>(e->qkv);
  for (int l = 0; l < c.enc_depth; ++l) {
    CK(rmsnorm(dt, e->x, H, e->WE(l, SB_RWE_NORM1), e->nbuf, H, n, H, 1e-6f, nullptr, st));
    CK(linear(e, e->nbuf, H, e->WE(l, SB_RWE_QKV_W), H, e->qkv, ldq, n, 3 * H, H, e->WE(l, SB_RWE_QKV_B), nullptr, 0,
              ACT_NONE, 0, st));
    CK(rope_vision(dt, e->qkv, ldq, pos_rc, static_cast<const float*>(e->W(SB_RW_ENC_INV_FREQ)), n, nh, hd, st));
    AttnArgs a;
    a.dtype = dt;
    a.q = qkv8; a.ldq = ldq;
    a.k = qkv8 + static_cast<size_t>(H) * e->esz; a.ldk = ldq;
    a.v = qkv8 + static_cast<size_t>(2 * H) * e->esz; a.ldv = ldq;
    a.out = e->ao; a.ldo = H;
    const bool full = (c.fullatt_mask >> l) & 1u;
    a.seq_start = full ? img_start : win_start;
    a.seq_len = full ? img_len : win_len;
    a.n_seq = full ? n_img : n_win;
    a.max_len = full ? max_img : max_win;
    a.n_heads = nh; a.n_kv_heads = nh; a.head_dim = hd; a.causal = 0;
    a.scale = 1.0f / sqrtf(static_cast<float>(hd));
    CK(attn_varlen(a, st));
    CK(linear(e, e->ao, H, e->WE(l, SB_RWE_PROJ_W), H, e->x, H, n, H, H, e->WE(l, SB_RWE_PROJ_B), e->x, H, ACT_NONE, 0, st));
    CK(rmsnorm(dt, e->x, H, e->WE(l, SB_RWE_NORM2), e->nbuf, H, n, H, 1e-6f, nullptr, st));
    CK(linear(e, e->nbuf, H, e->WE(l, SB_RWE_GU_W), H, e->act, c.enc_inter_pad, n, 2 * c.enc_inter_pad, H,
              e->WE(l, SB_RWE_GU_B), nullptr, 0, ACT_SILU, 1, st));
    CK(linear(e, e->act, c.enc_inter_pad, e->WE(l, SB_RWE_DOWN_W), c.enc_inter_pad, e->x, H, n, H, c.enc_inter_pad,
              e->WE(l, SB_RWE_DOWN_B), e->x, H, ACT_NONE, 0, st));
  }
  // merger: RMSNorm -> view [n/unit, unit*H] -> Linear+GELU -> Linear
  const int mu = c.merge_unit, MH = mu * H, nm = n / mu;
  CK(rmsnorm(dt, e->x, H, e->W(SB_RW_MERGER_LN), e->nbuf, H, n, H, 1e-6f, nullptr, st));
  CK(linear(e, e->nbuf, MH, e->W(SB_RW_MERGER_W0), MH, e->m1, MH, nm, MH, MH, e->W(SB_RW_MERGER_B0), nullptr, 0,
            ACT_GELU_ERF, 0, st));
  CK(linear(e, e->m1, MH, e->W(SB_RW_MERGER_W2), MH, e->feat, c.enc_out_hidden, nm, c.enc_out_hidden, MH,
            e->W(SB_RW_MERGER_B2), nullptr, 0, ACT_NONE, 0, st));
  return 0;
}

// ------------------------------------------------------------------------------------------------ decoder pieces
// Every decoder RMSNorm is folded into the GEMM that consumes it (W' = W * g packed by the host, the GEMM epilogue scales each
// row by 1/rms): the normalised activations never exist in memory and decode steps lose 25 launches.
struct HeadOut {
  void* logits = nullptr;
  long long* tok = nullptr; float* score = nullptr; long long* bbox = nullptr; float* bbox_sig = nullptr;
  unsigned char* done = nullptr; long long* next_ids = nullptr;
  // device-side greedy loop (sb_rec_decode_steps)
  int loop = 0;
  long long* tok_hist = nullptr; float* score_hist = nullptr; long long* bbox_hist = nullptr; unsigned char* done_hist = nullptr;
  long long* ids_io = nullptr; int* pos_io = nullptr;
};

// lm_head (tied embedding x final norm weight, online argmax epilogue) + decode_tail; `hidden` = residual stream rows BEFORE
// the final norm.  The [rows, vocab] logits are only written when the caller asks for them.
static int run_heads(sb_rec_engine* e, void* hidden, int rows, const HeadOut& o, cudaStream_t st) {
  const sb_rec_config& c = e->c;
  const int D = c.dec_hidden;
  GemmArgs a;
  a.dtype = c.dtype;
  a.A = hidden; a.lda = D; a.W = e->W(SB_RW_LM_W); a.ldw = D;
  a.C = o.logits ? o.logits : e->logits; a.ldc = c.vocab;
  a.M = rows; a.N = c.vocab; a.K = D;
  a.bias = static_cast<const float*>(e->W(SB_RW_LM_BIAS));
  a.w_constant = 1;
  // 1/rms of the final norm: separate pass + rowscale rather than the in-kernel sum of squares — this GEMM runs several tiles
  // per CTA, and the in-kernel pass would serialise each tile's main loop behind the previous tile's epilogue (lm_head
  // 63 vs 48 us, profiles/r02_decode_parts.md)
  CK(row_rstd(c.dtype, hidden, D, e->rs, rows, D, c.rms_eps, nullptr, st));
  a.rowscale = e->rs;
  a.am_val = e->am_val; a.am_idx = e->am_idx; a.am_sum = e->am_sum; a.am_ld = e->am_ld;
  a.store_c = o.logits ? 1 : 0;
  CK(gemm_launch(a, st));
  DecodeTailArgs t;
  t.rows = rows;
  t.am_val = e->am_val; t.am_idx = e->am_idx; t.am_sum = e->am_sum; t.am_ld = e->am_ld;
  t.n_tiles = (c.vocab + e->am_bn - 1) / e->am_bn;
  t.x = hidden; t.ldx = D; t.H = D; t.eps = c.rms_eps;
  t.bbox_w = e->W(SB_RW_BBOX_W); t.bbox_b = e->W(SB_RW_BBOX_B); t.n_box = 6; t.bbox_size = c.bbox_size;
  t.tok = o.tok; t.score = o.score; t.bbox = o.bbox; t.bbox_sig = o.bbox_sig; t.done = o.done; t.next_ids = o.next_ids;
  t.eos = c.eos_id; t.pad = c.pad_id;
  if (o.loop) {
    t.embed = e->W(SB_RW_EMBED); t.x_next = hidden; t.ldx_next = D;
    t.step = e->st_step; t.counter = e->st_counter;
    t.tok_hist = o.tok_hist; t.score_hist = o.score_hist; t.bbox_hist = o.bbox_hist; t.done_hist = o.done_hist;
    t.ids_io = o.ids_io; t.pos_io = o.pos_io;
    if (!t.bbox && o.bbox_hist) t.bbox = e->st_bbox;   // the tail computes boxes when any box output is requested
  }
  CK(decode_tail(c.dtype, t, st));
  if (o.loop && e->sc_gen) {
    if (!o.tok_hist || !o.done_hist) { set_error("device-side stop rules need the token and done histories"); return -9; }
    CK(stop_rules(o.tok_hist, o.done_hist, e->st_step, 0, rows, e->sc_gen, e->sc_ring, e->sc_done, e->sc_valid, e->sc_active,
                  e->sc_max_tokens, e->sc_max_repeats, st));
  }
  return 0;
}

static int run_decoder_prefill(sb_rec_engine* e, const long long* ids, int n_tok, const int* feat_row, const int* hidx,
                               const int* widx, const int* tok_pos, const int* tok_slot, const int* seq_start,
                               const int* seq_len, int n_seq, int max_len, const int* last_tok, const HeadOut& out,
                               cudaStream_t st) {
  const sb_rec_config& c = e->c;
  const int D = c.dec_hidden, nh = c.dec_heads, nkv = c.dec_kv_heads, hd = c.dec_head_dim;
  const int Q = (nh + 2 * nkv) * hd;
  const int dt = c.dtype;
  CK(embed_splice(dt, ids, feat_row, hidx, widx, e->W(SB_RW_EMBED), e->feat, c.enc_out_hidden, e->W(SB_RW_H_EMBED),
                  e->W(SB_RW_W_EMBED), e->x, D, n_tok, D, st));
  uint8_t* qkv8 = static_cast<uint8_t*>(e->qkv);
  for (int l = 0; l < c.dec_layers; ++l) {
    CK(row_rstd(dt, e->x, D, e->rs, n_tok, D, c.rms_eps, nullptr, st));
    CK(linear(e, e->x, D, e->WD(l, SB_RWD_QKV_W), D, e->qkv, Q, n_tok, Q, D, e->WD(l, SB_RWD_QKV_B), nullptr, 0, ACT_NONE, 0,
              st, 0, /*norm=*/1));
    CK(rope_kv_append(dt, e->qkv, Q, tok_pos, tok_slot, static_cast<const float*>(e->W(SB_RW_DEC_INV_FREQ)), e->kc(l),
                      e->vc(l), n_tok, nh, nkv, hd, c.s_max, st));
    AttnArgs a;
    a.dtype = dt;
    a.q = qkv8; a.ldq = Q;
    a.k = qkv8 + static_cast<size_t>(nh * hd) * e->esz; a.ldk = Q;
    a.v = qkv8 + static_cast<size_t>((nh + nkv) * hd) * e->esz; a.ldv = Q;
    a.out = e->ao; a.ldo = nh * hd;
    a.seq_start = seq_start; a.seq_len = seq_len; a.n_seq = n_seq; a.max_len = max_len;
    a.n_heads = nh; a.n_kv_heads = nkv; a.head_dim = hd; a.causal = 1;
    a.scale = 1.0f / sqrtf(static_cast<float>(hd));
    CK(attn_varlen(a, st));
    CK(linear(e, e->ao, nh * hd, e->WD(l, SB_RWD_O_W), nh * hd, e->x, D, n_tok, D, nh * hd, nullptr, e->x, D, ACT_NONE, 0, st));
    CK(row_rstd(dt, e->x, D, e->rs, n_tok, D, c.rms_eps, nullptr, st));
    CK(linear(e, e->x, D, e->WD(l, SB_RWD_GU_W), D, e->act, c.dec_inter_pad, n_tok, 2 * c.dec_inter_pad, D, nullptr, nullptr, 0,
              ACT_SILU, 1, st, 0, /*norm=*/1));
    CK(linear(e, e->act, c.dec_inter_pad, e->WD(l, SB_RWD_DOWN_W), c.dec_inter_pad, e->x, D, n_tok, D, c.dec_inter_pad,
              nullptr, e->x, D, ACT_NONE, 0, st));
  }
  // hidden[:, -1:, :] (surya/common/surya/__init__.py:323): the last real token of every sequence, still un-normalised
  CK(gather_pad_rows(dt, e->x, 0, D, last_tok, e->xl, D, n_seq, D, D, st));
  return run_heads(e, e->xl, n_seq, out, st);
}

// One greedy decode step for `B` rows: 5 launches per layer (qkv GEMM -> attention -> o GEMM -> gate/up GEMM -> down GEMM)
// + lm_head + tail.  ids == nullptr means e->x already holds the input embeddings (written by the previous step's tail).
static int run_decode_step(sb_rec_engine* e, const long long* ids, const int* slot, const int* pos, int B, const HeadOut& out,
                           cudaStream_t st) {
  const sb_rec_config& c = e->c;
  const int D = c.dec_hidden, nh = c.dec_heads, nkv = c.dec_kv_heads, hd = c.dec_head_dim;
  const int Q = (nh + 2 * nkv) * hd;
  const int dt = c.dtype;
  void* x = e->x;
  if (ids) CK(embed_rows(dt, ids, e->W(SB_RW_EMBED), x, D, B, D, st));
  for (int l = 0; l < c.dec_layers; ++l) {
    CK(linear(e, x, D, e->WD(l, SB_RWD_QKV_W), D, e->qkv, Q, B, Q, D, e->WD(l, SB_RWD_QKV_B), nullptr, 0, ACT_NONE, 0, st, 0,
              /*norm=*/2));
    DecodeAttnArgs a;
    a.dtype = dt; a.qkv = e->qkv; a.ld = Q; a.kcache = e->kc(l); a.vcache = e->vc(l); a.slot = slot; a.pos = pos;
    a.inv_freq = static_cast<const float*>(e->W(SB_RW_DEC_INV_FREQ));
    a.out = e->ao; a.ldo = nh * hd; a.batch = B; a.n_heads = nh; a.n_kv_heads = nkv; a.head_dim = hd; a.s_max = c.s_max;
    a.scale = 1.0f / sqrtf(static_cast<float>(hd));
    CK(decode_attn(a, st));
    CK(linear(e, e->ao, nh * hd, e->WD(l, SB_RWD_O_W), nh * hd, x, D, B, D, nh * hd, nullptr, x, D, ACT_NONE, 0, st));
    CK(linear(e, x, D, e->WD(l, SB_RWD_GU_W), D, e->act, c.dec_inter_pad, B, 2 * c.dec_inter_pad, D, nullptr, nullptr, 0,
              ACT_SILU, 1, st, 0, /*norm=*/2));
    CK(linear(e, e->act, c.dec_inter_pad, e->WD(l, SB_RWD_DOWN_W), c.dec_inter_pad, x, D, B, D, c.dec_inter_pad, nullptr, x, D,
              ACT_NONE, 0, st, /*allow_splitk=*/1));
  }
  return run_heads(e, x, B, out, st);
}

extern "C" {

int sb_rec_create(const sb_rec_config* cfg, const void* const* weights, int n_weights, sb_rec_engine** out) {
  if (!cfg || !weights || !out) { set_error("sb_rec_create: null argument"); return -1; }
  const int need = SB_RW_ENC_BASE + cfg->enc_depth * SB_RWE_STRIDE + cfg->dec_layers * SB_RWD_STRIDE;
  if (n_weights != need) { set_error("sb_rec_create: expected %d weight pointers, got %d", need, n_weights); return -2; }
  if (cfg->dec_hidden != cfg->enc_out_hidden) { set_error("decoder hidden must equal encoder out_hidden"); return -3; }
  if (cfg->patch_dim_pad % 8 || cfg->enc_inter_pad % 8 || cfg->dec_inter_pad % 8 || cfg->enc_hidden % 8 ||
      cfg->dec_hidden % 8 || cfg->vocab % 8) {
    set_error("sb_rec_create: padded dims and vocab must be multiples of 8 (16-byte TMA pitch rule)");
    return -4;
  }
  for (int i = 0; i < n_weights; ++i)
    if (!weights[i]) { set_error("sb_rec_create: weight pointer %d is null", i); return -5; }
  auto* e = new sb_rec_engine();
  e->c = *cfg;
  e->w.assign(weights, weights + n_weights);
  const sb_rec_config& c = e->c;
  const size_t es = e->esz;
  const size_t R = static_cast<size_t>(c.max_patches > c.max_tokens ? c.max_patches : c.max_tokens);
  const size_t Hm = c.enc_hidden > c.dec_hidden ? c.enc_hidden : c.dec_hidden;
  const int Q = (c.dec_heads + 2 * c.dec_kv_heads) * c.dec_head_dim;
  const size_t qkvw = (size_t)(3 * c.enc_hidden > Q ? 3 * c.enc_hidden : Q);
  const size_t aow = (size_t)(c.enc_hidden > c.dec_heads * c.dec_head_dim ? c.enc_hidden : c.dec_heads * c.dec_head_dim);
  const size_t actw = (size_t)(c.enc_inter_pad > c.dec_inter_pad ? c.enc_inter_pad : c.dec_inter_pad);
  const size_t nm = (size_t)c.max_patches / c.merge_unit + 1;
  const size_t kv_bytes = (size_t)c.dec_layers * c.max_slots * c.dec_kv_heads * c.s_max * c.dec_head_dim * es;
  const size_t rows_out = (size_t)(c.max_seqs > c.max_slots ? c.max_seqs : c.max_slots);
  e->am_bn = gemm_argmax_tile(static_cast<int>(rows_out), c.vocab);
  e->am_ld = (c.vocab + e->am_bn - 1) / e->am_bn;
  const size_t am_elems = rows_out * static_cast<size_t>(e->am_ld);
  size_t sizes[] = {
      R * Hm * es, R * Hm * es, R * qkvw * es, R * aow * es, R * actw * es,           // x nbuf qkv ao act
      (size_t)c.max_patches * c.patch_dim_pad * es, nm * c.merge_unit * c.enc_hidden * es,  // x0 m1
      nm * c.enc_out_hidden * es, rows_out * c.dec_hidden * es, rows_out * c.vocab * es,   // feat xl logits
      kv_bytes, kv_bytes,
      rows_out * 8, rows_out * 4, rows_out * 6 * 8, rows_out, rows_out * 8, 256, 256,
      R * 4, am_elems * 4, am_elems * 4, am_elems * 4};
  size_t total = 0;
  for (size_t s : sizes) total += al256(s);
  cudaError_t ce = cudaMalloc(&e->arena, total);
  if (ce != cudaSuccess) {
    set_error("sb_rec_create: cudaMalloc(%zu MiB) failed: %s", total >> 20, cudaGetErrorString(ce));
    delete e;
    return -6;
  }
  e->arena_bytes = total;
  uint8_t* p = e->arena;
  void** slots[] = {&e->x, &e->nbuf, &e->qkv, &e->ao, &e->act, &e->x0, &e->m1, &e->feat, &e->xl, &e->logits,
                    &e->kcache, &e->vcache, (void**)&e->st_tok, (void**)&e->st_score, (void**)&e->st_bbox,
                    (void**)&e->st_done, (void**)&e->st_next, (void**)&e->st_step, (void**)&e->st_counter,
                    (void**)&e->rs, (void**)&e->am_val, (void**)&e->am_idx, (void**)&e->am_sum};
  for (size_t i = 0; i < sizeof(sizes) / sizeof(sizes[0]); ++i) {
    *slots[i] = p;
    p += al256(sizes[i]);
  }
  cudaMemset(e->arena, 0, total);
  *out = e;
  return 0;
}

void sb_rec_destroy(sb_rec_engine* e) {
  if (!e) return;
  if (e->graph_exec) cudaGraphExecDestroy(e->graph_exec);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  if (e->arena) cudaFree(e->arena);
  delete e;
}

size_t sb_rec_workspace_bytes(const sb_rec_engine* e) { return e ? e->arena_bytes : 0; }

int sb_rec_prefill(sb_rec_engine* e, const void* tiles, int tiles_f32, int n_patches, const int* patch_perm,
                   const int* patch_pos_rc, const int* win_start, const int* win_len, int n_win, int max_win_len,
                   const int* img_start, const int* img_len, int n_img, int max_img_len, const long long* input_ids,
                   int n_tok, const int* tok_feat_row, const int* tok_hidx, const int* tok_widx, const int* tok_pos,
                   const int* tok_slot, const int* seq_start, const int* seq_len, int n_seq, int max_seq_len,
                   const int* last_tok, void* logits, long long* tok, float* score, long long* bbox, float* bbox_sig,
                   unsigned char* done, long long* next_ids, void* stream) {
  if (!e) { set_error("sb_rec_prefill: null engine"); return -1; }
  const sb_rec_config& c = e->c;
  if (n_patches > c.max_patches || n_tok > c.max_tokens || n_seq > c.max_seqs) {
    set_error("sb_rec_prefill: batch exceeds engine capacity (patches %d/%d tokens %d/%d seqs %d/%d)", n_patches,
              c.max_patches, n_tok, c.max_tokens, n_seq, c.max_seqs);
    return -2;
  }
  if (n_patches % c.merge_unit) { set_error("sb_rec_prefill: patch count must be a multiple of the merge unit"); return -3; }
  if (max_seq_len > c.s_max) { set_error("sb_rec_prefill: sequence longer than s_max"); return -4; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_patches > 0)
    CK(run_vision(e, tiles, tiles_f32, n_patches, patch_perm, patch_pos_rc, win_start, win_len, n_win, max_win_len,
                  img_start, img_len, n_img, max_img_len, st));
  HeadOut o;
  o.logits = logits; o.tok = tok; o.score = score; o.bbox = bbox; o.bbox_sig = bbox_sig; o.done = done; o.next_ids = next_ids;
  return run_decoder_prefill(e, input_ids, n_tok, tok_feat_row, tok_hidx, tok_widx, tok_pos, tok_slot, seq_start,
                             seq_len, n_seq, max_seq_len, last_tok, o, st);
}

int sb_rec_decode(sb_rec_engine* e, const long long* input_ids, const int* slot, const int* pos, int batch, void* logits,
                  long long* tok, float* score, long long* bbox, float* bbox_sig, unsigned char* done,
                  long long* next_ids, void* stream) {
  if (!e) { set_error("sb_rec_decode: null engine"); return -1; }
  if (batch > e->c.max_slots || batch > e->c.max_tokens) { set_error("sb_rec_decode: batch %d exceeds capacity", batch); return -2; }
  if (!input_ids) { set_error("sb_rec_decode: null input_ids"); return -3; }
  HeadOut o;
  o.logits = logits; o.tok = tok; o.score = score; o.bbox = bbox; o.bbox_sig = bbox_sig; o.done = done; o.next_ids = next_ids;
  return run_decode_step(e, input_ids, slot, pos, batch, o, static_cast<cudaStream_t>(stream));
}

int sb_rec_decode_steps(sb_rec_engine* e, long long* ids_io, const int* slot, int* pos_io, int batch, int n_steps,
                        long long* tok_hist, float* score_hist, long long* bbox_hist, unsigned char* done_hist,
                        int use_graph, void* stream) {
  if (!e) { set_error("sb_rec_decode_steps: null engine"); return -1; }
  if (batch > e->c.max_slots || batch > e->c.max_tokens) { set_error("sb_rec_decode_steps: batch exceeds capacity"); return -2; }
  cudaStream_t caller = static_cast<cudaStream_t>(stream);
  cudaStream_t st = caller;
  const bool hop = use_graph && (caller == nullptr || caller == cudaStreamLegacy || caller == cudaStreamPerThread);
  if (hop) {
    if (!e->own_stream) {
      if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming) != cudaSuccess ||
          cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        set_error("sb_rec_decode_steps: could not create the engine stream");
        return -8;
      }
    }
    cudaEventRecord(e->ev_in, caller);
    cudaStreamWaitEvent(e->own_stream, e->ev_in, 0);
    st = e->own_stream;
  }
  struct Rejoin {  // whatever happens below, order the caller's stream after the engine stream
    bool on; cudaStream_t own, caller; cudaEvent_t ev;
    ~Rejoin() { if (on) { cudaEventRecord(ev, own); cudaStreamWaitEvent(caller, ev, 0); } }
  } rejoin{hop, e->own_stream, caller, e->ev_out};
  if (cudaMemsetAsync(e->st_step, 0, sizeof(int), st) != cudaSuccess ||
      cudaMemsetAsync(e->st_counter, 0, sizeof(unsigned int), st) != cudaSuccess) { cudaGetLastError(); set_error("memset failed"); return -3; }
  if (e->sc_valid && cudaMemsetAsync(e->sc_valid, 0, sizeof(int) * batch, st) != cudaSuccess) { cudaGetLastError(); set_error("memset failed"); return -3; }
  // the first step's input embeddings; every later step finds them written by the previous step's tail kernel
  CK(embed_rows(e->c.dtype, ids_io, e->W(SB_RW_EMBED), e->x, e->c.dec_hidden, batch, e->c.dec_hidden, st));
  HeadOut ho;
  ho.loop = 1;
  ho.tok_hist = tok_hist; ho.score_hist = score_hist; ho.bbox_hist = bbox_hist; ho.done_hist = done_hist;
  ho.ids_io = ids_io; ho.pos_io = pos_io;
  auto one_step = [&](cudaStream_t s) -> int { return run_decode_step(e, nullptr, slot, pos_io, batch, ho, s); };
  if (!use_graph) {
    for (int i = 0; i < n_steps; ++i) CK(one_step(st));
    return 0;
  }
  const void* key[8] = {ids_io, slot, pos_io, tok_hist, score_hist, bbox_hist, done_hist, nullptr};
  bool hit = e->graph_exec && e->graph_batch == batch && std::memcmp(key, e->graph_key, sizeof(key)) == 0;
  if (!hit) {
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
    // one eager step first: sets kernel attributes (not capturable) and validates the launch parameters
    CK(one_step(st));
    n_steps -= 1;
    if (n_steps <= 0) return 0;
    cudaGraph_t graph = nullptr;
    cudaError_t cb = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
    if (cb != cudaSuccess) { cudaGetLastError(); set_error("graph capture begin failed: %s", cudaGetErrorString(cb)); return -4; }
    const long long before = launch_count();
    int rc = one_step(st);
    e->graph_nodes = launch_count() - before;
    count_launches(-e->graph_nodes);  // captured, not executed
    cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc || ce != cudaSuccess) { cudaGetLastError(); set_error("graph capture failed: rc=%d %s", rc, cudaGetErrorString(ce)); return -5; }
    ce = cudaGraphInstantiate(&e->graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { cudaGetLastError(); set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); e->graph_exec = nullptr; return -6; }
    e->graph_batch = batch;
    std::memcpy(e->graph_key, key, sizeof(key));
  }
  for (int i = 0; i < n_steps; ++i) {
    if (cudaGraphLaunch(e->graph_exec, st) != cudaSuccess) { cudaGetLastError(); set_error("cudaGraphLaunch failed"); return -7; }
    count_launches(e->graph_nodes);
  }
  return 0;
}

int sb_rec_set_sched(sb_rec_engine* e, int* gen_count, long long* ring, unsigned char* row_done, int* n_valid, int* n_active,
                     int max_tokens, int max_repeats) {
  if (!e) { set_error("sb_rec_set_sched: null engine"); return -1; }
  if (gen_count && (!ring || !row_done || !n_valid || max_tokens <= 0 || max_repeats < 2 || max_repeats > 64)) {
    set_error("sb_rec_set_sched: incomplete state (ring / row_done / n_valid) or max_tokens %d / max_repeats %d out of range", max_tokens,
              max_repeats);
    return -2;
  }
  const bool same = e->sc_gen == gen_count && e->sc_ring == ring && e->sc_done == row_done && e->sc_valid == n_valid &&
                    e->sc_active == n_active && e->sc_max_tokens == max_tokens && e->sc_max_repeats == max_repeats;
  if (!same && e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }   // the captured step changes
  e->sc_gen = gen_count; e->sc_ring = gen_count ? ring : nullptr; e->sc_done = gen_count ? row_done : nullptr;
  e->sc_valid = gen_count ? n_valid : nullptr; e->sc_active = gen_count ? n_active : nullptr;
  e->sc_max_tokens = gen_count ? max_tokens : 0; e->sc_max_repeats = gen_count ? max_repeats : 0;
  return 0;
}

int sb_rec_debug_copy(sb_rec_engine* e, const char* name, void* dst, size_t bytes, void* stream) {
  if (!e || !name || !dst) { set_error("sb_rec_debug_copy: null argument"); return -1; }
  std::string n(name);
  const void* src = nullptr;
  if (n == "feat") src = e->feat;
  else if (n == "x") src = e->x;
  else if (n == "xl") src = e->xl;
  else if (n == "logits") src = e->logits;
  else if (n == "qkv") src = e->qkv;
  else if (n == "kcache") src = e->kcache;
  else if (n == "vcache") src = e->vcache;
  if (!src) { set_error("sb_rec_debug_copy: unknown workspace '%s'", name); return -2; }
  cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream));
  if (ce != cudaSuccess) { set_error("sb_rec_debug_copy: %s", cudaGetErrorString(ce)); return -3; }
  return 0;
}

}  // extern "C"
