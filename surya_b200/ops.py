"""Torch-tensor wrappers over the op-level C ABI (include/surya_b200.h).

torch is used for device memory and streams only; every function launches hand-written sm_100a kernels from
libsurya_b200.so on torch's current CUDA stream and raises if the library or a GPU is missing.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import c_float, c_int, c_void_p, check, ptr, stream_ptr

ACT = {"none": 0, "gelu": 1, "gelu_erf": 1, "silu": 2, "hardswish": 3, "relu": 4, "gelu_tanh": 5}


def dt_code(dtype: torch.dtype) -> int:
    if dtype == torch.bfloat16:
        return 0
    if dtype == torch.float16:
        return 1
    raise _lib.SuryaB200Error(f"surya_b200 kernels compute in bf16 or fp16, got {dtype}")


def _rowmajor(t: torch.Tensor) -> int:
    assert t.dim() == 2 and t.stride(1) == 1, "expected a row-major 2-D tensor"
    return t.stride(0)


def gemm(a, w, bias=None, residual=None, act="none", swiglu=False, out=None, out_f32=False, force_bn=0, splitk=False,
         rms_eps=None, rowscale=None, argmax=None, argmax_only=False):
    """out[M, Nout] = epi(a[M,K] @ w[N,K]^T); bias fp32 [N]; see sb_gemm.  splitk=True lets the heuristic use the split-K
    cluster kernel (decode-sized M only).
    rms_eps / rowscale: RMSNorm folded into the GEMM (sb_gemm_rmsnorm): w already carries the norm weight, rows are scaled by
    `rowscale` (fp32 [M]) or by 1/rms computed in the kernel with rms_eps.  argmax: dict filled with the per-tile partials
    (val, idx, sum) of the online argmax epilogue; argmax_only skips writing the logits."""
    if splitk and force_bn == 0:
        force_bn = -1
    lib = _lib.load()
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K
    n_out = N // 2 if swiglu else N
    if out is None:
        out = torch.empty((M, n_out), device=a.device, dtype=torch.float32 if out_f32 else a.dtype)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() >= N
    if rms_eps is not None or rowscale is not None or argmax is not None or argmax_only:
        assert not out_f32
        am = None
        if argmax is not None or argmax_only:
            bn = force_bn if force_bn > 0 else int(lib.sb_gemm_argmax_tile(c_int(M), c_int(N)))
            nt = (N + bn - 1) // bn
            am = (torch.empty((M, nt), device=a.device, dtype=torch.float32), torch.empty((M, nt), device=a.device, dtype=torch.int32),
                  torch.empty((M, nt), device=a.device, dtype=torch.float32))
            if argmax is not None:
                argmax.update(val=am[0], idx=am[1], sum=am[2], tile=bn)
            force_bn = bn
        check(lib.sb_gemm_rmsnorm(dt_code(a.dtype), ptr(a), c_int(_rowmajor(a)), ptr(w), c_int(_rowmajor(w)), ptr(out),
                                  c_int(_rowmajor(out)), c_int(M), c_int(N), c_int(K), ptr(bias), ptr(residual),
                                  c_int(_rowmajor(residual) if residual is not None else 0), c_int(ACT[act]),
                                  c_int(1 if swiglu else 0), ptr(rowscale), c_float(rms_eps if rms_eps is not None else 0.0),
                                  ptr(am[0]) if am else c_void_p(0), ptr(am[1]) if am else c_void_p(0),
                                  ptr(am[2]) if am else c_void_p(0), c_int(am[0].shape[1] if am else 0),
                                  c_int(0 if argmax_only else 1), c_int(max(force_bn, 0)), stream_ptr()), "sb_gemm_rmsnorm")
        return out
    check(lib.sb_gemm(dt_code(a.dtype), ptr(a), c_int(_rowmajor(a)), ptr(w), c_int(_rowmajor(w)), ptr(out),
                      c_int(_rowmajor(out)), c_int(M), c_int(N), c_int(K), ptr(bias), ptr(residual),
                      c_int(_rowmajor(residual) if residual is not None else 0), c_int(ACT[act]),
                      c_int(1 if swiglu else 0), c_int(1 if out_f32 else 0), c_int(force_bn), stream_ptr()), "sb_gemm")
    return out


def row_rstd(x, eps=1e-6, src_rows=None):
    """fp32 [rows]: rsqrt(mean(x^2) + eps) per row, summed in the order the GEMM's in-kernel pass uses."""
    lib = _lib.load()
    rows = x.shape[0] if src_rows is None else src_rows.numel()
    out = torch.empty(rows, device=x.device, dtype=torch.float32)
    check(lib.sb_row_rstd(dt_code(x.dtype), ptr(x), c_int(_rowmajor(x)), ptr(out), c_int(rows), c_int(x.shape[1]), c_float(eps),
                          ptr(src_rows), stream_ptr()), "sb_row_rstd")
    return out


def rmsnorm(x, w, eps=1e-6, src_rows=None, out=None):
    lib = _lib.load()
    rows = x.shape[0] if src_rows is None else src_rows.numel()
    H = x.shape[1]
    if out is None:
        out = torch.empty((rows, H), device=x.device, dtype=x.dtype)
    check(lib.sb_rmsnorm(dt_code(x.dtype), ptr(x), c_int(_rowmajor(x)), ptr(w), ptr(out), c_int(_rowmajor(out)),
                         c_int(rows), c_int(H), c_float(eps), ptr(src_rows), stream_ptr()), "sb_rmsnorm")
    return out


def gather_pad_rows(src, perm, Kp, dtype):
    lib = _lib.load()
    rows = src.shape[0] if perm is None else perm.numel()
    K = src.shape[1]
    out = torch.empty((rows, Kp), device=src.device, dtype=dtype)
    check(lib.sb_gather_pad_rows(dt_code(dtype), ptr(src), c_int(1 if src.dtype == torch.float32 else 0),
                                 c_int(_rowmajor(src)), ptr(perm), ptr(out), c_int(Kp), c_int(rows), c_int(K),
                                 c_int(Kp), stream_ptr()), "sb_gather_pad_rows")
    return out


def rope_vision_(qkv, pos_rc, inv_freq, nh, d):
    lib = _lib.load()
    check(lib.sb_rope_vision(dt_code(qkv.dtype), ptr(qkv), c_int(_rowmajor(qkv)), ptr(pos_rc), ptr(inv_freq),
                             c_int(qkv.shape[0]), c_int(nh), c_int(d), stream_ptr()), "sb_rope_vision")
    return qkv


def rope_kv_append_(qkv, tok_pos, tok_slot, inv_freq, kcache, vcache, nh, nkv, d):
    lib = _lib.load()
    s_max = kcache.shape[2]
    check(lib.sb_rope_kv_append(dt_code(qkv.dtype), ptr(qkv), c_int(_rowmajor(qkv)), ptr(tok_pos), ptr(tok_slot),
                                ptr(inv_freq), ptr(kcache), ptr(vcache), c_int(qkv.shape[0]), c_int(nh), c_int(nkv),
                                c_int(d), c_int(s_max), stream_ptr()), "sb_rope_kv_append")
    return qkv


def attn_varlen(q, k, v, seq_start, seq_len, max_len, n_heads, n_kv_heads, head_dim, causal, scale, out=None):
    """q/k/v are 2-D row-major *views* whose column 0 is head 0 (e.g. qkv[:, 0:H], qkv[:, H:2H], ...)."""
    lib = _lib.load()
    n_tok = q.shape[0]
    if out is None:
        out = torch.empty((n_tok, n_heads * head_dim), device=q.device, dtype=q.dtype)
    check(lib.sb_attn_varlen(dt_code(q.dtype), ptr(q), c_int(q.stride(0)), ptr(k), c_int(k.stride(0)), ptr(v),
                             c_int(v.stride(0)), ptr(out), c_int(out.stride(0)), ptr(seq_start), ptr(seq_len),
                             c_int(seq_start.numel()), c_int(max_len), c_int(n_heads), c_int(n_kv_heads),
                             c_int(head_dim), c_int(1 if causal else 0), c_float(scale), stream_ptr()),
          "sb_attn_varlen")
    return out


def decode_attn(qkv, kcache, vcache, slot, pos, inv_freq, n_heads, n_kv_heads, head_dim, scale, out=None):
    lib = _lib.load()
    B = qkv.shape[0]
    if out is None:
        out = torch.empty((B, n_heads * head_dim), device=qkv.device, dtype=qkv.dtype)
    check(lib.sb_decode_attn(dt_code(qkv.dtype), ptr(qkv), c_int(_rowmajor(qkv)), ptr(kcache), ptr(vcache), ptr(slot),
                             ptr(pos), ptr(inv_freq), ptr(out), c_int(_rowmajor(out)), c_int(B), c_int(n_heads),
                             c_int(n_kv_heads), c_int(head_dim), c_int(kcache.shape[2]), c_float(scale),
                             stream_ptr()), "sb_decode_attn")
    return out


def embed_splice(ids, feat_row, hidx, widx, embed, feat, h_embed, w_embed):
    lib = _lib.load()
    n, H = ids.numel(), embed.shape[1]
    out = torch.empty((n, H), device=embed.device, dtype=embed.dtype)
    check(lib.sb_embed_splice(dt_code(embed.dtype), ptr(ids), ptr(feat_row), ptr(hidx), ptr(widx), ptr(embed),
                              ptr(feat), c_int(_rowmajor(feat) if feat is not None else 0), ptr(h_embed), ptr(w_embed),
                              ptr(out), c_int(H), c_int(n), c_int(H), stream_ptr()), "sb_embed_splice")
    return out


def embed_rows(ids, embed):
    lib = _lib.load()
    n, H = ids.numel(), embed.shape[1]
    out = torch.empty((n, H), device=embed.device, dtype=embed.dtype)
    check(lib.sb_embed_rows(dt_code(embed.dtype), ptr(ids), ptr(embed), ptr(out), c_int(H), c_int(n), c_int(H),
                            stream_ptr()), "sb_embed_rows")
    return out


def rec_stop_rules(tok_hist, done_hist, step, gen_count, ring, row_done, n_valid, n_active, max_tokens, max_repeats=40):
    """One evaluation of the decode loop's stop rules for host step `step` (sb_rec_stop_rules); state tensors update in place."""
    lib = _lib.load()
    B = gen_count.numel()
    assert tok_hist.dtype == torch.int64 and done_hist.dtype == torch.uint8 and tok_hist.shape[1] == B
    assert gen_count.dtype == torch.int32 and ring.dtype == torch.int64 and row_done.dtype == torch.uint8 and n_valid.dtype == torch.int32
    assert ring.shape == (B, max_repeats) and ring.is_contiguous() and tok_hist.is_contiguous() and done_hist.is_contiguous()
    check(lib.sb_rec_stop_rules(ptr(tok_hist), ptr(done_hist), c_int(step), c_int(B), ptr(gen_count), ptr(ring), ptr(row_done),
                                ptr(n_valid), ptr(n_active), c_int(max_tokens), c_int(max_repeats), stream_ptr()), "sb_rec_stop_rules")


def argmax_score(logits, eos, pad):
    lib = _lib.load()
    rows, V = logits.shape
    dev = logits.device
    tok = torch.empty(rows, device=dev, dtype=torch.int64)
    score = torch.empty(rows, device=dev, dtype=torch.float32)
    done = torch.empty(rows, device=dev, dtype=torch.uint8)
    nxt = torch.empty(rows, device=dev, dtype=torch.int64)
    check(lib.sb_argmax_score(dt_code(logits.dtype), ptr(logits), c_int(_rowmajor(logits)), c_int(rows), c_int(V),
                              ptr(tok), ptr(score), ptr(done), ptr(nxt), c_int(eos), c_int(pad), stream_ptr()),
          "sb_argmax_score")
    return tok, score, done, nxt


def small_head(x, w, b, sigmoid=True, box_scale=None):
    lib = _lib.load()
    rows, H = x.shape
    n_out = w.shape[0]
    out_f = torch.empty((rows, n_out), device=x.device, dtype=torch.float32)
    out_box = torch.empty((rows, n_out), device=x.device, dtype=torch.int64) if box_scale is not None else None
    check(lib.sb_small_head(dt_code(x.dtype), ptr(x), c_int(_rowmajor(x)), ptr(w), ptr(b), c_int(rows), c_int(H),
                            c_int(n_out), c_int(1 if sigmoid else 0), ptr(out_f), ptr(out_box),
                            c_float(box_scale if box_scale is not None else 0.0), stream_ptr()), "sb_small_head")
    return out_f, out_box


# ------------------------------------------------------------------------------------------------ detection ops (NHWC)
def conv2d_nhwc(x, w, bias=None, residual=None, ksize=3, stride=1, pad=1, act="none"):
    """x [N,H,W,Cin], w [Cout, k*k*Cin] (K ordered r,s,c), bias fp32 [Cout] -> [N,Ho,Wo,Cout]."""
    lib = _lib.load()
    N, H, W, Cin = x.shape
    Cout = w.shape[0]
    Ho, Wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    out = torch.empty((N, Ho, Wo, Cout), device=x.device, dtype=x.dtype)
    check(lib.sb_conv2d_nhwc(dt_code(x.dtype), ptr(x), ptr(w), ptr(bias), ptr(residual), ptr(out), c_int(N), c_int(H), c_int(W),
                             c_int(Cin), c_int(Cout), c_int(ksize), c_int(stride), c_int(pad), c_int(ACT[act]), stream_ptr()),
          "sb_conv2d_nhwc")
    return out


def dwconv_nhwc(x, w, bias=None, ksize=3, stride=1, pad=1, act="none"):
    """x [N,H,W,C], w [k*k, C]."""
    lib = _lib.load()
    N, H, W, C = x.shape
    Ho, Wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    out = torch.empty((N, Ho, Wo, C), device=x.device, dtype=x.dtype)
    check(lib.sb_dwconv_nhwc(dt_code(x.dtype), ptr(x), ptr(w), ptr(bias), ptr(out), c_int(N), c_int(H), c_int(W), c_int(C),
                             c_int(ksize), c_int(stride), c_int(pad), c_int(ACT[act]), stream_ptr()), "sb_dwconv_nhwc")
    return out


def gemm_grouped(a, w_pad, groups):
    """Block-diagonal 1x1 conv: a [M, C], w_pad [C, 64] (row o of group g holds its C/groups inputs, zero padded)."""
    lib = _lib.load()
    M, C = a.shape
    out = torch.empty((M, C), device=a.device, dtype=a.dtype)
    check(lib.sb_gemm_grouped(dt_code(a.dtype), ptr(a), c_int(a.stride(0)), c_int(C), ptr(w_pad), c_int(64), ptr(out), c_int(C),
                              c_int(M), c_int(C), c_int(64), c_int(C // groups), c_int(C // groups), stream_ptr()),
          "sb_gemm_grouped")
    return out


def lite_mla(qkv_a, qkv_b, B, HW, heads, dim, eps):
    lib = _lib.load()
    out = torch.empty((B * HW, 2 * heads * dim), device=qkv_a.device, dtype=qkv_a.dtype)
    check(lib.sb_lite_mla(dt_code(qkv_a.dtype), ptr(qkv_a), ptr(qkv_b), ptr(out), c_int(B), c_int(HW), c_int(heads), c_int(dim),
                          ctypes.c_float(eps), stream_ptr()), "sb_lite_mla")
    return out


# ------------------------------------------------------------------------------------------------ layout / table_rec ops
def rmsnorm_adetr(x, w, eps=1e-6):
    lib = _lib.load()
    out = torch.empty_like(x)
    check(lib.sb_rmsnorm_adetr(dt_code(x.dtype), ptr(x), c_int(_rowmajor(x)), ptr(w), ptr(out), c_int(_rowmajor(out)),
                               c_int(x.shape[0]), c_int(x.shape[1]), c_float(eps), stream_ptr()), "sb_rmsnorm_adetr")
    return out


def layernorm(x, w, b, eps=1e-5):
    lib = _lib.load()
    x = x.contiguous()
    out = torch.empty_like(x)
    check(lib.sb_layernorm(dt_code(x.dtype), ptr(x), ptr(w), ptr(b), ptr(out), c_int(x.shape[0]), c_int(x.shape[1]),
                           c_float(eps), stream_ptr()), "sb_layernorm")
    return out


def embed_pos_layernorm(ids, pos, word, ptab, w, b, eps=1e-12):
    """LayerNorm(word[ids] + ptab[pos]) over packed int32 token rows (sb_embed_pos_layernorm; ocr_error Embeddings)."""
    lib = _lib.load()
    assert ids.dtype == torch.int32 and pos.dtype == torch.int32 and ids.numel() == pos.numel()
    n, C = ids.numel(), word.shape[1]
    out = torch.empty((n, C), device=word.device, dtype=word.dtype)
    check(lib.sb_embed_pos_layernorm(dt_code(word.dtype), ptr(ids), ptr(pos), ptr(word), ptr(ptab), ptr(w), ptr(b), ptr(out),
                                     c_int(n), c_int(C), c_float(eps), stream_ptr()), "sb_embed_pos_layernorm")
    return out


def patch_gather(pixels, P, Kp, dtype):
    lib = _lib.load()
    B, C, H, W = pixels.shape
    pixels = pixels.contiguous()
    out = torch.empty((B * (-(-H // P)) * (-(-W // P)), Kp), device=pixels.device, dtype=dtype)
    check(lib.sb_patch_gather(dt_code(dtype), ptr(pixels), c_int(1 if pixels.dtype == torch.float32 else 0), ptr(out), c_int(B),
                              c_int(C), c_int(H), c_int(W), c_int(P), c_int(Kp), stream_ptr()), "sb_patch_gather")
    return out


def add_bcast_rows_(x, tab):
    lib = _lib.load()
    check(lib.sb_add_bcast_rows(dt_code(x.dtype), ptr(x), ptr(tab), ctypes.c_longlong(x.shape[0]), c_int(tab.shape[0]),
                                c_int(x.shape[1]), stream_ptr()), "sb_add_bcast_rows")
    return x


def patch_merge_gather(x, B, H, W):
    lib = _lib.load()
    C = x.shape[1]
    out = torch.empty((B * ((H + 1) // 2) * ((W + 1) // 2), 4 * C), device=x.device, dtype=x.dtype)
    check(lib.sb_patch_merge_gather(dt_code(x.dtype), ptr(x), ptr(out), c_int(B), c_int(H), c_int(W), c_int(C), stream_ptr()),
          "sb_patch_merge_gather")
    return out


def swin_window_attn(qkv, bias_table, B, H, W, nh, shift, qkv_bias=None):
    """qkv_bias (fp32 [3C]) is needed when H or W is not a multiple of the 8x8 window: pad tokens are Linear(0) = bias."""
    lib = _lib.load()
    C = qkv.shape[1] // 3
    out = torch.empty((qkv.shape[0], C), device=qkv.device, dtype=qkv.dtype)
    check(lib.sb_swin_window_attn(dt_code(qkv.dtype), ptr(qkv), ptr(qkv_bias) if qkv_bias is not None else None, ptr(bias_table),
                                  ptr(out), c_int(B), c_int(H), c_int(W), c_int(C), c_int(nh), c_int(shift), stream_ptr()),
          "sb_swin_window_attn")
    return out


def bbox_embed_sum(boxes, tables, hidden, bbox_size, dtype):
    """boxes int64 [n, 7]; tables: list of 15 device tensors (w,h,cx,cy,xskew,yskew,x1,y1,x2,y2,x3,y3,x4,y4,label)."""
    lib = _lib.load()
    n = boxes.shape[0]
    out = torch.empty((n, hidden), device=boxes.device, dtype=dtype)
    arr = (_lib.c_void_p * 15)(*[t.data_ptr() for t in tables])
    check(lib.sb_bbox_embed_sum(dt_code(dtype), ptr(boxes.contiguous()), arr, ptr(out), c_int(n), c_int(hidden), c_int(bbox_size),
                                stream_ptr()), "sb_bbox_embed_sum")
    return out


def attn_single_query(q, kv, n_keys, nh, nkv, hd, scale):
    """q [B, nh*hd]; kv [B*n_keys, 2*nkv*hd] = per token (K heads | V heads), i.e. the fused cross K/V projection output."""
    lib = _lib.load()
    B = q.shape[0]
    out = torch.empty_like(q)
    row = 2 * nkv * hd
    esz = kv.element_size()
    kptr = kv.data_ptr()
    vptr = kptr + nkv * hd * esz
    check(lib.sb_attn_single_query(dt_code(q.dtype), ptr(q), c_int(_rowmajor(q)), _lib.c_void_p(kptr), _lib.c_void_p(vptr),
                                   ctypes.c_longlong(n_keys * row), ctypes.c_longlong(hd), ctypes.c_longlong(row), ptr(out),
                                   c_int(_rowmajor(out)), c_int(B), c_int(nh), c_int(nkv), c_int(hd), c_int(n_keys), c_float(scale),
                                   stream_ptr()), "sb_attn_single_query")
    return out


def label_embed(boxes, tables, box_w, prop_w, bbox_size, vocab, dtype):
    """boxes int64 [n, 10]; tables: 13 device tensors (w,h,cx,cy,xskew,yskew,x1,y1,x3,y3 | category,merge,colspan)."""
    lib = _lib.load()
    n = boxes.shape[0]
    out = torch.empty((n, box_w + prop_w), device=boxes.device, dtype=dtype)
    arr = (_lib.c_void_p * 13)(*[t.data_ptr() for t in tables])
    check(lib.sb_label_embed(dt_code(dtype), ptr(boxes.contiguous()), arr, ptr(out), c_int(n), c_int(box_w), c_int(prop_w),
                             c_int(bbox_size), c_int(vocab), stream_ptr()), "sb_label_embed")
    return out


def box_next_token(bbox, heads, modes, bbox_size, done_head=-1, eos=1, pad=0, out=None, done=None, cache_pos=None,
                   hist_base=None, hist=None):
    """bbox fp32 [B,6]; heads: list of fp32 [B,n_k]; modes: 0 argmax / 1 colspan rounding -> tokens int64 [B, 6+len(heads)].
    Loop state (optional): cache_pos int32 [B] is advanced; hist = {"tok": i64 [T,B,ncol], "bbox": f32 [T,B,6],
    "heads": [f32 [T,B,n_k]...], "done": u8 [T,B]} rows are written at cache_pos - hist_base[0]."""
    lib = _lib.load()
    B, k = bbox.shape[0], len(heads)
    if out is None:
        out = torch.empty((B, 6 + k), device=bbox.device, dtype=torch.int64)
    if done is None and done_head >= 0:
        done = torch.empty((B,), device=bbox.device, dtype=torch.uint8)
    hp = (_lib.c_void_p * max(k, 1))(*[h.data_ptr() for h in heads])
    hn = (ctypes.c_int * max(k, 1))(*[h.shape[1] for h in heads])
    hm = (ctypes.c_int * max(k, 1))(*modes)
    for h in heads:
        assert h.dtype == torch.float32 and h.is_contiguous()
    hist = hist or {}
    hh = hist.get("heads")
    hhp = (_lib.c_void_p * max(k, 1))(*[t.data_ptr() for t in hh]) if hh else None
    T = hist["tok"].shape[0] if "tok" in hist else 0
    check(lib.sb_box_next_token(ptr(bbox), hp, hn, hm, c_int(k), c_float(float(bbox_size)), ptr(out), ptr(done), c_int(done_head),
                                c_int(eos), c_int(pad), c_int(B), ptr(cache_pos), ptr(hist_base), c_int(T), ptr(hist.get("tok")),
                                ptr(hist.get("bbox")), hhp, ptr(hist.get("done")), stream_ptr()), "sb_box_next_token")
    return out, done
