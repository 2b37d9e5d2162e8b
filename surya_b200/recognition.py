"""Recognition path: host-side mirror of the reference's model / predictor surface over the CUDA engine.

  * pack_rec_weights      state_dict (reference names) -> kernel-friendly device tensors (SB_RW_* order)
  * plan_vision / plan_tokens   integer index plans (window permutation, RoPE ids, ragged token layout)
  * RecEngine             ctypes wrapper of sb_rec_* (include/surya_b200.h)
  * B200SuryaModel        quacks like `RecognitionPredictor.model` (surya/recognition/__init__.py:332-339,
                          398-409): __call__(input_ids, image_tiles, grid_thw, attention_mask, position_ids,
                          past_key_values=SlotCache, ...) -> {"lm_logits", "bbox_logits"}
  * SlotCache             quacks like ContinuousBatchingCache (surya/recognition/cache.py:7-105): merge / trim_left
  * RecognitionRunner     mirror of RecognitionPredictor.prediction_loop (:501-607) on engine slots

Host code is Python/NumPy/torch plumbing only; every tensor op on the forward path is a kernel from
libsurya_b200.so.  Nothing here imports oracle/ and nothing falls back to PyTorch math.
"""
from __future__ import annotations

import ctypes
import math
from collections import deque
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import c_int, c_void_p, check, ptr, stream_ptr
from .config import RecConfig, align
from .ops import dt_code


# ------------------------------------------------------------------------------------------------ C structs
class _RecCfgC(ctypes.Structure):
    _fields_ = [
        ("dtype", c_int),
        ("enc_depth", c_int), ("enc_hidden", c_int), ("enc_heads", c_int), ("enc_inter", c_int), ("enc_inter_pad", c_int),
        ("patch_dim", c_int), ("patch_dim_pad", c_int), ("merge_unit", c_int), ("enc_out_hidden", c_int),
        ("fullatt_mask", ctypes.c_uint),
        ("dec_layers", c_int), ("dec_hidden", c_int), ("dec_heads", c_int), ("dec_kv_heads", c_int),
        ("dec_head_dim", c_int), ("dec_inter", c_int), ("dec_inter_pad", c_int),
        ("rms_eps", ctypes.c_float),
        ("vocab", c_int), ("eos_id", c_int), ("pad_id", c_int),
        ("bbox_size", ctypes.c_float),
        ("max_slots", c_int), ("s_max", c_int), ("max_patches", c_int), ("max_tokens", c_int), ("max_seqs", c_int),
    ]


# ------------------------------------------------------------------------------------------------ weight packing
def _interleave_rows(gate: torch.Tensor, up: torch.Tensor, rows_pad: int) -> torch.Tensor:
    """[I, K] x2 -> [2*rows_pad, K] with rows (gate_0, up_0, gate_1, up_1, ...), zero padded."""
    I, K = gate.shape
    out = torch.zeros((rows_pad, 2, K), dtype=gate.dtype)
    out[:I, 0] = gate
    out[:I, 1] = up
    return out.reshape(2 * rows_pad, K)


def _pad_cols(w: torch.Tensor, cols: int) -> torch.Tensor:
    if w.shape[1] == cols:
        return w
    out = torch.zeros((w.shape[0], cols), dtype=w.dtype)
    out[:, : w.shape[1]] = w
    return out


def pack_rec_weights(sd: Dict[str, torch.Tensor], cfg: RecConfig, dtype: torch.dtype, device) -> List[torch.Tensor]:
    """Pack a reference-named fp32 state dict into the SB_RW_* table (see include/surya_b200.h).

    16-bit tensors are rounded once from fp32 (= model.to(dtype)); Linear biases are kept as the fp32 image of
    the rounded 16-bit bias so the GEMM epilogue adds exactly the value the reference adds."""
    e, d = cfg.vision_encoder, cfg.decoder

    def T(x):
        return x.to(dtype).contiguous().to(device)

    def B32(x):  # bias: round to model dtype, keep fp32 container
        return x.to(dtype).float().contiguous().to(device)

    def F32(x):
        return x.float().contiguous().to(device)

    def FOLD(w, g):
        """Linear weight with the preceding RMSNorm weight folded in: W'[n, k] = W[n, k] * g[k], formed from the 16-bit images
        of both (what `model.to(dtype)` holds) in fp32 and rounded once.  The reference computes W @ (g * T(x * rstd))
        (decoder/__init__.py:241-258); the engine computes rstd * (W' @ x) with rstd applied to the fp32 accumulator in the GEMM
        epilogue — same algebra, one rounding moved from the activations to the weights."""
        return (w.to(dtype).float() * g.to(dtype).float()[None, :]).to(dtype).contiguous().to(device)

    ip_e, ip_d = align(e.intermediate_size, 8), align(d.intermediate_size, 8)
    pdp = align(e.patch_dim, 8)
    hd_e, hd_d = e.head_dim, d.head_dim
    p = "vision_encoder."
    g_final = sd["decoder.norm.weight"]
    fixed = [
        T(_pad_cols(sd[p + "patch_embed.proj.weight"].reshape(e.hidden_size, -1), pdp)),
        T(sd[p + "merger.ln_q.weight"]),
        T(sd[p + "merger.mlp.0.weight"]), B32(sd[p + "merger.mlp.0.bias"]),
        T(sd[p + "merger.mlp.2.weight"]), B32(sd[p + "merger.mlp.2.bias"]),
        F32(1.0 / (10000.0 ** (torch.arange(0, hd_e // 2, 2, dtype=torch.float) / (hd_e // 2)))),
        FOLD(sd["embedder.token_embed.weight"], g_final),       # lm_head is tied to the embedding (surya/common/surya/__init__.py:111-116)
        T(sd["embedder.token_embed.weight"]),
        B32(sd["lm_head.bias"]),
        FOLD(sd["bbox_head.weight"], g_final), T(sd["bbox_head.bias"]),
        T(sd["img_h_embed.weight"]), T(sd["img_w_embed.weight"]),
        F32(1.0 / (d.rope_theta ** (torch.arange(0, hd_d, 2, dtype=torch.int64).float() / hd_d))),
    ]
    enc = []
    for i in range(e.depth):
        b = f"{p}blocks.{i}."

        def pad_bias(g, u):
            out = torch.zeros((ip_e, 2), dtype=torch.float32)
            out[: e.intermediate_size, 0] = g
            out[: e.intermediate_size, 1] = u
            return out.reshape(-1)

        enc += [
            T(sd[b + "norm1.weight"]),
            T(sd[b + "attn.qkv.weight"]), B32(sd[b + "attn.qkv.bias"]),
            T(sd[b + "attn.proj.weight"]), B32(sd[b + "attn.proj.bias"]),
            T(sd[b + "norm2.weight"]),
            T(_interleave_rows(sd[b + "mlp.gate_proj.weight"], sd[b + "mlp.up_proj.weight"], ip_e)),
            B32(pad_bias(sd[b + "mlp.gate_proj.bias"], sd[b + "mlp.up_proj.bias"])),
            T(_pad_cols(sd[b + "mlp.down_proj.weight"], ip_e)), B32(sd[b + "mlp.down_proj.bias"]),
        ]
    dec = []
    for i in range(d.num_hidden_layers):
        b = f"decoder.layers.{i}."
        qkv_w = torch.cat([sd[b + "self_attn.q_proj.weight"], sd[b + "self_attn.k_proj.weight"],
                           sd[b + "self_attn.v_proj.weight"]], 0)
        qkv_b = torch.cat([sd[b + "self_attn.q_proj.bias"], sd[b + "self_attn.k_proj.bias"],
                           sd[b + "self_attn.v_proj.bias"]], 0)
        dec += [
            FOLD(qkv_w, sd[b + "input_layernorm.weight"]), B32(qkv_b),
            T(sd[b + "self_attn.o_proj.weight"]),
            FOLD(_interleave_rows(sd[b + "mlp.gate_proj.weight"], sd[b + "mlp.up_proj.weight"], ip_d),
                 sd[b + "post_attention_layernorm.weight"]),
            T(_pad_cols(sd[b + "mlp.down_proj.weight"], ip_d)),
        ]
    return fixed + enc + dec


# ------------------------------------------------------------------------------------------------ index plans
_GRID_CACHE: Dict[Tuple[int, int, int, int, int], dict] = {}


def _grid_plan(h: int, w: int, merge: int, window: int, patch: int) -> dict:
    """Per-image integer plan for a (1, h, w) patch grid — mirrors rot_pos_emb / get_window_index
    (surya/common/surya/encoder/__init__.py:523-597) and get_2d_learned_embeddings' index math
    (surya/common/surya/__init__.py:240-259).  All arrays are local to the image (offset by the caller)."""
    key = (h, w, merge, window, patch)
    hit = _GRID_CACHE.get(key)
    if hit is not None:
        return hit
    unit = merge * merge
    lh, lw = h // merge, w // merge
    # (row, col) of every patch in merge-block-major order
    hp = np.arange(h)[:, None].repeat(w, 1).reshape(lh, merge, lw, merge).transpose(0, 2, 1, 3).reshape(-1)
    wp = np.arange(w)[None, :].repeat(h, 0).reshape(lh, merge, lw, merge).transpose(0, 2, 1, 3).reshape(-1)
    pos = np.stack([hp, wp], -1).astype(np.int32)
    # window order of merged units
    vws = window // merge // patch
    index = np.arange(lh * lw).reshape(lh, lw)
    pad_h, pad_w = vws - lh % vws, vws - lw % vws
    nwh, nww = (lh + pad_h) // vws, (lw + pad_w) // vws
    padded = np.pad(index, ((0, pad_h), (0, pad_w)), constant_values=-100)
    padded = padded.reshape(nwh, vws, nww, vws).transpose(0, 2, 1, 3).reshape(nwh * nww, vws * vws)
    seqlens = (padded != -100).sum(1)
    flat = padded.reshape(-1)
    widx = flat[flat != -100].astype(np.int64)            # window position -> original merged unit
    win_len = (seqlens[seqlens > 0] * unit).astype(np.int32)
    win_start = (np.concatenate([[0], np.cumsum(win_len)[:-1]])).astype(np.int32)
    patch_perm = (widx[:, None] * unit + np.arange(unit)[None, :]).reshape(-1).astype(np.int32)
    inv = np.argsort(widx).astype(np.int32)                # original merged unit -> window position
    # learned 2-D embedding rows (fp32 arithmetic then truncation, as torch does)
    mult = np.float32(256)

    def emb_idx(n):
        v = np.arange(n, dtype=np.float32) / np.float32(max(1, n - 1)) * mult
        return v.astype(np.int64).astype(np.int32)

    hi = np.repeat(emb_idx(lh), lw)
    wi = np.tile(emb_idx(lw), lh)
    plan = dict(n_patches=h * w, n_units=lh * lw, patch_perm=patch_perm, pos_perm=pos[patch_perm],
                win_start=win_start, win_len=win_len, inv=inv, hidx=hi, widx=wi)
    _GRID_CACHE[key] = plan
    return plan


@dataclass
class PrefillPlan:
    ints: torch.Tensor            # pinned int32 buffer with every array below back to back
    off: Dict[str, Tuple[int, int]]
    ids: torch.Tensor             # pinned int64 [n_tok]
    n_patches: int
    n_win: int
    max_win: int
    n_img: int
    max_img: int
    n_tok: int
    n_seq: int
    max_seq: int


def build_prefill_plan(cfg: RecConfig, grid_thw: np.ndarray, seq_tokens: Sequence[np.ndarray],
                       slots: Sequence[int], image_multiplier: Optional[int] = None) -> PrefillPlan:
    """grid_thw [n_img, 3]; seq_tokens = per-sequence REAL token ids (no padding); slots = KV slot per sequence."""
    e = cfg.vision_encoder
    merge, unit = e.spatial_merge_size, e.spatial_merge_size ** 2
    mult = image_multiplier or cfg.image_embed_encoding_multiplier
    assert mult == 256, "index math assumes image_embed_encoding_multiplier == 256"
    parts = {k: [] for k in ("patch_perm", "pos_perm", "win_start", "win_len", "img_start", "img_len", "inv", "hidx", "widx")}
    p_off = u_off = 0
    for t, h, w in np.asarray(grid_thw).reshape(-1, 3):
        assert t == 1, "temporal grids are not used by surya (temporal_patch_size = 1)"
        g = _grid_plan(int(h), int(w), merge, e.window_size, e.patch_size)
        parts["patch_perm"].append(g["patch_perm"] + p_off)
        parts["pos_perm"].append(g["pos_perm"])
        parts["win_start"].append(g["win_start"] + p_off)
        parts["win_len"].append(g["win_len"])
        parts["img_start"].append(np.array([p_off], np.int32))
        parts["img_len"].append(np.array([g["n_patches"]], np.int32))
        parts["inv"].append(g["inv"] + u_off)
        parts["hidx"].append(g["hidx"])
        parts["widx"].append(g["widx"])
        p_off += g["n_patches"]
        u_off += g["n_units"]
    cat = {k: (np.concatenate(v).astype(np.int32) if v else np.zeros(0, np.int32)) for k, v in parts.items()}
    ids = np.concatenate([np.asarray(s, dtype=np.int64) for s in seq_tokens])
    lens = np.array([len(s) for s in seq_tokens], dtype=np.int32)
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32)
    tok_pos = np.concatenate([np.arange(n, dtype=np.int32) for n in lens])
    tok_slot = np.repeat(np.asarray(slots, dtype=np.int32), lens)
    is_img = ids == cfg.image_token_id
    n_img_tok = int(is_img.sum())
    assert n_img_tok == u_off, f"image tokens ({n_img_tok}) and image features ({u_off}) do not match"
    feat_row = np.full(ids.shape, -1, np.int32)
    hi = np.zeros(ids.shape, np.int32)
    wi = np.zeros(ids.shape, np.int32)
    feat_row[is_img] = cat["inv"]
    hi[is_img] = cat["hidx"]
    wi[is_img] = cat["widx"]
    arrays = {
        "patch_perm": cat["patch_perm"], "pos_rc": cat["pos_perm"].reshape(-1), "win_start": cat["win_start"],
        "win_len": cat["win_len"], "img_start": cat["img_start"], "img_len": cat["img_len"], "feat_row": feat_row,
        "hidx": hi, "widx": wi, "tok_pos": tok_pos, "tok_slot": tok_slot, "seq_start": starts, "seq_len": lens,
        "last_tok": (starts + lens - 1).astype(np.int32),
    }
    total = sum(a.size for a in arrays.values())
    buf = torch.empty(max(total, 1), dtype=torch.int32).pin_memory() if torch.cuda.is_available() else torch.empty(max(total, 1), dtype=torch.int32)
    off, o = {}, 0
    nb = buf.numpy()
    for k, a in arrays.items():
        nb[o:o + a.size] = a
        off[k] = (o, a.size)
        o += a.size
    ids_t = torch.from_numpy(ids)
    if torch.cuda.is_available():
        ids_t = ids_t.pin_memory()
    return PrefillPlan(ints=buf, off=off, ids=ids_t, n_patches=p_off, n_win=cat["win_len"].size,
                       max_win=int(cat["win_len"].max()) if cat["win_len"].size else 0, n_img=cat["img_len"].size,
                       max_img=int(cat["img_len"].max()) if cat["img_len"].size else 0, n_tok=ids.size,
                       n_seq=lens.size, max_seq=int(lens.max()))


# ------------------------------------------------------------------------------------------------ engine wrapper
class RecEngine:
    """Owns one sb_rec_engine (weights + KV slots + workspaces) on the current CUDA device."""

    def __init__(self, cfg: RecConfig, state_dict: Dict[str, torch.Tensor], dtype: torch.dtype = torch.bfloat16,
                 device: str | torch.device = "cuda", max_slots: int = 257, s_max: Optional[int] = None,
                 max_patches: int = 65536, max_tokens: int = 32768, max_seqs: Optional[int] = None,
                 packed_weights: Optional[List[torch.Tensor]] = None):
        self.lib = _lib.load()
        self.cfg, self.dtype, self.device = cfg, dtype, torch.device(device)
        e, d = cfg.vision_encoder, cfg.decoder
        self.weights = packed_weights if packed_weights is not None else pack_rec_weights(state_dict, cfg, dtype, self.device)
        self.s_max = s_max or cfg.max_sequence_length
        self.max_slots = max_slots
        self.max_patches, self.max_tokens = max_patches, max_tokens
        mask = 0
        for i in e.fullatt_block_indexes:
            mask |= 1 << i
        c = _RecCfgC(
            dtype=dt_code(dtype), enc_depth=e.depth, enc_hidden=e.hidden_size, enc_heads=e.num_heads,
            enc_inter=e.intermediate_size, enc_inter_pad=align(e.intermediate_size, 8), patch_dim=e.patch_dim,
            patch_dim_pad=align(e.patch_dim, 8), merge_unit=e.spatial_merge_size ** 2, enc_out_hidden=e.out_hidden_size,
            fullatt_mask=mask, dec_layers=d.num_hidden_layers, dec_hidden=d.hidden_size, dec_heads=d.num_attention_heads,
            dec_kv_heads=d.num_key_value_heads, dec_head_dim=d.head_dim, dec_inter=d.intermediate_size,
            dec_inter_pad=align(d.intermediate_size, 8), rms_eps=d.rms_norm_eps, vocab=cfg.vocab_size,
            eos_id=cfg.eos_token_id, pad_id=cfg.pad_token_id, bbox_size=float(cfg.bbox_size), max_slots=max_slots,
            s_max=self.s_max, max_patches=max_patches, max_tokens=max_tokens, max_seqs=max_seqs or max_slots)
        self._c = c
        arr = (c_void_p * len(self.weights))(*[w.data_ptr() for w in self.weights])
        self._h = c_void_p()
        self.lib.sb_rec_workspace_bytes.restype = ctypes.c_size_t
        with torch.cuda.device(self.device):
            check(self.lib.sb_rec_create(ctypes.byref(c), arr, c_int(len(self.weights)), ctypes.byref(self._h)),
                  "sb_rec_create")
        self.free_slots = deque(range(max_slots))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.sb_rec_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def workspace_bytes(self) -> int:
        return int(self.lib.sb_rec_workspace_bytes(self._h))

    # ---- slots
    def alloc_slots(self, n: int) -> List[int]:
        if n > len(self.free_slots):
            raise _lib.SuryaB200Error(f"out of KV slots: need {n}, free {len(self.free_slots)}")
        return [self.free_slots.popleft() for _ in range(n)]

    def release_slots(self, slots: Sequence[int]):
        self.free_slots.extend(int(s) for s in slots)

    # ---- calls
    def prefill(self, tiles: torch.Tensor, plan: PrefillPlan, want_logits: bool = False):
        """tiles: device or pinned-host [n_patches, patch_dim] (fp32 or engine dtype). Returns dict of device tensors."""
        dev = self.device
        if not tiles.is_cuda:
            tiles = tiles.to(dev, non_blocking=True)
        ints = plan.ints.to(dev, non_blocking=True)
        ids = plan.ids.to(dev, non_blocking=True)

        def ip(name):
            o, n = plan.off[name]
            return c_void_p(ints.data_ptr() + 4 * o) if n else c_void_p(0)

        n = plan.n_seq
        out = {
            "tok": torch.empty(n, dtype=torch.int64, device=dev), "score": torch.empty(n, dtype=torch.float32, device=dev),
            "bbox": torch.empty((n, 6), dtype=torch.int64, device=dev),
            "bbox_sig": torch.empty((n, 6), dtype=torch.float32, device=dev),
            "done": torch.empty(n, dtype=torch.uint8, device=dev), "next_ids": torch.empty(n, dtype=torch.int64, device=dev),
        }
        if want_logits:
            out["logits"] = torch.empty((n, self.cfg.vocab_size), dtype=self.dtype, device=dev)
        tiles_f32 = 1 if tiles.dtype == torch.float32 else 0
        if not tiles_f32 and tiles.dtype != self.dtype:
            raise _lib.SuryaB200Error(f"tiles must be float32 or {self.dtype}")
        check(self.lib.sb_rec_prefill(
            self._h, ptr(tiles), c_int(tiles_f32), c_int(plan.n_patches), ip("patch_perm"), ip("pos_rc"),
            ip("win_start"), ip("win_len"), c_int(plan.n_win), c_int(plan.max_win), ip("img_start"), ip("img_len"),
            c_int(plan.n_img), c_int(plan.max_img), ptr(ids), c_int(plan.n_tok), ip("feat_row"), ip("hidx"), ip("widx"),
            ip("tok_pos"), ip("tok_slot"), ip("seq_start"), ip("seq_len"), c_int(plan.n_seq), c_int(plan.max_seq),
            ip("last_tok"), ptr(out.get("logits")), ptr(out["tok"]), ptr(out["score"]), ptr(out["bbox"]),
            ptr(out["bbox_sig"]), ptr(out["done"]), ptr(out["next_ids"]), stream_ptr()), "sb_rec_prefill")
        out["_keep"] = (tiles, ints, ids)
        return out

    def decode(self, input_ids: torch.Tensor, slot: torch.Tensor, pos: torch.Tensor, want_logits: bool = False,
               max_pos: Optional[int] = None):
        dev = self.device
        B = input_ids.numel()
        if max_pos is None:
            max_pos = int(pos.max().item()) if B else 0
        if max_pos >= self.s_max:
            raise _lib.SuryaB200Error(f"decode at position {max_pos} but the engine was built with s_max={self.s_max}")
        out = {
            "tok": torch.empty(B, dtype=torch.int64, device=dev), "score": torch.empty(B, dtype=torch.float32, device=dev),
            "bbox": torch.empty((B, 6), dtype=torch.int64, device=dev),
            "bbox_sig": torch.empty((B, 6), dtype=torch.float32, device=dev),
            "done": torch.empty(B, dtype=torch.uint8, device=dev), "next_ids": torch.empty(B, dtype=torch.int64, device=dev),
        }
        if want_logits:
            out["logits"] = torch.empty((B, self.cfg.vocab_size), dtype=self.dtype, device=dev)
        check(self.lib.sb_rec_decode(self._h, ptr(input_ids), ptr(slot), ptr(pos), c_int(B), ptr(out.get("logits")),
                                     ptr(out["tok"]), ptr(out["score"]), ptr(out["bbox"]), ptr(out["bbox_sig"]),
                                     ptr(out["done"]), ptr(out["next_ids"]), stream_ptr()), "sb_rec_decode")
        return out

    def decode_steps(self, ids_io: torch.Tensor, slot: torch.Tensor, pos_io: torch.Tensor, n_steps: int,
                     hist: Optional[dict] = None, use_graph: bool = True, max_pos: Optional[int] = None):
        """n_steps greedy steps on the device; ids_io / pos_io advance in place. Returns step-major histories.
        max_pos: the largest value in pos_io as known by the host (callers that built pos_io on the host pass it for free);
        the last step writes cache row max_pos + n_steps - 1, which must exist."""
        dev = self.device
        B = ids_io.numel()
        if max_pos is None:
            max_pos = int(pos_io.max().item()) if B else 0
        if max_pos + n_steps > self.s_max:
            raise _lib.SuryaB200Error(
                f"decode would write KV row {max_pos + n_steps - 1} but the engine was built with s_max={self.s_max} "
                "(prompt length + max_tokens must not exceed s_max)")
        if hist is None:
            hist = {
                "tok": torch.empty((n_steps, B), dtype=torch.int64, device=dev),
                "score": torch.empty((n_steps, B), dtype=torch.float32, device=dev),
                "bbox": torch.empty((n_steps, B, 6), dtype=torch.int64, device=dev),
                "done": torch.empty((n_steps, B), dtype=torch.uint8, device=dev),
            }
        check(self.lib.sb_rec_decode_steps(self._h, ptr(ids_io), ptr(slot), ptr(pos_io), c_int(B), c_int(n_steps),
                                           ptr(hist["tok"]), ptr(hist["score"]), ptr(hist["bbox"]), ptr(hist["done"]),
                                           c_int(1 if use_graph else 0), stream_ptr()), "sb_rec_decode_steps")
        return hist

    def set_sched(self, state: Optional[dict], max_tokens: int = 0, max_repeats: int = 40):
        """Device-side stop rules for decode_steps (sb_rec_set_sched, SURVEY §8 f3).  state: dict of device tensors
        gen (int32 [B]), ring (int64 [B, max_repeats]), done (uint8 [B]), valid (int32 [B]), active (int32 [1]); None = off."""
        if state is None:
            check(self.lib.sb_rec_set_sched(self._h, c_void_p(0), c_void_p(0), c_void_p(0), c_void_p(0), c_void_p(0), c_int(0), c_int(0)),
                  "sb_rec_set_sched")
            return
        assert state["gen"].dtype == torch.int32 and state["ring"].dtype == torch.int64 and state["done"].dtype == torch.uint8
        assert state["valid"].dtype == torch.int32 and state["active"].dtype == torch.int32
        assert state["ring"].shape == (state["gen"].numel(), max_repeats) and state["ring"].is_contiguous()
        check(self.lib.sb_rec_set_sched(self._h, ptr(state["gen"]), ptr(state["ring"]), ptr(state["done"]), ptr(state["valid"]),
                                        ptr(state["active"]), c_int(max_tokens), c_int(max_repeats)), "sb_rec_set_sched")

    def debug_tensor(self, name: str, rows: int, cols: int) -> torch.Tensor:
        """Copy of an engine workspace (parity taps): feat / x / xl / logits / qkv."""
        out = torch.empty((rows, cols), dtype=self.dtype, device=self.device)
        check(self.lib.sb_rec_debug_copy(self._h, name.encode(), ptr(out),
                                         ctypes.c_size_t(rows * cols * out.element_size()), stream_ptr()),
              "sb_rec_debug_copy")
        return out


# ------------------------------------------------------------------------------------------------ model / cache mirrors
class SlotCache:
    """ContinuousBatchingCache stand-in (surya/recognition/cache.py:7-105).  The KV data lives in engine slots (no left
    padding is ever materialised), so merge() re-points batch rows at the new sequences' slots and trim_left() moves no
    data.  What the predictor's own bookkeeping relies on is kept exact: the padded sequence length (`get_seq_length`,
    advanced by every model call like DynamicCache.update does), the offset merge() returns (cache.py:70-77, consumed by
    surya/recognition/__init__.py:447-457 to left-pad the attention masks) and truthiness (:424).

    Constructible without arguments because RecognitionPredictor.prefill builds its cache itself with
    `ContinuousBatchingCache()` (:391-395): surya_b200.dropin.install() points that module-level name at this class
    and B200SuryaModel binds the engine on first use."""

    def __init__(self, engine: Optional[RecEngine] = None):
        self.engine = engine
        self.slots: Optional[torch.Tensor] = None  # int32 [B] on device
        self._host: List[int] = []
        self._seen_tokens = 0

    def bind(self, engine: RecEngine) -> "SlotCache":
        if self.engine is not None and self.engine is not engine:
            raise _lib.SuryaB200Error("SlotCache is already bound to another engine")
        self.engine = engine
        return self

    def __bool__(self):
        return self.slots is not None

    def __len__(self):   # DynamicCache.__len__ = number of layers holding data (cache.py:64-66 compares the two)
        return 0 if self.slots is None or self.engine is None else self.engine.cfg.decoder.num_hidden_layers

    def get_seq_length(self, layer_idx: int = 0) -> int:
        return self._seen_tokens

    @property
    def batch_size(self) -> int:
        return len(self._host)

    def assign(self, slots: Sequence[int], seq_len: int = 0):
        self._host = [int(s) for s in slots]
        self.slots = torch.tensor(self._host, dtype=torch.int32, device=self.engine.device)
        self._seen_tokens = int(seq_len)

    def advance(self, n: int = 1):
        self._seen_tokens += n

    def merge(self, new_cache: "SlotCache", merge_idxs: Sequence[int], device=None) -> int:
        """cache.py:57-105 — rows merge_idxs now hold the new sequences (their previous slots are recycled); returns
        current_seq_length - new_seq_length exactly like the reference, whose caller pads the masks with it."""
        if not isinstance(new_cache, SlotCache):
            raise _lib.SuryaB200Error("SlotCache.merge needs a SlotCache (call surya_b200.dropin.install() before prefill)")
        merge_idxs = [int(i) for i in merge_idxs]
        if len(merge_idxs) != len(new_cache._host):
            raise _lib.SuryaB200Error(f"merge of {len(new_cache._host)} sequences into {len(merge_idxs)} rows")
        offset = self._seen_tokens - new_cache._seen_tokens
        if offset < 0:                       # the resident cache is the shorter one: it is (notionally) left-padded
            self._seen_tokens += -offset
        old = [self._host[i] for i in merge_idxs]
        for i, s in zip(merge_idxs, new_cache._host):
            self._host[i] = s
        self.engine.release_slots(old)
        self.slots = torch.tensor(self._host, dtype=torch.int32, device=self.engine.device)
        new_cache.slots, new_cache._host = None, []
        return offset

    def trim_left(self, n):
        """cache.py:39-46 — only the notional padded length changes; left padding is never materialised."""
        self._seen_tokens -= int(n)

    def release(self):
        if self._host and self.engine is not None:
            self.engine.release_slots(self._host)
        self._host, self.slots = [], None

    def __del__(self):
        # RecognitionPredictor.prediction_loop drops its cache with `del self.kv_cache` (surya/recognition/__init__.py:603-605)
        # and never calls a release hook: the slots go back to the engine when the cache object dies.
        try:
            self.release()
        except Exception:
            pass


class _Cfg:
    def __init__(self, cfg: RecConfig):
        self.__dict__.update(cfg.to_dict())
        self.bbox_size = cfg.bbox_size


class B200SuryaModel:
    """Call-compatible with the attributes RecognitionPredictor touches on `self.model`
    (surya/recognition/__init__.py:112, 296-297, 315, 332-339, 398-409): __call__, .config.bbox_size, .device, .dtype.
    `engine` is a RecEngine (or any object with its prefill / decode / alloc_slots / release_slots surface)."""

    def __init__(self, engine: RecEngine):
        self.engine = engine
        self.config = _Cfg(engine.cfg)
        self.device = engine.device
        self.dtype = engine.dtype

    def to(self, *a, **k):
        return self

    def eval(self):
        return self

    def new_cache(self) -> SlotCache:
        return SlotCache(self.engine)

    def __call__(self, input_ids=None, image_tiles=None, grid_thw=None, inputs_embeds=None, attention_mask=None,
                 position_ids=None, past_key_values: Optional[SlotCache] = None, use_cache=True, logits_to_keep=1,
                 encoder_chunk_size=None, **kwargs):
        if inputs_embeds is not None:
            raise NotImplementedError("inputs_embeds is not part of the predictor call surface")
        if not isinstance(past_key_values, SlotCache):
            raise _lib.SuryaB200Error(
                "B200SuryaModel needs a SlotCache as past_key_values: call surya_b200.dropin.install() once so that "
                "RecognitionPredictor.prefill's `ContinuousBatchingCache()` builds one (or pass model.new_cache())")
        cache = past_key_values.bind(self.engine)
        eng, cfg = self.engine, self.engine.cfg
        B, S = input_ids.shape
        if S > 1 or image_tiles is not None:      # ---- prefill
            if cache:
                raise _lib.SuryaB200Error("prefill into a non-empty cache: the predictor prefills a fresh cache and merges it")
            ids_h = input_ids.detach().cpu().numpy()
            m_h = attention_mask.detach().cpu().numpy().astype(bool)
            seqs = [ids_h[b][m_h[b]] for b in range(B)]
            slots = eng.alloc_slots(B)
            try:
                g = grid_thw.detach().cpu().numpy() if grid_thw is not None else np.zeros((0, 3), np.int64)
                plan = build_prefill_plan(cfg, g, seqs, slots)
                tiles = image_tiles if image_tiles is not None else \
                    torch.empty((0, cfg.vision_encoder.patch_dim), dtype=self.dtype, device=self.device)
                out = eng.prefill(tiles, plan, want_logits=True)
            except Exception:
                eng.release_slots(slots)
                raise
            cache.assign(slots, seq_len=S)
        else:                                     # ---- decode
            if not cache or cache.batch_size != B:
                raise _lib.SuryaB200Error(f"decode of {B} rows on a cache holding {cache.batch_size}")
            ids = input_ids.reshape(-1).to(torch.int64).contiguous()
            # rows the predictor has already retired keep decoding (it steps the whole batch, :326-352) and their positions
            # keep growing until a merge replaces them: pin such rows to the last cache row instead of running off the slot.
            # Live rows never get there as long as s_max >= prompt + max_tokens (RecEngine's default: max_sequence_length).
            pos = position_ids.reshape(-1).to(torch.int32).clamp_(max=eng.s_max - 1).contiguous()
            out = eng.decode(ids, cache.slots, pos, want_logits=True, max_pos=0)
            cache.advance(1)
        return {
            "lm_logits": out["logits"].unsqueeze(1),
            "bbox_logits": out["bbox_sig"].to(self.dtype).unsqueeze(1),
            "past_key_values": cache,
        }


# ------------------------------------------------------------------------------------------------ host processor mirror
IMAGE_MEAN = np.array((0.485, 0.456, 0.406), dtype=np.float32)
IMAGE_STD = np.array((0.229, 0.224, 0.225), dtype=np.float32)


def scale_to_fit(img: np.ndarray, max_size=(1024, 256), min_size=(168, 168)) -> np.ndarray:
    """Mirror of SuryaOCRProcessor.scale_to_fit (surya/common/surya/processor/__init__.py:140-178)."""
    import cv2

    h, w = img.shape[:2]
    if w == 0 or h == 0:
        return img
    cur, mx, mn = w * h, max_size[0] * max_size[1], min_size[0] * min_size[1]
    if cur > mx:
        s = (mx / cur) ** 0.5
        nw, nh = math.floor(w * s), math.floor(h * s)
    elif cur < mn:
        s = (mn / cur) ** 0.5
        nw, nh = math.ceil(w * s), math.ceil(h * s)
    else:
        return img
    return cv2.resize(img, (nw, nh), interpolation=cv2.INTER_LANCZOS4)


def tile_image(image: np.ndarray, patch: int = 14, merge: int = 2) -> Tuple[np.ndarray, Tuple[int, int, int]]:
    """Mirror of _process_and_tile (processor/__init__.py:185-230): resize to x28, normalise, merge-block-major tiles."""
    import cv2

    factor = patch * merge
    h, w = image.shape[:2]
    hb, wb = math.ceil(h / factor) * factor, math.ceil(w / factor) * factor
    if hb != h or wb != w:
        image = cv2.resize(image, (wb, hb), interpolation=cv2.INTER_CUBIC)
    image = image.astype(np.float64) * (1 / 255.0)
    image = (image.astype(np.float32) - IMAGE_MEAN) / IMAGE_STD
    h, w = image.shape[:2]
    gh, gw = h // patch, w // patch
    x = image.transpose(2, 0, 1).reshape(3, gh // merge, merge, patch, gw // merge, merge, patch)
    x = x.transpose(1, 4, 2, 5, 0, 3, 6)          # [gh/m, gw/m, m, m, C, P, P]
    return np.ascontiguousarray(x).reshape(gh * gw, 3 * patch * patch), (1, gh, gw)


def fit_size(h: int, w: int, max_size=(1024, 256), min_size=(168, 168)) -> Tuple[int, int]:
    """(h, w) after SuryaOCRProcessor.scale_to_fit (processor/__init__.py:148-174) — the reference's own float arithmetic."""
    cur, mx, mn = w * h, max_size[0] * max_size[1], min_size[0] * min_size[1]
    if cur > mx:
        s = (mx / cur) ** 0.5
        return math.floor(h * s), math.floor(w * s)
    if cur < mn:
        s = (mn / cur) ** 0.5
        return math.ceil(h * s), math.ceil(w * s)
    return h, w


PP_DESC = 9     # int32 words per crop in sb_rec_preprocess's descriptor table


def build_preprocess_plan(crops: Sequence[np.ndarray], cfg: RecConfig, max_size=(1024, 256), staging=None) -> dict:
    """Host plan of the device preprocessing path (sb_rec_preprocess, SURVEY §8 f2): uint8 HWC crops packed back to back (16-byte
    aligned), one descriptor per crop {byte offset, h, w, size after scale_to_fit, size rounded up to patch*merge, scratch offset,
    first tile row} and the tile grids — only sizes are computed here, with the reference's arithmetic; every pixel is touched on
    the device.  staging(nbytes) may hand out the (pinned) uint8 buffer the crops are packed into."""
    P, m = cfg.vision_encoder.patch_size, cfg.merge_size
    factor = P * m
    desc = np.zeros((len(crops), PP_DESC), dtype=np.int32)
    grids, off, scratch, row = [], 0, 0, 0
    for i, c in enumerate(crops):
        c = np.asarray(c)
        if c.ndim != 3 or c.shape[2] != 3 or c.shape[0] == 0 or c.shape[1] == 0:
            raise _lib.SuryaB200Error(f"crop {i}: expected a non-empty [h, w, 3] image, got shape {c.shape}")
        if c.dtype != np.uint8:
            raise _lib.SuryaB200Error(f"crop {i}: the device preprocessing path takes uint8 pixels (page slices), got {c.dtype}")
        h, w = c.shape[:2]
        nh, nw = fit_size(h, w, max_size)
        hb, wb = math.ceil(nh / factor) * factor, math.ceil(nw / factor) * factor
        desc[i] = (off, h, w, nh, nw, hb, wb, scratch, row)
        grids.append((1, hb // P, wb // P))
        off += (h * w * 3 + 15) // 16 * 16
        if (nh, nw) != (h, w):
            scratch += nh * nw * 3
        row += (hb // P) * (wb // P)
        if off >= 2 ** 31 or scratch >= 2 ** 31:
            raise _lib.SuryaB200Error("device preprocessing: more than 2 GiB of crops in one call; split the batch")
    nbytes = max(off, 16)
    packed = np.zeros(nbytes, dtype=np.uint8) if staging is None else staging(nbytes)
    for i, c in enumerate(crops):
        o, h, w = int(desc[i, 0]), int(desc[i, 1]), int(desc[i, 2])
        packed[o:o + h * w * 3] = np.ascontiguousarray(c).reshape(-1)
    mx = tuple(int(desc[:, k].max()) if len(crops) else 0 for k in (3, 4, 5, 6))
    return {"packed": packed, "desc": desc.reshape(-1), "grids": grids, "n_rows": row, "scratch_floats": scratch,
            "any_stage1": int(scratch > 0), "max": mx, "nbytes": nbytes}


def prompt_tokens(cfg: RecConfig, n_image_tokens: int, math_mode: bool = True, text_ids: Sequence[int] = ()) -> np.ndarray:
    """Token layout of one ocr_with_boxes prompt (processor/__init__.py:247-248, 260-274, 312)."""
    ids = [cfg.image_token_id] * n_image_tokens + list(cfg.register_token_ids[: cfg.num_register_tokens])
    ids += [cfg.ocr_with_boxes_bos_id] + ([] if math_mode else [cfg.nomath_token_id]) + list(text_ids) + [cfg.eoi_token_id]
    return np.asarray(ids, dtype=np.int64)


def detect_repeat_token(tokens: List[int], max_repeats: int = 40) -> bool:
    """Mirror of surya/recognition/util.py:59-69."""
    if len(tokens) < max_repeats:
        return False
    last_n = tokens[-max_repeats:]
    u = len(set(last_n))
    if u > 5:
        return False
    return last_n[-u:] == last_n[-u * 2: -u]


def _pin(t: torch.Tensor) -> torch.Tensor:
    """Page-locked copy of a host tensor (asynchronous H2D / D2H); a no-op for device tensors, already pinned tensors, and in a
    process without CUDA (the CPU tests drive the runner over the oracle engine)."""
    if t.is_cuda or t.is_pinned() or not torch.cuda.is_available():
        return t
    return t.pin_memory()


class RecognitionRunner:
    """Mirror of RecognitionPredictor.prediction_loop (surya/recognition/__init__.py:501-607) on engine slots.

    Same scheduling rule (prefill when more than `min_prefill_ratio` of the slots are free and prompts wait,
    else decode), same stop rules (EOS / NO_OUTPUT after prefill; EOS / PAD / max_tokens / repeat during
    decode), same outputs (token list, score list, bbox [max_tokens, 6] per crop).  Differences are internal:
    ragged prefill instead of left padding, slot cache instead of merge/trim, `poll` decode steps per host
    round-trip instead of one (tokens generated past a stop are dropped; per-prompt results are unchanged
    because rows are independent, SURVEY.md §9.5)."""

    min_prefill_ratio = 0.2

    MAX_REPEATS = 40     # detect_repeat_token's default window (surya/recognition/util.py:59)

    def __init__(self, engine: RecEngine, batch_size: int = 256, max_tokens: int = 128, poll: int = 8, stop_rules: str = "device"):
        """stop_rules: "device" (default) — EOS / PAD / max_tokens / detect_repeat_token are evaluated by a kernel after every decode
        step (sb_rec_set_sched) and the host reads one count per row and round trip; "host" — the per-token Python loop of the
        reference.  Both give identical results (tests/test_rec_gpu.py::test_device_stop_rules_equal_host_rules)."""
        if stop_rules not in ("device", "host"):
            raise ValueError("stop_rules must be 'device' or 'host'")
        self.engine, self.batch_size, self.max_tokens, self.poll = engine, batch_size, max_tokens, max(1, poll)
        self.stop_rules = stop_rules

    def preprocess(self, crops: Sequence[np.ndarray], math_mode: bool = True, workers: Optional[int] = None):
        """Host side of SuryaOCRProcessor for one crop each (scale_to_fit -> resize to x28 -> normalise -> merge-block-major
        tiles, processor/__init__.py:140-230) — the OpenCV resizes release the GIL, so crops are processed by a small thread
        pool; results are in input order and identical to the serial loop."""
        cfg = self.engine.cfg

        def one(crop):
            img = scale_to_fit(np.asarray(crop, dtype=np.float32), (1024, 256))
            t, g = tile_image(img, cfg.vision_encoder.patch_size, cfg.merge_size)
            return t, g, prompt_tokens(cfg, t.shape[0] // cfg.merge_size ** 2, math_mode)

        n = len(crops)
        if workers is None:
            import os
            try:
                avail = len(os.sched_getaffinity(0))
            except AttributeError:
                avail = os.cpu_count() or 1
            workers = max(1, min(16, avail, n // 8))
        if workers <= 1 or n < 16:
            res = [one(c) for c in crops]
        else:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=workers) as ex:
                res = list(ex.map(one, crops))
        return [r[0] for r in res], [r[1] for r in res], [r[2] for r in res]

    def preprocess_device(self, crops: Sequence[np.ndarray], math_mode: bool = True):
        """Device side of SuryaOCRProcessor for uint8 crops (SURVEY §8 f2): ONE pinned uint8 upload (3 B / pixel), then
        sb_rec_preprocess does scale_to_fit (Lanczos4), the resize to x28 (cubic), normalisation and tiling on the GPU and leaves the
        fp32 tiles in HBM, where run_preprocessed's prefill reads them.  Same return contract as preprocess(), tiles as one packed
        CUDA tensor."""
        eng, cfg = self.engine, self.engine.cfg
        dev = eng.device
        P, m = cfg.vision_encoder.patch_size, cfg.merge_size
        if len(crops) == 0:
            return torch.zeros((0, 3 * P * P), dtype=torch.float32, device=dev), [], []

        def staging(nbytes):        # grow-only pinned staging buffer: crops are packed straight into page-locked memory
            torch.cuda.current_stream().synchronize()        # the previous call's asynchronous copy out of it must have finished
            pin = getattr(self, "_pp_pin", None)
            if pin is None or pin.numel() < nbytes:
                pin = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8).pin_memory()
                self._pp_pin = pin
            return pin.numpy()[:nbytes]

        plan = build_preprocess_plan(crops, cfg, staging=staging)
        seqs = [prompt_tokens(cfg, g[1] * g[2] // m ** 2, math_mode) for g in plan["grids"]]
        host = self._pp_pin[:plan["nbytes"]]
        desc_h = torch.from_numpy(plan["desc"]).pin_memory()
        packed = host.to(dev, non_blocking=True)
        desc = desc_h.to(dev, non_blocking=True)
        tiles = torch.empty((plan["n_rows"], 3 * P * P), dtype=torch.float32, device=dev)
        scratch = torch.empty(max(plan["scratch_floats"], 1), dtype=torch.float32, device=dev)
        mean = (ctypes.c_float * 3)(*IMAGE_MEAN.tolist())
        std = (ctypes.c_float * 3)(*IMAGE_STD.tolist())
        mx = plan["max"]
        check(eng.lib.sb_rec_preprocess(ptr(packed), ptr(desc), c_int(len(crops)), c_int(mx[0]), c_int(mx[1]), c_int(mx[2]), c_int(mx[3]),
                                        c_int(plan["any_stage1"]), ptr(scratch), ptr(tiles), c_int(tiles.stride(0)), c_int(P), c_int(m),
                                        mean, std, stream_ptr()), "sb_rec_preprocess")
        # the pinned staging buffers must outlive the asynchronous copies: keep them until the next call
        self._pp_keep = (host, desc_h, packed, desc, scratch)
        return tiles, plan["grids"], seqs

    def run_preprocessed(self, tiles, grids, seqs, fixed_steps: bool = False):
        """tiles: per-crop list of [P_i, patch_dim] arrays, or ONE packed [sum P_i, patch_dim] array / torch tensor in crop
        order (pinned host memory makes the upload a single async DMA with no staging copy).
        Returns (tokens: List[List[int]], scores: List[List[float]], bboxes: np.ndarray [N, max_tokens, 6])."""
        eng, cfg = self.engine, self.engine.cfg
        dev = eng.device
        N = len(seqs)
        if N == 0:       # the predictor returns before touching the model on empty input (surya/recognition/__init__.py:835-837)
            return [], [], np.zeros((0, self.max_tokens, 6), dtype=np.int64)
        packed = None
        if not isinstance(tiles, (list, tuple)):
            packed = tiles if isinstance(tiles, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(tiles))
            n_rows = np.array([int(g[0] * g[1] * g[2]) for g in grids], dtype=np.int64)
            row_off = np.concatenate([[0], np.cumsum(n_rows)])
            if packed.shape[0] != row_off[-1]:
                raise _lib.SuryaB200Error("packed tiles do not match grid_thw")

        def tiles_for(take):
            if packed is None:
                return _pin(torch.from_numpy(np.concatenate([tiles[i] for i in take], 0)))
            if all(b == a + 1 for a, b in zip(take, take[1:])):
                tl = packed[row_off[take[0]]: row_off[take[-1] + 1]]
            else:
                tl = torch.cat([packed[row_off[i]: row_off[i + 1]] for i in take], 0)
            return _pin(tl)
        tokens: List[List[int]] = [[] for _ in range(N)]
        scores: List[List[float]] = [[] for _ in range(N)]
        bboxes = np.zeros((N, self.max_tokens, 6), dtype=np.int64)
        queue = deque(range(N))
        Bsz = self.batch_size
        if eng.max_slots < Bsz + 1:
            raise _lib.SuryaB200Error(f"RecognitionRunner(batch_size={Bsz}) needs an engine with max_slots >= {Bsz + 1} "
                                      f"(one scratch slot for idle rows); this engine has {eng.max_slots}")
        scratch = eng.alloc_slots(1)[0]      # idle rows decode into a scratch slot (the reference decodes every row too)
        row_prompt: List[Optional[int]] = [None] * Bsz
        row_slot = [scratch] * Bsz
        # persistent per-runner buffers: same device pointers every call (the captured decode graph is reused) and no
        # cudaHostAlloc / cudaMalloc on the per-batch path
        T = max(1, self.max_tokens)
        bufs = getattr(self, "_bufs", None)
        if bufs is None or bufs["key"] != (Bsz, T):
            bufs = {"key": (Bsz, T),
                    "ids_io": torch.empty((Bsz,), dtype=torch.int64, device=dev),
                    "pos_host": _pin(torch.zeros(Bsz, dtype=torch.int32)),
                    "slot_host": _pin(torch.zeros(Bsz, dtype=torch.int32)),
                    "pos_io": torch.zeros(Bsz, dtype=torch.int32, device=dev),
                    "slot_t": torch.zeros(Bsz, dtype=torch.int32, device=dev),
                    "hist": {"tok": torch.empty((T, Bsz), dtype=torch.int64, device=dev),
                             "score": torch.empty((T, Bsz), dtype=torch.float32, device=dev),
                             "bbox": torch.empty((T, Bsz, 6), dtype=torch.int64, device=dev),
                             "done": torch.empty((T, Bsz), dtype=torch.uint8, device=dev)}}
            self._bufs = bufs
        ids_io, pos_host, slot_host = bufs["ids_io"], bufs["pos_host"], bufs["slot_host"]
        pos_io, slot_t, hist = bufs["pos_io"], bufs["slot_t"], bufs["hist"]
        ids_io.fill_(cfg.pad_token_id)
        # device-side stop rules (SURVEY §8 f3): per-row generated-token count, last-40-token ring and sticky done flag live on the
        # device and are advanced by stop_rules_kernel after every step; the host reads one count + one flag per row and round trip
        sched = None
        if self.stop_rules == "device" and not fixed_steps:
            sched = bufs.get("sched")
            if sched is None:
                sched = {"gen": torch.zeros(Bsz, dtype=torch.int32, device=dev),
                         "ring": torch.zeros((Bsz, self.MAX_REPEATS), dtype=torch.int64, device=dev),
                         "done": torch.ones(Bsz, dtype=torch.uint8, device=dev),
                         "valid": torch.zeros(Bsz, dtype=torch.int32, device=dev),
                         "active": torch.zeros(1, dtype=torch.int32, device=dev),
                         "gen_host": _pin(torch.zeros(Bsz, dtype=torch.int32)),
                         "done_host": _pin(torch.ones(Bsz, dtype=torch.uint8))}
                bufs["sched"] = sched
            eng.set_sched(sched, self.max_tokens, self.MAX_REPEATS)

        def finish(row):
            eng.release_slots([row_slot[row]])
            row_slot[row] = scratch
            row_prompt[row] = None

        try:
            while queue or any(p is not None for p in row_prompt):
                empty = [r for r in range(Bsz) if row_prompt[r] is None]
                if queue and len(empty) / Bsz > self.min_prefill_ratio:
                    # at most one prompt per empty row (the reference's rule, :356-359), further bounded by what the engine
                    # can take in ONE prefill: free KV slots, patch rows and token rows of its workspaces (the reference
                    # bounds the same thing with encoder_chunk_size); the rest of the queue waits for the next prefill
                    take, n_p, n_t = [], 0, 0
                    while queue and len(take) < min(len(empty), len(eng.free_slots)):
                        i = queue[0]
                        p_i = int(grids[i][0] * grids[i][1] * grids[i][2])
                        if take and (n_p + p_i > eng.max_patches or n_t + len(seqs[i]) > eng.max_tokens):
                            break
                        if p_i > eng.max_patches or len(seqs[i]) > eng.max_tokens or len(seqs[i]) + self.max_tokens > eng.s_max:
                            raise _lib.SuryaB200Error(
                                f"crop {i} needs {p_i} patches / {len(seqs[i])} prompt tokens + {self.max_tokens} generated: beyond "
                                f"the engine's capacity (max_patches={eng.max_patches}, max_tokens={eng.max_tokens}, s_max={eng.s_max})")
                        take.append(queue.popleft())
                        n_p, n_t = n_p + p_i, n_t + len(seqs[i])
                    rows = empty[: len(take)]
                    new_slots = eng.alloc_slots(len(take))
                    try:
                        tl = tiles_for(take)
                        if not tl.is_cuda:     # start the (pinned, asynchronous) upload first; the index plan is built meanwhile
                            tl = tl.to(dev, non_blocking=True)
                        plan = build_prefill_plan(cfg, np.array([grids[i] for i in take]), [seqs[i] for i in take], new_slots)
                        out = eng.prefill(tl, plan)
                    except Exception:
                        eng.release_slots(new_slots)
                        raise
                    rows_t = torch.tensor(rows, dtype=torch.int64, device=dev)
                    ids_io[rows_t] = out["next_ids"]
                    if sched is not None:           # the prefill token is token 0 of the row's repeat window
                        sched["ring"][rows_t, 0] = out["tok"]
                    tok_h, sc_h, bb_h = out["tok"].cpu().numpy(), out["score"].cpu().numpy(), out["bbox"].cpu().numpy()
                    for j, (r, p) in enumerate(zip(rows, take)):
                        row_prompt[r], row_slot[r] = p, new_slots[j]
                        tokens[p].append(int(tok_h[j]))
                        scores[p].append(float(sc_h[j]))
                        bboxes[p, 0] = bb_h[j]
                        stop = (not fixed_steps) and tokens[p][-1] in (cfg.eos_token_id, cfg.no_output_token_id)
                        if stop or self.max_tokens <= 1:
                            finish(r)
                else:
                    active = [r for r in range(Bsz) if row_prompt[r] is not None]
                    remaining = min(self.max_tokens - len(tokens[row_prompt[r]]) for r in active)
                    n = max(1, remaining if fixed_steps else min(self.poll, remaining))
                    # one vectorised write per (page-locked) staging array instead of a tensor element store per row; the previous
                    # round trip's asynchronous copies out of them finished with its history read-back
                    pos_host.numpy()[:] = [0 if p is None else len(seqs[p]) + len(tokens[p]) - 1 for p in row_prompt]
                    slot_host.numpy()[:] = row_slot
                    pos_io.copy_(pos_host, non_blocking=True)
                    slot_t.copy_(slot_host, non_blocking=True)
                    if sched is not None:
                        sched["gen_host"].numpy()[:] = [0 if p is None else len(tokens[p]) for p in row_prompt]
                        sched["done_host"].numpy()[:] = [1 if p is None else 0 for p in row_prompt]
                        sched["gen"].copy_(sched["gen_host"], non_blocking=True)
                        sched["done"].copy_(sched["done_host"], non_blocking=True)
                    eng.decode_steps(ids_io, slot_t, pos_io, n, hist=hist, max_pos=int(pos_host.numpy().max()))
                    th, sh, bh = hist["tok"][:n].cpu().numpy(), hist["score"][:n].cpu().numpy(), hist["bbox"][:n].cpu().numpy()
                    if sched is not None:
                        valid_h, done_h = sched["valid"].cpu().numpy(), sched["done"].cpu().numpy()
                        for r in active:             # the device already applied the stop rules: take each row's valid prefix
                            p = row_prompt[r]
                            k, m = len(tokens[p]), int(valid_h[r])
                            tokens[p].extend(th[:m, r].tolist())
                            scores[p].extend(sh[:m, r].tolist())
                            bboxes[p, k:k + m] = bh[:m, r]
                            if done_h[r]:
                                finish(r)
                        continue
                    for r in active:
                        p = row_prompt[r]
                        if fixed_steps:           # no stop rules to evaluate: unpack the whole chunk at once
                            k = len(tokens[p])
                            m = min(n, self.max_tokens - k)
                            tokens[p].extend(th[:m, r].tolist())
                            scores[p].extend(sh[:m, r].tolist())
                            bboxes[p, k:k + m] = bh[:m, r]
                            if len(tokens[p]) >= self.max_tokens:
                                finish(r)
                            continue
                        for s in range(n):
                            k = len(tokens[p])
                            tokens[p].append(int(th[s, r]))
                            scores[p].append(float(sh[s, r]))
                            bboxes[p, k] = bh[s, r]
                            full = len(tokens[p]) >= self.max_tokens
                            if fixed_steps:
                                stop = full
                            else:
                                stop = tokens[p][-1] in (cfg.eos_token_id, cfg.pad_token_id) or full or \
                                    detect_repeat_token(tokens[p], self.MAX_REPEATS)
                            if stop:
                                finish(r)
                                break
        finally:
            for r in range(Bsz):
                if row_prompt[r] is not None:
                    finish(r)
            eng.release_slots([scratch])
            if sched is not None:
                eng.set_sched(None)          # the state tensors belong to this runner: never leave the engine pointing at them
        return tokens, scores, bboxes

    def run(self, crops: Sequence[np.ndarray], math_mode: bool = True, fixed_steps: bool = False, preprocess: str = "host"):
        """preprocess: "host" — the OpenCV thread pool (any pixel dtype); "device" — uint8 crops, resized / normalised / tiled by
        sb_rec_preprocess on the GPU (equal to the OpenCV path to float32 rounding, tests/test_preproc_gpu.py)."""
        if preprocess not in ("host", "device"):
            raise ValueError("preprocess must be 'host' or 'device'")
        tiles, grids, seqs = self.preprocess_device(crops, math_mode) if preprocess == "device" else self.preprocess(crops, math_mode)
        return self.run_preprocessed(tiles, grids, seqs, fixed_steps=fixed_steps)
