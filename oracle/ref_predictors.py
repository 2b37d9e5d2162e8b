"""ORACLE TOOLING (test infrastructure, build container only) — drive the reference's *unmodified predictor classes*.

  * install_predictors()      ref_shim.install() + the two transformers names surya.recognition imports that 5.x dropped
                              (QuantizedCacheConfig, HQQQuantizedCache: only constructed on the HQQ path, never here)
  * synthetic_ocr_processor   the reference's real SuryaOCRProcessor over a stand-in tokenizer table whose special-token
                              ids are the ones surya_b200.config.RecConfig declares (the shipped tokenizer needs
                              checkpoint files that are unavailable offline, SURVEY.md §8c)
  * OracleRecEngine           RecEngine's call surface (alloc/release slots, prefill(tiles, plan), decode(ids, slot, pos))
                              computed by the CPU oracle — lets the reference RecognitionPredictor run over
                              B200SuryaModel + SlotCache (the drop-in boundary code) in a container without a GPU
  * record_rec_trace          run RecognitionPredictor.prediction_loop and log every model call / cache operation, so the
                              GPU tests can replay the exact call sequence against the CUDA engine (tests/golden/
                              rec_predictor_trace.pt; the tests run without the reference)

Only tests/ and oracle/make_golden.py import this module.
"""
from __future__ import annotations

import sys
from collections import deque
from typing import Dict, List, Sequence

import numpy as np
import torch

from . import rec_oracle as O
from . import ref_shim


def install_predictors() -> None:
    ref_shim.install()
    import surya.common.surya  # noqa: F401  (importing it swaps sys.modules['transformers'] for the loaded lazy module)

    tr = sys.modules["transformers"]
    if "HQQQuantizedCache" not in tr.__dict__:
        tr.__dict__["HQQQuantizedCache"] = type("HQQQuantizedCache", (object,), {})
    if "QuantizedCacheConfig" not in tr.__dict__:
        tr.__dict__["QuantizedCacheConfig"] = type("QuantizedCacheConfig", (object,), {"__init__": lambda self, *a, **k: None})


# ------------------------------------------------------------------------------------------------ processor
class _TokenTable:
    """Stand-in for SuryaOCRTokenizer (surya/common/surya/processor/tokenizer.py:228-256): just the tables and the
    call the processor uses (processor/__init__.py:63-121, 264)."""

    def __init__(self, cfg):
        from surya.common.surya.processor import (BLOCK_WITHOUT_BOXES_TOKEN, EOI_TOKEN, EOS_TOKEN, IMAGE_ROTATED_TOKEN,
                                                  IMAGE_TOKEN, NO_OUTPUT_TOKEN, NOMATH_TOKEN, OCR_WITH_BOXES_BOS_TOKEN,
                                                  OCR_WITHOUT_BOXES_BOS_TOKEN, PAD_TOKEN, REGISTER_TOKENS)

        self.vocab_size = cfg.vocab_size
        sysmap = {EOS_TOKEN: cfg.eos_token_id, PAD_TOKEN: cfg.pad_token_id, IMAGE_TOKEN: cfg.image_token_id,
                  OCR_WITH_BOXES_BOS_TOKEN: cfg.ocr_with_boxes_bos_id, EOI_TOKEN: cfg.eoi_token_id,
                  NO_OUTPUT_TOKEN: cfg.no_output_token_id, NOMATH_TOKEN: cfg.nomath_token_id,
                  IMAGE_ROTATED_TOKEN: 12, OCR_WITHOUT_BOXES_BOS_TOKEN: 13, BLOCK_WITHOUT_BOXES_TOKEN: 14}
        for name, tid in zip(REGISTER_TOKENS, cfg.register_token_ids):
            sysmap[name] = tid
        self.system_tokens = dict(sysmap)
        self.SPECIAL_TOKEN_MAPPING = dict(sysmap)
        self.special_tokens = {"math_external": [], "system": list(sysmap), "formatting": [], "all": list(sysmap)}

    def __call__(self, texts, tasks=None, **kw):
        if isinstance(texts, str):
            texts = [texts]
        out = []
        for t in texts:
            if t:
                raise NotImplementedError("the synthetic tokenizer table only handles empty input text")
            out.append([])
        return {"input_ids": out}


def synthetic_ocr_processor(cfg):
    install_predictors()
    from surya.common.surya.processor import SuryaOCRProcessor

    return SuryaOCRProcessor(ocr_tokenizer=_TokenTable(cfg), blank_bbox_token_id=cfg.bbox_size,
                             num_register_tokens=cfg.num_register_tokens, patch_size=cfg.vision_encoder.patch_size,
                             merge_size=cfg.merge_size, model_device="cpu")


# ------------------------------------------------------------------------------------------------ engine double
class OracleRecEngine:
    """Same surface as surya_b200.recognition.RecEngine, computed by oracle.rec_oracle on the CPU (one OracleCache per
    slot, sequences stored unpadded exactly like the engine's slot cache)."""

    def __init__(self, cfg, state_dict: Dict[str, torch.Tensor], dtype=torch.float32, max_slots: int = 16, s_max: int = 256):
        self.cfg, self.dtype, self.device = cfg, dtype, torch.device("cpu")
        self.sd = O.cast_sd(state_dict, dtype)
        self.s_max, self.max_slots = s_max, max_slots
        self.max_patches, self.max_tokens = 1 << 30, 1 << 30
        self.free_slots = deque(range(max_slots))
        self.caches: Dict[int, O.OracleCache] = {}
        self.calls: List[str] = []

    def alloc_slots(self, n: int) -> List[int]:
        if n > len(self.free_slots):
            raise RuntimeError(f"out of KV slots: need {n}, free {len(self.free_slots)}")
        return [self.free_slots.popleft() for _ in range(n)]

    def release_slots(self, slots: Sequence[int]):
        for s in slots:
            self.caches.pop(int(s), None)
            self.free_slots.append(int(s))

    def _pack(self, lm, bb):
        nxt, preds, bx, done, sc = O.process_outputs(lm, bb, self.cfg)
        return {"logits": lm[:, 0], "tok": preds[:, 0], "score": sc[:, 0], "bbox": bx[:, 0],
                "bbox_sig": bb[:, 0].float(), "done": done.to(torch.uint8), "next_ids": nxt[:, 0]}

    def prefill(self, tiles: torch.Tensor, plan, want_logits: bool = False):
        cfg = self.cfg
        ints = plan.ints.numpy()

        def arr(name):
            o, n = plan.off[name]
            return ints[o:o + n]

        ids = plan.ids.numpy()
        starts, lens, slots = arr("seq_start"), arr("seq_len"), arr("tok_slot")
        img_start, img_len, pos_rc = arr("img_start"), arr("img_len"), arr("pos_rc").reshape(-1, 2)
        unit = cfg.merge_size ** 2
        img = 0
        lms, bbs = [], []
        self.calls.append(f"prefill:{len(lens)}")
        with torch.inference_mode():
            for s0, ln in zip(starts, lens):
                seq = torch.from_numpy(ids[s0:s0 + ln].copy()).unsqueeze(0)
                need = int((seq == cfg.image_token_id).sum()) * unit
                t_parts, grids = [], []
                while need > 0:
                    a, n = int(img_start[img]), int(img_len[img])
                    rc = pos_rc[a:a + n]
                    grids.append((1, int(rc[:, 0].max()) + 1, int(rc[:, 1].max()) + 1))
                    t_parts.append(tiles[a:a + n])
                    need -= n
                    img += 1
                assert need == 0, "image tokens and image patches do not line up"
                cache = O.OracleCache()
                mask = torch.ones_like(seq)
                pos = torch.arange(ln, dtype=torch.long).unsqueeze(0)
                lm, bb = O.model_forward(self.sd, cfg, seq, mask, pos, cache,
                                         torch.cat(t_parts, 0).to(self.dtype) if t_parts else None,
                                         np.array(grids, dtype=np.int64) if grids else None)
                self.caches[int(slots[s0])] = cache
                lms.append(lm)
                bbs.append(bb)
        return self._pack(torch.cat(lms, 0), torch.cat(bbs, 0))

    def decode(self, input_ids: torch.Tensor, slot: torch.Tensor, pos: torch.Tensor, want_logits: bool = False, max_pos=None):
        lms, bbs = [], []
        self.calls.append(f"decode:{input_ids.numel()}")
        with torch.inference_mode():
            for b in range(input_ids.numel()):
                cache = self.caches[int(slot[b])]
                n = cache.seq_len()
                lm, bb = O.model_forward(self.sd, self.cfg, input_ids[b].reshape(1, 1).long(),
                                         torch.ones((1, n + 1), dtype=torch.long), pos[b].reshape(1, 1).long(), cache)
                lms.append(lm)
                bbs.append(bb)
        return self._pack(torch.cat(lms, 0), torch.cat(bbs, 0))


    # -- device-loop surface of RecEngine (sb_rec_decode_steps / sb_rec_set_sched), so that RecognitionRunner's scheduling logic
    #    runs on the CPU exactly as it runs over the CUDA engine (tests/test_runner_cpu.py)
    def set_sched(self, state, max_tokens: int = 0, max_repeats: int = 40):
        self.sched = None if state is None else (state, int(max_tokens), int(max_repeats))

    def decode_steps(self, ids_io, slot, pos_io, n_steps, hist=None, use_graph=True, max_pos=None):
        cfg, B = self.cfg, ids_io.numel()
        if max_pos is not None and max_pos + n_steps > self.s_max:
            raise RuntimeError("decode would run past s_max")
        sched = getattr(self, "sched", None)
        if sched is not None:
            sched[0]["valid"].zero_()
        for s in range(n_steps):
            live = [b for b in range(B) if int(slot[b]) in self.caches]
            hist["tok"][s].fill_(cfg.pad_token_id)
            hist["score"][s].zero_()
            hist["bbox"][s].zero_()
            hist["done"][s].fill_(1)
            if live:
                idx = torch.tensor(live, dtype=torch.long)
                out = self.decode(ids_io[idx], slot[idx], pos_io[idx])
                hist["tok"][s, idx], hist["score"][s, idx] = out["tok"], out["score"]
                hist["bbox"][s, idx], hist["done"][s, idx] = out["bbox"], out["done"]
                ids_io[idx] = out["next_ids"]
            pos_io += 1
            if sched is not None:
                stop_rules_step(hist["tok"], hist["done"], s, *[sched[0][k] for k in ("gen", "ring", "done", "valid", "active")],
                                sched[1], sched[2])
        return hist


def stop_rules_step(tok_hist, done_hist, s, gen, ring, row_done, n_valid, n_active, max_tokens, R):
    """Python mirror of stop_rules_kernel (surya_b200/csrc/ops.cu): the stop rules of RecognitionPredictor.prediction_loop
    (surya/recognition/__init__.py:585-598, util.py:59-69) on the per-row scheduler state, one call per decode step."""
    active = 0
    for r in range(gen.numel()):
        if int(row_done[r]):
            continue
        tok = int(tok_hist[s, r])
        cnt = int(gen[r]) + 1
        gen[r] = cnt
        ring[r, (cnt - 1) % R] = tok
        stop = bool(done_hist[s, r]) or cnt >= max_tokens
        if not stop and cnt >= R:
            last = [int(ring[r, (cnt + j) % R]) for j in range(R)]          # oldest first
            u = len(set(last))
            if u <= 5 and 2 * u <= R:
                stop = last[R - u:] == last[R - 2 * u: R - u]
        n_valid[r] = s + 1
        if stop:
            row_done[r] = 1
        else:
            active += 1
    n_active[0] = active


# ------------------------------------------------------------------------------------------------ trace recording
class TracingModel:
    """Wraps a B200SuryaModel: logs the inputs of every call the predictor makes and the tokens that came back."""

    def __init__(self, inner, events: list):
        self.inner, self.events = inner, events
        self.config, self.device, self.dtype = inner.config, inner.device, inner.dtype

    def to(self, *a, **k):
        return self

    def __call__(self, **kw):
        out = self.inner(**kw)
        ev = {"kind": "prefill" if kw.get("image_tiles") is not None else "decode",
              "input_ids": kw["input_ids"].detach().cpu().clone(),
              "attention_mask": kw["attention_mask"].detach().cpu().clone(),
              "position_ids": kw["position_ids"].detach().cpu().clone(),
              "cache_id": id(kw["past_key_values"]),
              "tok": out["lm_logits"][:, -1].float().argmax(-1).cpu().clone(),
              "margin": (lambda t: (t.values[:, 0] - t.values[:, 1]))(out["lm_logits"][:, -1].float().topk(2, -1)).cpu().clone(),
              "bbox": out["bbox_logits"][:, -1].float().cpu().clone()}
        if ev["kind"] == "prefill":
            ev["grid_thw"] = kw["grid_thw"].detach().cpu().clone()
            ev["tiles_sum"] = float(kw["image_tiles"].double().sum())
            ev["n_tiles"] = int(kw["image_tiles"].shape[0])
        self.events.append(ev)
        return out


def record_rec_trace(cfg, state_dict, crops: List[np.ndarray], batch_size: int, max_tokens: int, dtype=torch.float32,
                     min_trim_length: int | None = None):
    """Run the reference RecognitionPredictor.prediction_loop (unmodified) over B200SuryaModel(OracleRecEngine) and
    return (events, predicted_tokens, bboxes, scores).  Cache operations are logged by wrapping SlotCache methods."""
    install_predictors()
    from surya.common.surya.schema import TaskNames
    from surya.settings import settings
    from surya_b200 import dropin
    from surya_b200.recognition import B200SuryaModel, SlotCache

    events: list = []
    eng = OracleRecEngine(cfg, state_dict, dtype=dtype, max_slots=4 * batch_size + 4)
    model = TracingModel(B200SuryaModel(eng), events)
    pred = dropin.recognition_predictor(model, synthetic_ocr_processor(cfg), device="cpu", dtype=dtype)
    if min_trim_length is not None:
        pred.min_trim_length = min_trim_length
    orig_merge, orig_trim = SlotCache.merge, SlotCache.trim_left

    def merge(self, new_cache, idxs, device=None):
        off = orig_merge(self, new_cache, idxs, device)
        events.append({"kind": "merge", "cache_id": id(self), "new_id": id(new_cache), "idxs": [int(i) for i in idxs], "offset": int(off)})
        return off

    def trim(self, n):
        events.append({"kind": "trim", "cache_id": id(self), "n": int(n)})
        return orig_trim(self, n)

    SlotCache.merge, SlotCache.trim_left = merge, trim
    old_max = settings.RECOGNITION_MAX_TOKENS
    settings.RECOGNITION_MAX_TOKENS = max_tokens
    pred.disable_tqdm = True
    try:
        flat = {"slices": [np.asarray(c, dtype=np.float32) for c in crops], "input_text": [None] * len(crops),
                "task_names": [TaskNames.ocr_with_boxes] * len(crops)}
        tokens, bboxes, scores = pred.prediction_loop(flat, recognition_batch_size=batch_size, math_mode=True)
    finally:
        SlotCache.merge, SlotCache.trim_left = orig_merge, orig_trim
        settings.RECOGNITION_MAX_TOKENS = old_max
    # stable small ids for the caches
    ids = {}
    for ev in events:
        for k in ("cache_id", "new_id"):
            if k in ev:
                ev[k] = ids.setdefault(ev[k], len(ids))
    return events, tokens, bboxes, scores, eng


# ------------------------------------------------------------------------------------------------ trace replay (no reference)
def replay_rec_trace(model, trace: dict, crops: List[np.ndarray], tile_fn, check):
    """Re-issue the recorded model calls / cache operations of a RecognitionPredictor.prediction_loop run against `model`
    (a B200SuryaModel over any engine) without the reference: prefill events carry the padded ids / masks / position ids the
    reference's processor built (tiles are regenerated from the seeded crops with `tile_fn` and checked against the recorded
    checksum), decode events carry the masks and position ids the predictor maintained, merge / trim events are applied to
    the SlotCache objects exactly where the predictor applied them.  check(event_index, event, out) compares the outputs."""
    from surya_b200.recognition import SlotCache

    caches: Dict[int, SlotCache] = {}
    queue = deque(range(len(crops)))
    dev = model.device
    for i, ev in enumerate(trace["events"]):
        kind = ev["kind"]
        if kind == "prefill":
            n = ev["input_ids"].shape[0]
            take = [queue.popleft() for _ in range(n)]
            tiles = torch.cat([tile_fn(crops[j]) for j in take], 0)
            assert tiles.shape[0] == ev["n_tiles"] and abs(float(tiles.double().sum()) - ev["tiles_sum"]) < 1e-3 * max(1.0, abs(ev["tiles_sum"])), \
                "regenerated tiles differ from the ones the reference processor produced"
            cache = caches.setdefault(ev["cache_id"], SlotCache())
            out = model(input_ids=ev["input_ids"].to(dev), image_tiles=tiles.to(dev, model.dtype), grid_thw=ev["grid_thw"].to(dev),
                        attention_mask=ev["attention_mask"].to(dev), position_ids=ev["position_ids"].to(dev), inputs_embeds=None,
                        past_key_values=cache, use_cache=True, logits_to_keep=1, encoder_chunk_size=4096)
            check(i, ev, out)
        elif kind == "decode":
            out = model(input_ids=ev["input_ids"].to(dev), attention_mask=ev["attention_mask"].to(dev),
                        position_ids=ev["position_ids"].to(dev), use_cache=True, past_key_values=caches[ev["cache_id"]],
                        logits_to_keep=1)
            check(i, ev, out)
        elif kind == "merge":
            off = caches[ev["cache_id"]].merge(caches.pop(ev["new_id"]), ev["idxs"], dev)
            assert off == ev["offset"], f"event {i}: merge offset {off} != recorded {ev['offset']}"
        elif kind == "trim":
            caches[ev["cache_id"]].trim_left(ev["n"])
    for c in caches.values():
        c.release()


# ------------------------------------------------------------------------------------------------ detection
class OracleDetEngine:
    """DetEngine's forward surface computed by oracle.det_oracle (CPU)."""

    def __init__(self, cfg, state_dict, dtype=torch.float32):
        self.cfg, self.sd, self.dtype, self.device = cfg, state_dict, dtype, torch.device("cpu")

    def forward(self, pixel_values: torch.Tensor, out=None):
        from . import det_oracle as D

        with torch.inference_mode():
            return D.forward(self.sd, self.cfg, pixel_values.float()).to(self.dtype)


def synthetic_det_processor(size: int = 1024):
    """The reference's SegformerImageProcessor configured like the shipped preprocessor_config.json would (size forced,
    SURVEY.md §8d config 1: the checkpoint's json is unavailable offline)."""
    ref_shim.install()
    from surya.detection.processor import SegformerImageProcessor

    return SegformerImageProcessor(size={"height": size, "width": size})


def conftest_page(size: int = 1024):
    """The reference's own test page (tests/conftest.py:50-61)."""
    from PIL import Image, ImageDraw

    image = Image.new("RGB", (size, size), "white")
    draw = ImageDraw.Draw(image)
    draw.text((10, 10), "Hello World", fill="black", font_size=72)
    draw.text((10, 200), "This is a sentence of text.\nNow it is a paragraph.\nA three-line one.", fill="black", font_size=24)
    return image
