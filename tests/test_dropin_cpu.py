"""Drop-in boundary (SURVEY.md §8b) on CPU.

The reference's UNMODIFIED predictor classes were run over the B200 model mirrors (B200SuryaModel + SlotCache, B200EfficientViT)
with the CPU oracle as the engine, and its host post-processing on seeded heat maps; oracle/make_golden.py stored what they
returned under tests/golden/ (rec_predictor_trace.pt, reference_host.pt).  These tests hold the oracle, the boundary code and the
product's host stages to those outputs without the reference installed.  tests/test_rec_gpu.py replays the same predictor trace
against the CUDA engine.
"""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import rec_oracle as O

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"


def _tile_fn(cfg):
    def fn(crop):
        img = O.scale_to_fit(np.asarray(crop, dtype=np.float32), (1024, 256))
        return O.process_and_tile(img, cfg.vision_encoder.patch_size, cfg.merge_size)[0]
    return fn


def test_reference_recognition_predictor_dropin_cpu():
    """What RecognitionPredictor.prediction_loop (reference code, unmodified: prefill with its own `ContinuousBatchingCache()`,
    merge, mask/position bookkeeping, maybe_trim_cache_padding, stop rules, `del self.kv_cache`) returned over B200SuryaModel +
    SlotCache (tests/golden/rec_predictor_trace.pt, reference_host.pt): every crop decodes exactly as the oracle decodes it alone, the run merged
    with both offset signs and trimmed, and a second, shorter run gave the same token prefixes."""
    from oracle.make_golden import trace_crops
    from surya_b200.config import tiny_rec
    from surya_b200.synth import rec_state_dict

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    crops = trace_crops()
    g = torch.load(GOLDEN / "rec_predictor_trace.pt")
    events, tokens, bboxes, scores = g["events"], g["tokens"], g["bboxes"], g["scores"]
    offsets = [e["offset"] for e in events if e["kind"] == "merge"]
    assert any(o > 0 for o in offsets) and any(o < 0 for o in offsets), offsets
    assert any(e["kind"] == "trim" for e in events)
    assert len(tokens) == len(crops)
    for i, crop in enumerate(crops):
        otok, osc, obox, hist = O.greedy_decode(sd, cfg, O.build_batch([crop], cfg), 10, torch.float32, stop_rules=True)
        assert tokens[i] == hist[0], f"crop {i}: {tokens[i]} vs oracle {hist[0]}"
        assert np.allclose(scores[i], osc[0, : len(hist[0])].numpy(), atol=1e-5)
        assert torch.equal(torch.as_tensor(bboxes[i][: len(hist[0])]).long(), obox[0, : len(hist[0])])
    rerun = torch.load(GOLDEN / "reference_host.pt")["rec_rerun"]
    assert rerun["tokens"] == [t[: rerun["max_tokens"]] for t in tokens[: rerun["n_crops"]]]


def test_predictor_trace_replay_cpu():
    """Replay of the committed predictor trace (no reference needed) against B200SuryaModel(OracleRecEngine): same tokens,
    same merge offsets, no slot leaked.  Pins the boundary code on every box; the GPU test replays it on the CUDA engine."""
    from oracle import ref_predictors as RP
    from oracle.make_golden import trace_crops
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import B200SuryaModel
    from surya_b200.synth import rec_state_dict

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    g = torch.load(GOLDEN / "rec_predictor_trace.pt")
    eng = RP.OracleRecEngine(cfg, sd, dtype=torch.float32, max_slots=16)
    model = B200SuryaModel(eng)
    seen = []

    def check(i, ev, out):
        tok = out["lm_logits"][:, -1].float().argmax(-1)
        assert torch.equal(tok, ev["tok"]), f"event {i} ({ev['kind']}): {tok.tolist()} vs {ev['tok'].tolist()}"
        assert (out["bbox_logits"][:, -1].float() - ev["bbox"]).abs().max() < 1e-5
        seen.append(i)

    RP.replay_rec_trace(model, g, trace_crops(), _tile_fn(cfg), check)
    assert len(seen) == sum(e["kind"] in ("prefill", "decode") for e in g["events"])
    assert len(eng.free_slots) == eng.max_slots


def test_slot_cache_contract():
    """merge / trim_left / get_seq_length arithmetic of surya/recognition/cache.py:39-46, 57-105 without any engine math."""
    from surya_b200 import _lib
    from surya_b200.recognition import SlotCache

    class Eng:
        device = torch.device("cpu")

        class cfg:
            class decoder:
                num_hidden_layers = 2
        released = []

        def release_slots(self, s):
            self.released += list(s)

    e = Eng()
    a, b = SlotCache().bind(e), SlotCache(e)
    assert not a and len(a) == 0
    a.assign([0, 1, 2], seq_len=20)
    a.advance(3)
    b.assign([7], seq_len=30)
    assert a and a.get_seq_length() == 23 and len(a) == 2
    off = a.merge(b, [1], "cpu")
    assert off == -7 and a.get_seq_length() == 30 and a._host == [0, 7, 2] and e.released == [1] and not b
    c = SlotCache(e)
    c.assign([9, 8], seq_len=12)
    assert a.merge(c, [0, 2]) == 18 and a.get_seq_length() == 30 and a._host == [9, 7, 8]
    a.trim_left(torch.tensor(11))
    assert a.get_seq_length() == 19
    with pytest.raises(_lib.SuryaB200Error):
        a.merge(object(), [0])
    a.release()
    assert sorted(e.released) == [0, 1, 2, 7, 8, 9] and not a
    del c, b


def test_dropin_install_is_reversible():
    import types

    from surya_b200 import dropin
    from surya_b200.recognition import SlotCache

    mod = types.SimpleNamespace(ContinuousBatchingCache=dict)
    assert dropin.install(mod).ContinuousBatchingCache is SlotCache
    assert dropin.install(mod).ContinuousBatchingCache is SlotCache          # idempotent
    assert dropin.uninstall(mod).ContinuousBatchingCache is dict
    L = dropin.loader_for("m", "p")
    assert L("ckpt").model("cpu", None) == "m" and L().processor() == "p"


def test_reference_detection_predictor_config1_and_dropin_cpu():
    """BASELINE config 1: one 1024x1024 synthetic page (the reference's own conftest page) through the reference
    DetectionPredictor over its own model on CPU (tests/golden/reference_host.pt) against B200EfficientViT over the oracle engine:
    the same segmentation logits (seeded sample) up to fp32 noise, and the same polygons from the product's host stages on the
    heat map upsampled like the predictor does."""
    import torch.nn.functional as F

    from oracle import det_oracle as D
    from oracle import ref_predictors as RP
    from oracle.make_golden import array_digest
    from surya_b200.config import det_default
    from surya_b200.detection import B200EfficientViT, text_boxes_from_front
    from surya_b200.pipeline import page_polygons
    from surya_b200.synth import det_normalize, det_state_dict

    g = torch.load(GOLDEN / "reference_host.pt")["det_config1"]
    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    page = np.asarray(RP.conftest_page(1024), dtype=np.uint8)
    assert array_digest(page) == g["page_digest"], "the conftest page renders differently here"
    assert g["image_bbox"] == [0, 0, 1024, 1024]
    x = det_normalize(page[None])
    logits = B200EfficientViT(RP.OracleDetEngine(cfg, sd))(pixel_values=x).logits.float()
    assert tuple(logits.shape[1:]) == g["logits_shape"]
    assert (logits[0].reshape(logits.shape[1], -1)[:, g["logit_index"]] - g["logits"]).abs().max().item() < 1e-4
    heat = F.interpolate(logits, size=(1024, 1024), mode="bilinear", align_corners=False)[0, 0].numpy()
    tt, low, _ = D.dynamic_thresholds(heat)
    boxes, conf = text_boxes_from_front(heat, (heat > low).astype(np.uint8), float(tt), float(low))
    polys, pconf = page_polygons(boxes, conf, (1024, 1024), (1024, 1024))
    assert [[[float(v) for v in pt] for pt in p] for p in polys] == g["polygons"]
    assert np.allclose(pconf, g["conf"], atol=1e-6)


def test_det_postprocess_oracle_pinned_to_reference():
    """oracle.det_oracle.dynamic_thresholds / detect_boxes and the product's text_boxes_from_front against what the reference's own
    surya.detection.heatmap functions returned on the same synthetic heat maps (smooth blobs of text-line shape; stored in
    tests/golden/reference_host.pt): identical thresholds, boxes and confidences."""
    from oracle import det_oracle as D
    from oracle.make_golden import array_digest, det_postprocess_maps
    from surya_b200.detection import text_boxes_from_front

    golden = torch.load(GOLDEN / "reference_host.pt")["det_boxes"]
    maps = det_postprocess_maps()
    assert len(maps) == len(golden)
    for m, ref in zip(maps, golden):
        assert array_digest(m) == ref["map_digest"], "the synthetic heat map differs from the one the reference saw"
        tt, low, _ = D.dynamic_thresholds(m)
        assert (float(tt), float(low)) == ref["thresholds"]
        ref_boxes, ref_conf = [b.numpy() for b in ref["boxes"]], ref["conf"].numpy()
        boxes, conf = D.detect_boxes(m)
        pboxes, pconf = text_boxes_from_front(m.astype(np.float16), (m > low).astype(np.uint8), float(tt), float(low))
        assert len(ref_boxes) == len(boxes) == len(pboxes) and len(boxes) > 3
        for a, b, c in zip(ref_boxes, boxes, pboxes):
            assert np.array_equal(a, b) and np.array_equal(a, c)
        assert np.allclose(ref_conf, conf, atol=0) and np.allclose(ref_conf, pconf, atol=1e-7)


def test_pipeline_host_stages_pinned_to_reference():
    """surya_b200.pipeline.page_polygons / slice_polygon against what the reference's get_and_clean_boxes + parallel_get_boxes
    expansion (surya/detection/heatmap.py:125-175) and slice_polys_from_image (surya/input/processing.py:57-101) returned on the same
    synthetic heat maps and pages (tests/golden/reference_host.pt; slices compared through sha256 digests of their bytes)."""
    from oracle import det_oracle as D
    from oracle.make_golden import array_digest, pipeline_host_cases
    from surya_b200.detection import text_boxes_from_front
    from surya_b200.pipeline import page_polygons, slice_polygon

    golden = torch.load(GOLDEN / "reference_host.pt")["page_polys"]
    cases = pipeline_host_cases()
    assert len(cases) == len(golden)
    for (m, img_size, page), ref in zip(cases, golden):
        assert array_digest(m) == ref["map_digest"], "the synthetic heat map differs from the one the reference saw"
        H, W = m.shape
        tt, low, _ = D.dynamic_thresholds(m)
        boxes, conf = text_boxes_from_front(m, (m > low).astype(np.uint8), float(tt), float(low))
        polys, pconf = page_polygons(boxes, conf, img_size, (W, H))
        assert len(polys) == len(ref["polygons"]) and len(polys) > 3
        for p, r, c, rc in zip(polys, ref["polygons"], pconf, ref["conf"]):
            assert [[float(v) for v in pt] for pt in p] == r, (p, r)
            assert abs(c - rc) < 1e-6
        assert (page is None) == (ref["slice_digests"] is None)
        if page is not None:
            assert [array_digest(slice_polygon(page, p)) for p in polys] == ref["slice_digests"]
