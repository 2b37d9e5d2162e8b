"""ORACLE TOOLING — generate golden vectors from the reference's own nn.Modules (run in the build container).

    SURYA_REFERENCE=<reference checkout> python -m oracle.make_golden [rec det layout table trace ocr_error host]

The reference (imported unmodified from the SURYA_REFERENCE checkout through oracle/ref_shim.py) is instantiated for a
declared config, loaded with surya_b200.synth's seeded weights, and driven exactly like
RecognitionPredictor.prefill/decode drive it (surya/recognition/__init__.py:326-352, 398-409): one prefill
with a fresh cache, then greedy decode steps feeding process_outputs' input_ids back.  Outputs are stored in
fp32; inputs are regenerated from seeds by the tests, so the fixtures stay small.
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import rec_oracle as O  # noqa: E402
from oracle import ref_shim  # noqa: E402
from surya_b200.config import syn_rec, tiny_rec  # noqa: E402
from surya_b200.synth import rec_state_dict, rec_synthetic_crops  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"


def golden_crops(kind: str):
    """The seeded inputs the goldens are defined on (tests regenerate them with this same function)."""
    if kind == "tiny":
        crops = list(rec_synthetic_crops(3, 48, 512, seed=1234))
        crops.append(rec_synthetic_crops(1, 40, 300, seed=5)[0])    # shorter prompt -> left padding
        crops.append(rec_synthetic_crops(1, 64, 900, seed=6)[0])    # wider crop -> more windows
        return crops
    if kind == "synrec":
        return list(rec_synthetic_crops(2, 48, 512, seed=1234))
    raise ValueError(kind)


def run_reference(cfg, sd, batch, steps: int, attn: str = "sdpa"):
    from transformers import DynamicCache

    model = ref_shim.build_reference_rec_model(cfg, sd, attn=attn)
    ids, mask, pos = batch["input_ids"], batch["attention_mask"], batch["position_ids"]
    lms, bbs = [], []
    with torch.inference_mode():
        cache = DynamicCache()
        out = model(input_ids=ids, image_tiles=batch["image_tiles"], grid_thw=torch.from_numpy(batch["grid_thw"]),
                    attention_mask=mask, position_ids=pos, inputs_embeds=None, past_key_values=cache, use_cache=True,
                    logits_to_keep=1, encoder_chunk_size=4096)
        for step in range(steps):
            lm, bb = out["lm_logits"], out["bbox_logits"]
            lms.append(lm[:, 0].float().clone())
            bbs.append(bb[:, 0].float().clone())
            if step == steps - 1:
                break
            nxt, *_ = O.process_outputs(lm, bb, cfg)
            mask = F.pad(mask, (0, 1), value=1)
            pos = pos[:, -1:] + 1
            out = model(input_ids=nxt, attention_mask=mask, position_ids=pos, use_cache=True, past_key_values=cache,
                        logits_to_keep=1)
    return torch.stack(lms, 1), torch.stack(bbs, 1)


def summarise(lm: torch.Tensor, bb: torch.Tensor, cfg, full_logits: bool):
    tok = lm.argmax(-1)
    top2 = lm.topk(2, dim=-1).values
    g = {
        "tokens": tok,
        "margin": (top2[..., 0] - top2[..., 1]),
        "score": lm.softmax(-1).max(-1).values,
        "logsumexp": lm.logsumexp(-1),
        "bbox": bb,
        "boxes": (bb * cfg.bbox_size).to(torch.long),
        "logit_idx": torch.arange(0, lm.shape[-1], 97),
    }
    g["logit_sample"] = lm[..., g["logit_idx"]].clone()
    g["logit_max"] = lm.max(-1).values
    if full_logits:
        g["logits"] = lm
    return g


def make_layout_golden():
    """Reference Swin encoder + ADETR decoder driven like LayoutPredictor.batch_layout_detection
    (surya/layout/__init__.py:83-137): encoder once, prefill call, greedy box steps."""
    from surya_b200.config import layout_tiny
    from surya_b200.synth import adetr_layout_state_dict, layout_synthetic_pages, swin_state_dict

    cfg = layout_tiny()
    e, d = cfg.encoder, cfg.decoder
    sde, sdd = swin_state_dict(e, 0), adetr_layout_state_dict(d, 0)
    enc, dec = ref_shim.build_reference_layout_models(cfg, sde, sdd)
    x = layout_synthetic_pages(2, e.image_size, seed=7)
    steps = 8
    with torch.inference_mode():
        ref_enc = enc(pixel_values=x)[0]
        dec.model._setup_cache(dec.config, 2, "cpu", torch.float32)
        boxes = torch.full((2, 1, 7), d.bos_token_id, dtype=torch.long)
        pos = torch.arange(1)
        toks, bbs, cls = [], [], []
        for s in range(steps):
            out = dec(input_boxes=boxes, encoder_hidden_states=ref_enc, cache_position=pos, use_cache=True, prefill=(s == 0))
            pos = pos[-1:] + 1
            b, c = out["bbox_logits"][:, -1, :], out["class_logits"][:, -1, :]
            boxes = torch.cat([(b * d.bbox_size).unsqueeze(1), c.argmax(-1).unsqueeze(1).unsqueeze(1)], dim=-1).to(torch.long)
            toks.append(boxes[:, 0].clone())
            bbs.append(b.float().clone())
            cls.append(c.float().clone())
    g = {"encoder": ref_enc.float().clone(), "tokens": torch.stack(toks, 1), "bbox": torch.stack(bbs, 1),
         "class_logits": torch.stack(cls, 1), "input_checksum": x.double().sum(),
         "meta": {"kind": "layout_tiny", "steps": steps, "seed": 0, "page_seed": 7, "torch": str(torch.__version__),
                  "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), fp32 CPU, eager attention"}}
    torch.save(g, GOLDEN / "layout_tiny.pt")
    top2 = g["class_logits"].topk(2, -1).values
    print(f"[golden] layout_tiny: tokens[0,:2]={g['tokens'][0, :2].tolist()} min class margin={(top2[..., 0] - top2[..., 1]).min():.4f}")


def make_table_golden():
    """Reference table_rec encoder + decoder driven like TableRecPredictor.inference_loop (table_rec/__init__.py:33-131):
    3-token query prompt prefill, then greedy steps with the predictor's own token formation."""
    from oracle import layout_oracle as L
    from surya_b200.config import table_tiny
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    cfg = table_tiny()
    e, d = cfg.encoder, cfg.decoder
    sde, sdd = swin_state_dict(e, 1), adetr_table_state_dict(d, 1)
    enc, dec = ref_shim.build_reference_table_models(cfg, sde, sdd)
    x = layout_synthetic_pages(2, e.image_size, seed=9)
    ids = table_query_tokens(d, 2)
    steps = 8
    with torch.inference_mode():
        ref_enc = enc(pixel_values=x).last_hidden_state
        dec.model._setup_cache(dec.config, 2, "cpu", torch.float32)
        pos = torch.ones_like(ids[0, :, 0], dtype=torch.int64).cumsum(0) - 1
        toks, heads = [], []
        for s in range(steps):
            out = dec(input_ids=ids, encoder_hidden_states=ref_enc, cache_position=pos, use_cache=True, prefill=(s == 0))
            pos = pos[-1:] + 1
            logits = out["box_property_logits"]
            tok, done = L.table_next_tokens(logits, d)
            ids = tok.unsqueeze(1)
            toks.append(tok)
            heads.append({k: v[:, -1].float().clone() for k, v in logits.items()})
    g = {"encoder": ref_enc.float().clone(), "tokens": torch.stack(toks, 1),
         "heads": {k: torch.stack([h[k] for h in heads], 1) for k in heads[0]}, "input_checksum": x.double().sum(),
         "meta": {"kind": "table_tiny", "steps": steps, "seed": 1, "page_seed": 9, "torch": str(torch.__version__),
                  "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), fp32 CPU, eager attention"}}
    torch.save(g, GOLDEN / "table_tiny.pt")
    print(f"[golden] table_tiny: tokens[0,:2]={g['tokens'][0, :2].tolist()}")


def make_layout_variants_golden():
    """Extra pins for the oracle only (CPU test): a NON-SQUARE Swin input (256x512: exercises the (W, H) order of the
    sin-cos tables, window partition of unequal sides and the shift masks) and a table_rec CELL-pass prompt (query + 4 column
    boxes, q_len = 7 prefill; table_rec/__init__.py:206-222, processor.py:78-82)."""
    from oracle import layout_oracle as L
    from surya_b200.config import AdetrConfig, LayoutConfig, SwinConfig, table_decoder
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    enc_cfg = SwinConfig(image_size=(256, 512), depths=(2, 2, 2, 2), encoder_length=128)
    cfg = LayoutConfig(encoder=enc_cfg, decoder=table_decoder(2))
    sde, sdd = swin_state_dict(enc_cfg, 3), adetr_table_state_dict(cfg.decoder, 3)
    enc, dec = ref_shim.build_reference_table_models(cfg, sde, sdd)
    x = layout_synthetic_pages(2, enc_cfg.image_size, seed=21)
    d = cfg.decoder
    q = table_query_tokens(d, 2)
    rng = np.random.default_rng(5)
    cols = []
    for _ in range(4):
        b = rng.integers(0, 1025, size=6).tolist()
        cols.append(b + [2 + d.special_token_count, d.special_token_count, 0, d.special_token_count])
    ids = torch.cat([q, torch.tensor(cols, dtype=torch.long).unsqueeze(0).repeat(2, 1, 1)], dim=1)     # [2, 7, 10]
    steps = 5
    with torch.inference_mode():
        ref_enc = enc(pixel_values=x).last_hidden_state
        dec.model._setup_cache(dec.config, 2, "cpu", torch.float32)
        pos = torch.ones_like(ids[0, :, 0], dtype=torch.int64).cumsum(0) - 1
        cur, toks, heads = ids, [], []
        for s in range(steps):
            out = dec(input_ids=cur, encoder_hidden_states=ref_enc, cache_position=pos, use_cache=True, prefill=(s == 0))
            pos = pos[-1:] + 1
            logits = out["box_property_logits"]
            tok, _ = L.table_next_tokens(logits, d)
            cur = tok.unsqueeze(1)
            toks.append(tok)
            heads.append({k: v[:, -1].float().clone() for k, v in logits.items()})
    # a seeded sample of the 2 x 128 encoder rows keeps the fixture small; the decoder heads depend on all of them
    rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(2 * 128, size=16, replace=False)))
    g = {"encoder_rows": rows, "encoder": ref_enc.float().reshape(2 * 128, -1)[rows].clone(), "encoder_shape": tuple(ref_enc.shape),
         "prompt": ids, "tokens": torch.stack(toks, 1), "heads": {k: torch.stack([h[k] for h in heads], 1) for k in heads[0]},
         "meta": {"kind": "table_nonsquare_cellpass", "steps": steps, "seed": 3, "page_seed": 21, "image_size": [256, 512],
                  "torch": str(torch.__version__), "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), fp32 CPU"}}
    torch.save(g, GOLDEN / "table_nonsquare_cellpass.pt")
    print(f"[golden] table_nonsquare_cellpass: enc {tuple(ref_enc.shape)} tokens[0,0]={g['tokens'][0, 0].tolist()}")


def make_det_golden():
    """Reference EfficientViT segmentation logits for one seeded 512x512 page (surya/detection/__init__.py:94-104)."""
    from surya_b200.config import det_default
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    m = ref_shim.build_reference_det_model(cfg, sd)
    x = det_normalize(det_synthetic_pages(1, 512, seed=11, text_like=True))
    with torch.inference_mode():
        logits = m(pixel_values=x).logits.float()
        logits16 = m.half()(pixel_values=x.half()).logits.float()    # the reference's own fp16 path (settings MODEL_DTYPE on GPU)
    g = {"logits": logits, "logits_fp16_path": logits16, "input_checksum": x.double().sum(),
         "meta": {"reference": "VikParuchuri/surya@80e9a7e EfficientViTForSemanticSegmentation, CPU; fp32 and model.half() runs",
                  "size": 512, "seed": 11}}
    torch.save(g, GOLDEN / "det_default.pt")
    print(f"[golden] det_default: logits {tuple(logits.shape)} max={logits.max():.4f}")


def trace_crops():
    """Seeded crops of mixed widths for the predictor-trace golden: prompts of different lengths (left padding, merge offsets of
    both signs) through 3 batch rows."""
    widths = [512, 300, 700, 256, 900, 380, 620]
    return [rec_synthetic_crops(1, 48, w, seed=200 + i)[0] for i, w in enumerate(widths)]


def make_predictor_trace_golden():
    """The reference's UNMODIFIED RecognitionPredictor.prediction_loop (prefill / decode / merge / maybe_trim_cache_padding,
    surya/recognition/__init__.py:326-607) run over B200SuryaModel + SlotCache with the CPU oracle as the engine
    (oracle/ref_predictors.py); every model call and cache operation is logged so the GPU test can replay the exact sequence
    against the CUDA engine.  fp32, tiny config, 7 crops through 3 rows, max_tokens 10, trim threshold lowered to 2."""
    from oracle import ref_predictors as RP

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    t0 = time.time()
    events, tokens, bboxes, scores, eng = RP.record_rec_trace(cfg, sd, trace_crops(), batch_size=3, max_tokens=10,
                                                              min_trim_length=2)
    assert len(eng.free_slots) == eng.max_slots, "the predictor run leaked KV slots"
    g = {"events": events, "tokens": tokens, "scores": scores, "bboxes": bboxes,
         "meta": {"kind": "rec_predictor_trace", "batch_size": 3, "max_tokens": 10, "min_trim_length": 2, "seed": 0,
                  "torch": str(torch.__version__), "reference": "VikParuchuri/surya@80e9a7e RecognitionPredictor.prediction_loop, fp32 CPU"}}
    torch.save(g, GOLDEN / "rec_predictor_trace.pt")
    kinds = [e["kind"] for e in events]
    print(f"[golden] rec_predictor_trace: {time.time() - t0:.1f}s {len(events)} events "
          f"({kinds.count('prefill')} prefill, {kinds.count('decode')} decode, merges "
          f"{[(e['idxs'], e['offset']) for e in events if e['kind'] == 'merge']}, trims {[e['n'] for e in events if e['kind'] == 'trim']}) "
          f"tokens[0]={tokens[0]}")


def preproc_crops():
    """Seeded uint8 crops for the crop-chain pin against the reference's SuryaOCRProcessor."""
    rng = np.random.default_rng(11)
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            for h, w in ((48, 512), (40, 300), (300, 2000), (20, 60), (56, 560), (97, 1403))]


def det_postprocess_maps():
    """Synthetic 512x640 heat maps of text-line-shaped blobs, 16-bit valued like the engine's maps (3 trials)."""
    import cv2

    rng = np.random.default_rng(5)
    maps = []
    for _ in range(3):
        m = np.zeros((512, 640), np.float32)
        for _ in range(25):
            x, y = int(rng.integers(0, 560)), int(rng.integers(0, 480))
            w, h = int(rng.integers(30, 200)), int(rng.integers(6, 24))
            m[y:y + h, x:x + w] = rng.uniform(0.3, 1.0)
        maps.append(cv2.GaussianBlur(m, (0, 0), 2.0).astype(np.float16).astype(np.float32))
    return maps


def pipeline_host_cases():
    """(heat map, image size, page or None) for the page-polygon / polygon-slice pin: trial 1 is rescaled to twice the map size
    and has no page; the others slice a random float32 page."""
    import cv2

    rng = np.random.default_rng(9)
    H, W = 512, 640
    cases = []
    for trial in range(3):
        m = np.zeros((H, W), np.float32)
        for _ in range(20):
            x, y = int(rng.integers(0, W - 60)), int(rng.integers(0, H - 30))
            w, h = int(rng.integers(30, 220)), int(rng.integers(6, 30))
            m[y:y + h, x:x + w] = rng.uniform(0.3, 1.0)
        m[40:60, 100:300] = 0.9
        m[44:56, 150:250] = 0.95                                   # a box contained in another one
        m = cv2.GaussianBlur(m, (0, 0), 1.5).astype(np.float16).astype(np.float32)
        img_size = (W * 2, H * 2) if trial == 1 else (W, H)
        page = rng.integers(0, 256, size=(H, W, 3)).astype(np.float32) if trial != 1 else None
        cases.append((m, img_size, page))
    return cases


def ocr_error_texts():
    """Seeded word strings for the OCRErrorPredictor pin (8 texts of 2..29 words)."""
    rng = np.random.default_rng(0)
    words = [f"w{i}" for i in range(300)]
    return [" ".join(rng.choice(words, size=int(rng.integers(2, 30)))) for _ in range(8)]


def array_digest(a) -> str:
    """sha256 of an array's dtype, shape and bytes: exact equality of large outputs without storing them."""
    import hashlib

    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype}{a.shape}".encode() + a.tobytes()).hexdigest()


def make_reference_host_golden():
    """What the reference's own host code and predictor classes return on seeded inputs, so that the oracle restatements and the
    product's host stages stay pinned to the reference without the reference installed:
      crop_chain   SuryaOCRProcessor.scale_to_fit + _process_and_tile (grids, per-row sums and sums of squares, a seeded sample
                   of tile rows)
      det_boxes    surya.detection.heatmap get_dynamic_thresholds / detect_boxes
      page_polys   get_and_clean_boxes + the predictor's box expansion, and slice_polys_from_image (digests of the slices)
      det_config1  DetectionPredictor over the reference EfficientViT on the reference's own 1024x1024 test page (BASELINE
                   config 1): polygons, confidences and a seeded sample of the segmentation logits
      ocr_error    OCRErrorPredictor over the reference DistilBERT: labels of 8 texts, batches of 3
      rec_rerun    tokens of a second, shorter RecognitionPredictor run over the predictor-trace crops (see
                   make_predictor_trace_golden)
    """
    from oracle import ocr_error_oracle as E
    from oracle import ref_predictors as RP
    from surya_b200 import dropin
    from surya_b200.config import det_default, ocr_error_tiny
    from surya_b200.synth import det_normalize, det_state_dict, ocr_error_state_dict

    RP.install_predictors()
    from surya.detection import DetectionPredictor
    from surya.detection.heatmap import detect_boxes, get_and_clean_boxes, get_dynamic_thresholds
    from surya.input.processing import slice_polys_from_image
    from surya.settings import settings

    g = {"meta": {"kind": "reference_host", "torch": str(torch.__version__),
                  "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), CPU"}}
    cfg = tiny_rec()
    proc = RP.synthetic_ocr_processor(cfg)
    sample = np.random.default_rng(0)
    g["crop_chain"] = []
    for crop in preproc_crops():
        tiles, grid = proc._process_and_tile(proc.scale_to_fit(np.asarray(crop, dtype=np.float32), (1024, 256)))
        tiles = tiles.numpy()
        rows = np.sort(sample.choice(tiles.shape[0], size=min(4, tiles.shape[0]), replace=False))
        g["crop_chain"].append({"shape": tuple(crop.shape), "grid": tuple(int(v) for v in grid), "rows": torch.from_numpy(rows),
                                "tile_rows": torch.from_numpy(tiles[rows].copy()),
                                "row_sums": torch.from_numpy(tiles.astype(np.float64).sum(1)),
                                "row_sq": torch.from_numpy((tiles.astype(np.float64) ** 2).sum(1))})

    g["det_boxes"] = []
    for m in det_postprocess_maps():
        tt, low = get_dynamic_thresholds(m, 0.6, 0.35)
        boxes, conf = detect_boxes(m, 0.6, 0.35)
        g["det_boxes"].append({"map_digest": array_digest(m), "thresholds": (float(tt), float(low)),
                               "boxes": [torch.from_numpy(np.array(b)) for b in boxes],
                               "conf": torch.from_numpy(np.asarray(conf, dtype=np.float64))})

    g["page_polys"] = []
    for m, img_size, page in pipeline_host_cases():
        H, W = m.shape
        ref = get_and_clean_boxes(m, [W, H], img_size)
        for box in ref:
            if box.height < 3 * box.width:
                box.expand(x_margin=0, y_margin=settings.DETECTOR_BOX_Y_EXPAND_MARGIN)
                box.fit_to_bounds([0, 0, img_size[0], img_size[1]])
        polys = [[[float(v) for v in pt] for pt in r.polygon] for r in ref]
        slices = None
        if page is not None:
            slices = [array_digest(s) for s in slice_polys_from_image(page, [[[int(v) for v in pt] for pt in p] for p in polys])]
        g["page_polys"].append({"map_digest": array_digest(m), "polygons": polys, "conf": [float(r.confidence) for r in ref],
                                "slice_digests": slices})

    dcfg = det_default()
    dsd = det_state_dict(dcfg, seed=0)
    dmodel = ref_shim.build_reference_det_model(dcfg, dsd)
    dproc = RP.synthetic_det_processor(1024)
    page = RP.conftest_page(1024)
    stock = type("StockDetectionPredictor", (DetectionPredictor,), {"model_loader_cls": dropin.loader_for(dmodel, dproc)})(
        device="cpu", dtype=torch.float32)
    stock.disable_tqdm = True
    res = stock([page])[0]
    x = torch.from_numpy(dproc(np.asarray(page, dtype=np.uint8))["pixel_values"][0])[None]
    assert (x - det_normalize(np.asarray(page, dtype=np.uint8)[None])).abs().max().item() < 1e-6
    with torch.inference_mode():
        logits = dmodel(pixel_values=x).logits.float()[0]
    idx = torch.from_numpy(np.sort(sample.choice(logits[0].numel(), size=4096, replace=False)).astype(np.int32))
    g["det_config1"] = {"page_digest": array_digest(np.asarray(page, dtype=np.uint8)), "image_bbox": list(res.image_bbox),
                        "polygons": [[[float(v) for v in pt] for pt in b.polygon] for b in res.bboxes],
                        "conf": [float(b.confidence) for b in res.bboxes], "logit_index": idx,
                        "logits": logits.reshape(logits.shape[0], -1)[:, idx].clone(), "logits_shape": tuple(logits.shape)}

    ecfg = ocr_error_tiny()
    emodel = ref_shim.build_reference_ocr_error_model(ecfg, ocr_error_state_dict(ecfg, seed=0))
    from surya.ocr_error import OCRErrorPredictor      # after install() has re-applied the tokenizer-helper names

    texts = ocr_error_texts()
    stock = type("StockOCRErrorPredictor", (OCRErrorPredictor,), {"model_loader_cls": dropin.loader_for(emodel, E.HashTokenizer(ecfg))})(
        device="cpu", dtype=torch.float32)
    stock.disable_tqdm = True
    g["ocr_error"] = {"texts": texts, "batch_size": 3, "labels": list(stock(texts, batch_size=3).labels)}
    _, rerun, *_ = RP.record_rec_trace(cfg, rec_state_dict(cfg, seed=0), trace_crops()[:4], batch_size=3, max_tokens=4)
    g["rec_rerun"] = {"n_crops": 4, "batch_size": 3, "max_tokens": 4, "tokens": rerun}
    torch.save(g, GOLDEN / "reference_host.pt")
    print(f"[golden] reference_host: {len(g['det_config1']['polygons'])} config-1 polygons, ocr_error labels {g['ocr_error']['labels']}")


def make_swin_window_padding_golden():
    """Oracle pin for DonutSwinLayer.maybe_pad (donut/encoder.py:591-596, crop :657-659): a 288x352 input gives token grids
    72x88 / 36x44 / 18x22 / 9x11 -- every merge sees even sides (the reference's floor-sized stage position tables demand it) but
    stages 1-3 are not multiples of the 8x8 window, so their layers run on zero-padded grids with the shift mask of the padded
    size.  Encoder output only (1 page)."""
    from surya_b200.config import LayoutConfig, SwinConfig, table_decoder
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict

    enc_cfg = SwinConfig(image_size=(288, 352), depths=(2, 2, 2, 2), encoder_length=99)
    cfg = LayoutConfig(encoder=enc_cfg, decoder=table_decoder(2))
    sde, sdd = swin_state_dict(enc_cfg, 5), adetr_table_state_dict(cfg.decoder, 5)
    enc, _ = ref_shim.build_reference_table_models(cfg, sde, sdd)
    x = layout_synthetic_pages(1, enc_cfg.image_size, seed=23)
    with torch.inference_mode():
        ref_enc = enc(pixel_values=x).last_hidden_state
    g = {"encoder": ref_enc.float().clone(), "input_checksum": x.double().sum(),
         "meta": {"kind": "swin_window_padding", "seed": 5, "page_seed": 23, "image_size": [288, 352], "torch": str(torch.__version__),
                  "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), fp32 CPU"}}
    torch.save(g, GOLDEN / "swin_window_padding.pt")
    print(f"[golden] swin_window_padding: enc {tuple(ref_enc.shape)} absmax {ref_enc.abs().max():.3f}")


def make_ocr_error_golden():
    """Reference DistilBertForSequenceClassification (surya/ocr_error/model/encoder.py:697-766, eager attention, fp32 CPU) on seeded
    right-padded batches: logits, [CLS] hidden state and the predictor's argmax labels (surya/ocr_error/__init__.py:55-57)."""
    from surya_b200.config import ocr_error_default, ocr_error_tiny
    from surya_b200.synth import ocr_error_state_dict, ocr_error_synthetic_batch

    for kind, cfg, n, max_len, seed in (("tiny", ocr_error_tiny(), 12, 40, 3), ("default", ocr_error_default(), 16, 96, 3)):
        sd = ocr_error_state_dict(cfg, seed=0)
        m = ref_shim.build_reference_ocr_error_model(cfg, sd)
        ids, mask = ocr_error_synthetic_batch(cfg, n, max_len, seed=seed)
        with torch.inference_mode():
            logits = m(ids, attention_mask=mask).logits.float()
            hidden = m.distilbert(ids, attention_mask=mask)[0].float()
        g = {"input_ids": ids, "attention_mask": mask, "logits": logits, "cls_hidden": hidden[:, 0].clone(), "labels": logits.argmax(1),
             "meta": {"reference": "VikParuchuri/surya@80e9a7e DistilBertForSequenceClassification, eager attention, fp32 CPU",
                      "n": n, "max_len": max_len, "seed": seed, "kind": kind}}
        torch.save(g, GOLDEN / f"ocr_error_{kind}.pt")
        print(f"[golden] ocr_error_{kind}: logits {tuple(logits.shape)} labels={g['labels'].tolist()}")


def main():
    GOLDEN.mkdir(parents=True, exist_ok=True)
    torch.set_num_threads(8)
    which = set(sys.argv[1:]) or {"rec", "det", "layout", "table", "trace", "ocr_error", "host"}
    if "layout" in which:
        make_layout_golden()
    if "table" in which:
        make_table_golden()
        make_layout_variants_golden()
        make_swin_window_padding_golden()
    if "det" in which:
        make_det_golden()
    if "trace" in which:
        make_predictor_trace_golden()
    if "ocr_error" in which:
        make_ocr_error_golden()
    if "host" in which:
        make_reference_host_golden()
    if "rec" not in which:
        return
    for kind, cfg, steps in (("tiny", tiny_rec(), 32), ("synrec", syn_rec(), 40)):
        t0 = time.time()
        sd = rec_state_dict(cfg, seed=0)
        batch = O.build_batch(golden_crops(kind), cfg)
        lm, bb = run_reference(cfg, sd, batch, steps)
        g = summarise(lm, bb, cfg, full_logits=(kind == "tiny"))
        g["meta"] = {"kind": kind, "steps": steps, "seed": 0, "torch": str(torch.__version__),
                     "reference": "VikParuchuri/surya@80e9a7e (v0.14.6), fp32 CPU, attn=sdpa",
                     "input_ids_shape": list(batch["input_ids"].shape), "n_tiles": int(batch["image_tiles"].shape[0])}
        g["input_ids"] = batch["input_ids"]
        g["grid_thw"] = torch.from_numpy(batch["grid_thw"])
        g["tiles_checksum"] = batch["image_tiles"].double().sum()
        torch.save(g, GOLDEN / f"rec_{kind}.pt")
        print(f"[golden] {kind}: {time.time() - t0:.1f}s tokens={g['tokens'].tolist()} min margin={g['margin'].min():.4f}")


if __name__ == "__main__":
    main()
