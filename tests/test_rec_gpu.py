"""Recognition path parity (GPU): CUDA engine through the C ABI vs the CPU oracle and the committed goldens
(goldens = outputs of the reference's own nn.Modules, see oracle/make_golden.py).

Tolerances (north star: logits within 1e-3 fp16 atol, token ids exact):
  * 1e-3 is one fp16 ulp at 1.0; logits here reach |7|.  A 12-layer 16-bit pipeline cannot sit inside one ulp of an fp32
    path — the reference's OWN 16-bit path does not: every test measures that gap in the same run (`ref_gap` = the oracle,
    i.e. the reference algorithm, evaluated in the engine's dtype vs the fp32 golden; 4e-3 .. 9e-3 in fp16, 3e-2 .. 8e-2
    in bf16 on these weights) and requires   engine error vs fp32 golden  <=  max(floor, 1.5 x ref_gap)
    with floor 6e-3 (fp16) / 6e-2 (bf16): the engine may not be worse than the reference's own half-precision path.
  * engine vs oracle evaluated in the SAME dtype: fp16 <= 8e-3, bf16 <= 8e-2 (two 16-bit pipelines with different — both
    legal — rounding points; since round 2 the decoder RMSNorms are folded into the following GEMM, DESIGN.md §4).
  * token ids: exact wherever the reference's top-2 logit margin exceeds 4x the logit tolerance; every divergence is
    required to sit on such a near-tie (teacher forcing keeps later steps comparable).  Measured values are written to
    gpurun_out/rec_parity.json.
"""
import json
import os
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import rec_oracle as O

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
OUT = ROOT / "gpurun_out"

TOL_SAME = {torch.float16: 8e-3, torch.bfloat16: 8e-2}
TOL_GOLD = {torch.float16: 6e-3, torch.bfloat16: 6e-2}


def _report(name, payload):
    OUT.mkdir(exist_ok=True)
    path = OUT / "rec_parity.json"
    data = json.loads(path.read_text()) if path.exists() else {}
    data[name] = payload
    path.write_text(json.dumps(data, indent=1))


def _golden_crops(kind):
    from oracle.make_golden import golden_crops

    return golden_crops(kind)


def _engine(cfg, sd, dtype, **kw):
    from surya_b200.recognition import RecEngine

    return RecEngine(cfg, sd, dtype=dtype, **kw)


def _prefill_ragged(eng, cfg, batch, want_logits=True):
    from surya_b200.recognition import build_prefill_plan

    ids, mask = batch["input_ids"].numpy(), batch["attention_mask"].numpy().astype(bool)
    seqs = [ids[b][mask[b]] for b in range(ids.shape[0])]
    slots = eng.alloc_slots(len(seqs))
    plan = build_prefill_plan(cfg, batch["grid_thw"], seqs, slots)
    out = eng.prefill(batch["image_tiles"].cuda(), plan, want_logits=want_logits)
    return out, slots, [len(s) for s in seqs]


def _teacher_forced(eng, cfg, batch, forced, steps):
    """prefill + decode steps feeding `forced` tokens; returns logits [B, steps, V] fp32, tokens, boxes."""
    out, slots, lens = _prefill_ragged(eng, cfg, batch)
    slot_t = torch.tensor(slots, dtype=torch.int32, device="cuda")
    pos = torch.tensor(lens, dtype=torch.int32, device="cuda")
    logits, toks, boxes, scores = [out["logits"].float().cpu()], [out["tok"].cpu()], [out["bbox"].cpu()], [out["score"].cpu()]
    for s in range(steps - 1):
        nxt = forced[:, s].clone()
        nxt[(nxt == cfg.eos_token_id) | (nxt == cfg.pad_token_id)] = cfg.pad_token_id
        o = eng.decode(nxt.cuda(), slot_t, pos, want_logits=True)
        pos = pos + 1
        logits.append(o["logits"].float().cpu())
        toks.append(o["tok"].cpu())
        boxes.append(o["bbox"].cpu())
        scores.append(o["score"].cpu())
    eng.release_slots(slots)
    return torch.stack(logits, 1), torch.stack(toks, 1), torch.stack(boxes, 1), torch.stack(scores, 1)


def _tol(dtype, ref_gap):
    return max(TOL_GOLD[dtype], 1.5 * ref_gap)


def _check_tokens(tok, ref_tok, ref_margin, tol, what):
    diff = tok != ref_tok
    if diff.any():
        bad = diff & (ref_margin > 4 * tol)
        assert not bad.any(), f"{what}: token mismatch away from a near-tie: {tok[bad].tolist()} vs {ref_tok[bad].tolist()}"
    return int(diff.sum())


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tiny_vs_golden_and_oracle(built_lib, dtype):
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.synth import rec_state_dict

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    g = torch.load(GOLDEN / "rec_tiny.pt")
    steps = g["meta"]["steps"]
    batch = O.build_batch(_golden_crops("tiny"), cfg)
    assert torch.equal(batch["input_ids"], g["input_ids"])
    eng = _engine(cfg, sd, dtype, max_slots=16, s_max=256, max_patches=4096, max_tokens=1024)
    logits, tok, boxes, scores = _teacher_forced(eng, cfg, batch, g["tokens"], steps)
    # the reference algorithm in the engine's dtype (oracle), same forced tokens: its gap to the fp32 golden is the yardstick
    sdt = O.cast_sd(sd, dtype)
    otok, osc, obox, ologits = O.greedy_decode(sdt, cfg, batch, steps, dtype, forced_tokens=g["tokens"], return_logits=True)
    ref_gap = (ologits - g["logits"]).abs().max().item()
    tol = _tol(dtype, ref_gap)
    # (a) vs golden (reference modules, fp32)
    err_g = (logits - g["logits"]).abs().max().item()
    n_flip = _check_tokens(tok, g["tokens"], g["margin"], tol, "tiny/golden")
    box_err = (boxes - g["boxes"]).abs().max().item()
    ref_box_gap = (obox - g["boxes"]).abs().max().item()
    # (b) vs oracle in the same dtype
    err_o = (logits - ologits).abs().max().item()
    _report(f"tiny_{str(dtype).split('.')[-1]}", {"max_abs_err_vs_reference_fp32": err_g, "reference_own_16bit_gap": ref_gap,
                                                   "max_abs_err_vs_oracle_same_dtype": err_o, "tolerance_used": tol,
                                                   "token_flips_vs_reference": n_flip, "of_tokens": int(tok.numel()),
                                                   "max_box_err": box_err, "reference_own_box_gap": ref_box_gap,
                                                   "logit_absmax": g["logits"].abs().max().item()})
    assert err_g <= tol, f"logits vs reference golden: {err_g} (reference's own {dtype} gap {ref_gap})"
    assert err_o <= TOL_SAME[dtype], f"logits vs same-dtype oracle: {err_o}"
    assert box_err <= max(2 if dtype == torch.float16 else 12, 2 * ref_box_gap)
    eng.close()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_synrec_vs_golden(built_lib, dtype):
    """Declared SYN-REC config (BASELINE config 2 shapes), 2 crops x 40 steps (80 distinct token ids) teacher-forced against
    the golden produced by the reference's own SuryaModel."""
    from oracle import rec_oracle as O
    from surya_b200.config import syn_rec
    from surya_b200.synth import rec_state_dict

    cfg = syn_rec()
    sd = rec_state_dict(cfg, seed=0)
    g = torch.load(GOLDEN / "rec_synrec.pt")
    steps = g["meta"]["steps"]
    batch = O.build_batch(_golden_crops("synrec"), cfg)
    assert abs(batch["image_tiles"].double().sum().item() - g["tiles_checksum"].item()) < 1e-6
    eng = _engine(cfg, sd, dtype, max_slots=8, s_max=256, max_patches=1024, max_tokens=512)
    logits, tok, boxes, scores = _teacher_forced(eng, cfg, batch, g["tokens"], steps)
    idx = g["logit_idx"]
    err = (logits[..., idx] - g["logit_sample"]).abs().max().item()
    err_max = (logits.max(-1).values - g["logit_max"]).abs().max().item()
    lse = (logits.logsumexp(-1) - g["logsumexp"]).abs().max().item()
    # yardstick: the reference algorithm in this dtype (oracle on the host), first 12 of the 40 steps
    k = 12
    torch.set_num_threads(max(1, min(64, len(os.sched_getaffinity(0)))))
    _, _, _, ologits = O.greedy_decode(O.cast_sd(sd, dtype), cfg, batch, k, dtype, forced_tokens=g["tokens"], return_logits=True)
    ref_gap = (ologits[..., idx] - g["logit_sample"][:, :k]).abs().max().item()
    tol = _tol(dtype, ref_gap)
    n_flip = _check_tokens(tok, g["tokens"], g["margin"], tol, "synrec/golden")
    score_err = (scores - g["score"]).abs().max().item()
    _report(f"synrec_{str(dtype).split('.')[-1]}", {"max_abs_err_logit_sample": err, "max_abs_err_logit_max": err_max,
                                                     "reference_own_16bit_gap_first12": ref_gap, "tolerance_used": tol,
                                                     "logsumexp_err": lse, "token_flips": n_flip, "of_tokens": int(tok.numel()),
                                                     "score_err": score_err, "min_margin": g["margin"].min().item(),
                                                     "distinct_tokens": len(set(g["tokens"].flatten().tolist()))})
    assert err <= tol and err_max <= tol, f"{err} / {err_max} vs tol {tol} (reference's own gap {ref_gap})"
    assert lse <= tol
    eng.close()


def test_model_surface_left_padded(built_lib):
    """B200SuryaModel called exactly like RecognitionPredictor.prefill/decode call self.model (left-padded ids,
    attention_mask, position_ids, caller-owned cache) vs the oracle on the same padded batch."""
    import torch.nn.functional as F

    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import B200SuryaModel
    from surya_b200.synth import rec_state_dict

    dtype = torch.float16
    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    batch = O.build_batch(_golden_crops("tiny"), cfg)
    eng = _engine(cfg, sd, dtype, max_slots=16, s_max=256, max_patches=4096, max_tokens=1024)
    model = B200SuryaModel(eng)
    cache = model.new_cache()
    dev = "cuda"
    ids, mask, pos = batch["input_ids"].to(dev), batch["attention_mask"].to(dev), batch["position_ids"].to(dev)
    out = model(input_ids=ids, image_tiles=batch["image_tiles"].to(dev, dtype), grid_thw=torch.from_numpy(batch["grid_thw"]).to(dev),
                attention_mask=mask, position_ids=pos, inputs_embeds=None, past_key_values=cache, use_cache=True,
                logits_to_keep=1, encoder_chunk_size=32768)
    sdt = O.cast_sd(sd, dtype)
    oc = O.OracleCache()
    with torch.inference_mode():
        lm, bb = O.model_forward(sdt, cfg, batch["input_ids"], batch["attention_mask"], batch["position_ids"], oc,
                                 batch["image_tiles"].to(dtype), batch["grid_thw"])
    assert out["lm_logits"].shape == lm.shape and out["bbox_logits"].shape == bb.shape
    assert (out["lm_logits"].float().cpu() - lm.float()).abs().max().item() <= TOL_SAME[dtype]
    assert (out["bbox_logits"].float().cpu() - bb.float()).abs().max().item() <= 2e-3
    # three decode steps driven the way RecognitionPredictor.decode drives them
    o_ids, *_ = O.process_outputs(lm, bb, cfg)
    o_mask, o_pos = batch["attention_mask"], batch["position_ids"]
    for _ in range(3):
        o_mask = F.pad(o_mask, (0, 1), value=1)
        o_pos = o_pos[:, -1:] + 1
        with torch.inference_mode():
            lm, bb = O.model_forward(sdt, cfg, o_ids, o_mask, o_pos, oc)
        out = model(input_ids=o_ids.to(dev), attention_mask=o_mask.to(dev), position_ids=o_pos.to(dev), use_cache=True,
                    past_key_values=cache, logits_to_keep=1)
        assert (out["lm_logits"].float().cpu() - lm.float()).abs().max().item() <= TOL_SAME[dtype]
        o_ids, *_ = O.process_outputs(lm, bb, cfg)
    cache.release()
    eng.close()


def test_runner_continuous_batching_matches_oracle(built_lib):
    """RecognitionRunner (slots, prefill-when-20%-free, stop rules, device-side multi-step decode) returns, for
    every crop, what the oracle's single-batch greedy loop returns (rows are independent of co-tenants)."""
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    dtype = torch.float16
    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    crops = [rec_synthetic_crops(1, 48, 256 + 37 * i, seed=100 + i)[0] for i in range(11)]
    eng = _engine(cfg, sd, dtype, max_slots=8, s_max=256, max_patches=4096, max_tokens=1024)
    steps = 24
    runner = RecognitionRunner(eng, batch_size=4, max_tokens=steps, poll=5)
    tokens, scores, bboxes = runner.run(crops)
    runner_nograph = RecognitionRunner(eng, batch_size=3, max_tokens=steps, poll=1)
    tokens2, _, _ = runner_nograph.run(crops)
    assert tokens == tokens2, "results must not depend on batch size / polling interval"
    sdt = O.cast_sd(sd, dtype)
    flips = 0
    for i, crop in enumerate(crops):
        batch = O.build_batch([crop], cfg)
        otok, osc, obox, hist, ologits = O.greedy_decode(sdt, cfg, batch, steps, dtype, stop_rules=True, return_logits=True)
        ref = hist[0]
        if tokens[i] != ref:
            # accept only a divergence that starts on a near-tie of the oracle
            k = next(j for j in range(min(len(ref), len(tokens[i]))) if tokens[i][j] != ref[j])
            top2 = ologits[0, k].topk(2).values
            assert (top2[0] - top2[1]).item() <= 4 * TOL_SAME[dtype], f"crop {i} diverges at step {k} without a tie"
            flips += 1
        else:
            assert np.allclose(scores[i], osc[0, : len(ref)].numpy(), atol=2e-2)
    _report("runner_tiny_fp16", {"crops": len(crops), "tie_divergences": flips})
    assert flips <= 2
    eng.close()


def test_fullsize_properties_synrec(built_lib):
    """BASELINE config-2 sizes (B=256, 46-token prompts, bf16): size-independent properties instead of a CPU
    oracle run — replica invariance (identical crops in different rows/slots give identical ids and scores),
    CUDA-graph replay == eager launches, and the teacher-forced first step equals a fresh prefill."""
    from surya_b200.config import syn_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    cfg = syn_rec()
    sd = rec_state_dict(cfg, seed=0)
    eng = _engine(cfg, sd, torch.bfloat16, max_slots=260, s_max=256, max_patches=256 * 160, max_tokens=256 * 46)
    base = rec_synthetic_crops(8, 48, 512, seed=1234)
    crops = [base[i % 8] for i in range(256)]
    runner = RecognitionRunner(eng, batch_size=256, max_tokens=16)
    tiles, grids, seqs = runner.preprocess(crops)
    assert tiles[0].shape == (160, 588) and grids[0] == (1, 4, 40) and len(seqs[0]) == 46
    tokens, scores, bboxes = runner.run_preprocessed(tiles, grids, seqs, fixed_steps=True)
    for i in range(8, 256):
        assert tokens[i] == tokens[i % 8], f"row {i} differs from its replica"
        assert np.array_equal(bboxes[i], bboxes[i % 8])
        assert np.allclose(scores[i], scores[i % 8], rtol=0, atol=0)
    # graph replay vs eager launches
    import surya_b200.recognition as R

    orig = R.RecEngine.decode_steps

    def eager(self, ids_io, slot, pos_io, n_steps, hist=None, use_graph=True, max_pos=None):
        return orig(self, ids_io, slot, pos_io, n_steps, hist, use_graph=False, max_pos=max_pos)

    R.RecEngine.decode_steps = eager
    try:
        tokens_e, scores_e, _ = runner.run_preprocessed(tiles, grids, seqs, fixed_steps=True)
    finally:
        R.RecEngine.decode_steps = orig
    assert tokens_e == tokens
    assert scores_e == scores
    eng.close()


def test_synrec_fullsize_vs_oracle(built_lib):
    """BASELINE config 2 at full length against the CPU oracle (VERDICT r1 weak #2): SYN-REC, bf16, 8 distinct 48x512 crops,
    128 greedy tokens.  (a) teacher-forced with the oracle's tokens: every step's logits inside the bf16 envelope, token ids
    equal wherever the oracle's top-2 margin exceeds 4x that envelope, boxes within 12/1024;  (b) free-running through the
    device-side decode loop at B = 256 (the 8 crops replicated 32x): each row follows the oracle until a step whose oracle
    margin is a near-tie, and replicas are bit-identical.  Flip statistics are written to gpurun_out/rec_parity.json."""
    from oracle import rec_oracle as O
    from surya_b200.config import syn_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    dtype, steps = torch.bfloat16, 128
    cfg = syn_rec()
    sd = rec_state_dict(cfg, seed=0)
    base = list(rec_synthetic_crops(8, 48, 512, seed=1234))
    batch = O.build_batch(base, cfg)
    torch.set_num_threads(max(1, min(64, len(os.sched_getaffinity(0)))))
    otok, osc, obox, ologits = O.greedy_decode(sd, cfg, batch, steps, torch.float32, return_logits=True)
    top2 = ologits.topk(2, -1).values
    margin = top2[..., 0] - top2[..., 1]
    eng = _engine(cfg, sd, dtype, max_slots=260, s_max=256, max_patches=256 * 160, max_tokens=256 * 46)
    # yardstick: the reference algorithm in bf16 on two of the crops, all 128 steps, same forced tokens
    b2 = O.build_batch(base[:2], cfg)
    _, _, rbox, rlogits = O.greedy_decode(O.cast_sd(sd, dtype), cfg, b2, steps, dtype, forced_tokens=otok[:2], return_logits=True)
    ref_gap = (rlogits - ologits[:2]).abs().max().item()
    ref_box_gap = (rbox - obox[:2]).abs().max().item()
    tol = _tol(dtype, ref_gap)
    # (a) teacher forced
    logits, tok, boxes, scores = _teacher_forced(eng, cfg, batch, otok, steps)
    err = (logits - ologits).abs().max().item()
    flips = _check_tokens(tok, otok, margin, tol, "synrec fullsize / oracle")
    box_err = (boxes - obox).abs().max().item()
    score_err = (scores - osc).abs().max().item()
    assert err <= tol, f"teacher-forced logits vs fp32 oracle: {err} (reference's own bf16 gap {ref_gap})"
    assert box_err <= max(12, 2 * ref_box_gap) and score_err <= 2e-2
    assert len(set(otok[0].tolist())) >= 64, "the synthetic model is supposed to walk through the vocabulary"
    # (b) free running, B = 256
    crops = [base[i % 8] for i in range(256)]
    runner = RecognitionRunner(eng, batch_size=256, max_tokens=steps)
    tokens, rscores, bboxes = runner.run(crops, fixed_steps=True)
    first_div = []
    for i in range(8):
        ref = otok[i].tolist()
        k = next((j for j in range(steps) if tokens[i][j] != ref[j]), None)
        first_div.append(k)
        if k is not None:
            assert margin[i, k].item() <= 4 * tol, f"row {i} leaves the oracle at step {k} (margin {margin[i, k].item():.4f})"
    for i in range(8, 256):
        assert tokens[i] == tokens[i % 8] and np.array_equal(bboxes[i], bboxes[i % 8])
    _report("synrec_fullsize_bf16", {"crops": 8, "steps": steps, "max_abs_err_logits_teacher_forced": err,
                                     "reference_own_bf16_gap": ref_gap, "tolerance_used": tol, "reference_own_box_gap": ref_box_gap,
                                     "teacher_forced_token_flips_on_near_ties": flips, "of_tokens": 8 * steps,
                                     "max_box_err": box_err, "max_score_err": score_err,
                                     "free_running_first_divergence_step": first_div,
                                     "oracle_margin_median": margin.median().item(), "oracle_margin_min": margin.min().item(),
                                     "distinct_tokens_row0": len(set(otok[0].tolist()))})
    eng.close()


def test_predictor_trace_replay_gpu(built_lib):
    """The call sequence of the reference's unmodified RecognitionPredictor.prediction_loop (recorded in the build container,
    tests/golden/rec_predictor_trace.pt: left-padded prefills, `ContinuousBatchingCache()` per prefill, merges with offsets of
    both signs, maybe_trim_cache_padding, retired rows that keep decoding) replayed call by call against B200SuryaModel +
    SlotCache on the CUDA engine.  Tokens must equal the recorded (fp32) ones except on recorded near-ties."""
    from oracle import ref_predictors as RP
    from oracle.make_golden import trace_crops
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import B200SuryaModel
    from surya_b200.synth import rec_state_dict

    dtype = torch.float16
    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    g = torch.load(GOLDEN / "rec_predictor_trace.pt")
    eng = _engine(cfg, sd, dtype, max_slots=16, s_max=256, max_patches=4096, max_tokens=1024)
    model = B200SuryaModel(eng)
    stats = {"calls": 0, "rows": 0, "flips": 0, "bbox_err": 0.0}

    def tile_fn(crop):
        img = O.scale_to_fit(np.asarray(crop, dtype=np.float32), (1024, 256))
        return O.process_and_tile(img, cfg.vision_encoder.patch_size, cfg.merge_size)[0]

    def check(i, ev, out):
        tok = out["lm_logits"][:, -1].float().argmax(-1).cpu()
        diff = tok != ev["tok"]
        bad = diff & (ev["margin"] > 4 * TOL_GOLD[dtype])
        assert not bad.any(), f"event {i} ({ev['kind']}): {tok[bad].tolist()} vs recorded {ev['tok'][bad].tolist()}"
        stats["calls"] += 1
        stats["rows"] += tok.numel()
        stats["flips"] += int(diff.sum())
        stats["bbox_err"] = max(stats["bbox_err"], (out["bbox_logits"][:, -1].float().cpu() - ev["bbox"]).abs().max().item())

    free0 = len(eng.free_slots)
    RP.replay_rec_trace(model, g, trace_crops(), tile_fn, check)
    assert len(eng.free_slots) == free0, "replay leaked KV slots"
    assert stats["bbox_err"] < 5e-3
    _report("predictor_trace_replay_fp16", stats)
    eng.close()


def test_capacity_and_bounds_are_loud(built_lib):
    """ADVICE r1: decode past s_max must raise (never write into a neighbour's KV rows), the runner must chunk prefills by
    engine capacity and give slots back when a prefill fails."""
    from surya_b200 import _lib
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    eng = _engine(cfg, sd, torch.float16, max_slots=5, s_max=64, max_patches=400, max_tokens=200)
    crops = list(rec_synthetic_crops(6, 48, 512, seed=3))            # 160 patches, 46 prompt tokens each
    with pytest.raises(_lib.SuryaB200Error):                         # 46 + 32 > s_max
        RecognitionRunner(eng, batch_size=4, max_tokens=32).run(crops[:1])
    assert len(eng.free_slots) == 5
    with pytest.raises(_lib.SuryaB200Error):                         # runner needs batch_size + 1 slots
        RecognitionRunner(eng, batch_size=5, max_tokens=4).run(crops[:1])
    # max_patches = 400 admits two crops per prefill: six crops through four rows still all decode, identically to solo runs
    runner = RecognitionRunner(eng, batch_size=4, max_tokens=6)
    tok, sc, bb = runner.run(crops, fixed_steps=True)
    for i in (0, 5):
        t1, s1, b1 = runner.run([crops[i]], fixed_steps=True)
        assert tok[i] == t1[0] and np.array_equal(bb[i], b1[0])
    assert len(eng.free_slots) == 5
    # raw decode at a full slot
    slot = torch.tensor(eng.alloc_slots(1), dtype=torch.int32, device="cuda")
    with pytest.raises(_lib.SuryaB200Error):
        eng.decode(torch.zeros(1, dtype=torch.int64, device="cuda"), slot, torch.tensor([64], dtype=torch.int32, device="cuda"))
    with pytest.raises(_lib.SuryaB200Error):
        eng.decode_steps(torch.zeros(1, dtype=torch.int64, device="cuda"), slot, torch.tensor([60], dtype=torch.int32, device="cuda"), 8)
    eng.close()


def test_empty_single_and_ragged_batches(built_lib):
    """Edge cases of the runner: no crops, one crop, more crops than batch rows with ragged widths (prompts of different
    lengths, different window counts) — every crop must decode exactly as it does alone."""
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    cfg = tiny_rec()
    eng = _engine(cfg, rec_state_dict(cfg, seed=0), torch.float16, max_slots=8, s_max=160, max_patches=4096, max_tokens=1024)
    runner = RecognitionRunner(eng, batch_size=3, max_tokens=6)
    tok, sc, bb = runner.run([])
    assert tok == [] and sc == [] and bb.shape == (0, 6, 6)
    crops = [rec_synthetic_crops(1, h, w, seed=s)[0] for s, (h, w) in enumerate([(48, 512), (40, 300), (64, 900), (48, 512), (32, 200), (56, 700), (48, 640)])]
    alone = [runner.run([c], fixed_steps=True) for c in crops]
    tok, sc, bb = runner.run(crops, fixed_steps=True)      # 7 crops through 3 batch rows: slots are recycled
    for i in range(len(crops)):
        assert tok[i] == alone[i][0][0] and sc[i] == alone[i][1][0] and np.array_equal(bb[i], alone[i][2][0]), i
    eng.close()


@pytest.mark.parametrize("R,max_tokens,poll", [(40, 100, 8), (40, 60, 1), (6, 1000, 5), (2, 50, 7)])
def test_stop_rules_kernel_matches_python_rules(built_lib, R, max_tokens, poll):
    """SURVEY §8 f3: stop_rules_kernel (EOS / PAD flag, max_tokens, detect_repeat_token) against the host rules of
    RecognitionRunner (mirror of surya/recognition/__init__.py:585-598 + util.py:59-69) on crafted token streams — integer work,
    exact: per round trip the valid-step count, the sticky done flag, the generated count and the active-row count."""
    from surya_b200 import ops
    from surya_b200.recognition import detect_repeat_token

    rng = np.random.default_rng(R * 1000 + max_tokens)
    T_total, EOS = 130, 1
    streams = []
    streams.append(rng.permutation(5000)[:T_total] + 10)                                  # all distinct: only max_tokens stops it
    s1 = rng.permutation(5000)[:T_total] + 10; s1[17] = EOS; streams.append(s1)           # EOS at step 17
    streams.append(np.full(T_total, 77))                                                  # one token for ever
    s3 = rng.permutation(5000)[:T_total] + 10; s3[10:] = np.tile([5, 6, 7], T_total)[:T_total - 10]; streams.append(s3)
    s4 = rng.permutation(5000)[:T_total] + 10; s4[3:] = np.tile([11, 12, 13, 14, 15], T_total)[:T_total - 3]; streams.append(s4)
    streams.append(np.tile([21, 22, 23, 24, 25, 26], T_total)[:T_total])                  # period 6: u = 6 > 5, never a repeat stop
    streams.append(rng.integers(10, 5000, T_total))                                       # idle row (row_done seeded 1)
    s7 = np.tile([31, 32], T_total)[:T_total].copy(); s7[45] = 999; streams.append(s7)     # period 2 with one glitch
    s8 = rng.integers(10, 14, T_total); streams.append(s8)                                 # 4 symbols at random: u <= 5, rarely periodic
    B = len(streams)
    first = rng.integers(10, 5000, B)                                                      # the prefill tokens
    first[2], first[7] = 77, 32
    idle = [6]
    toks = np.stack(streams, 1).astype(np.int64)                                           # [T_total, B]
    dones = (toks == EOS).astype(np.uint8)

    # host rules, token by token
    hist = [[int(first[r])] for r in range(B)]
    alive = [r not in idle for r in range(B)]
    dev = "cuda"
    gen = torch.tensor([0 if r in idle else 1 for r in range(B)], dtype=torch.int32, device=dev)
    ring = torch.zeros((B, R), dtype=torch.int64, device=dev)
    ring[:, 0] = torch.from_numpy(first).to(dev)
    row_done = torch.tensor([1 if r in idle else 0 for r in range(B)], dtype=torch.uint8, device=dev)
    valid = torch.zeros(B, dtype=torch.int32, device=dev)
    active = torch.zeros(1, dtype=torch.int32, device=dev)
    t0 = 0
    while t0 < T_total and any(alive):
        n = min(poll, T_total - t0)
        th = torch.from_numpy(toks[t0:t0 + n]).contiguous().to(dev)
        dh = torch.from_numpy(dones[t0:t0 + n]).contiguous().to(dev)
        valid.zero_()
        for s in range(n):
            ops.rec_stop_rules(th, dh, s, gen, ring, row_done, valid, active, max_tokens, R)
        torch.cuda.synchronize()
        exp_valid = [0] * B
        for r in range(B):
            if not alive[r]:
                continue
            for s in range(n):
                hist[r].append(int(toks[t0 + s, r]))
                exp_valid[r] = s + 1
                if hist[r][-1] == EOS or len(hist[r]) >= max_tokens or detect_repeat_token(hist[r], R):
                    alive[r] = False
                    break
        assert valid.cpu().tolist() == exp_valid, f"chunk at {t0}: valid {valid.cpu().tolist()} vs {exp_valid}"
        assert row_done.cpu().tolist() == [0 if a else 1 for a in alive], f"chunk at {t0}: done flags"
        assert gen.cpu().tolist() == [0 if r in idle else len(hist[r]) for r in range(B)], f"chunk at {t0}: generated counts"
        assert int(active.item()) == sum(alive)
        t0 += n
    assert not any(alive) or max_tokens > T_total
    if R == 40 and max_tokens == 100:
        assert len(hist[2]) == 40 and len(hist[1]) == 19 and len(hist[0]) == 100 and len(hist[5]) == 100      # the rules all fired


@pytest.mark.parametrize("max_repeats,steps,poll", [(40, 24, 5), (2, 30, 8), (3, 12, 1)])
def test_device_stop_rules_equal_host_rules(built_lib, max_repeats, steps, poll):
    """RecognitionRunner with the stop rules on the device (default) returns exactly what the per-token host loop returns: tokens,
    scores and boxes of every crop, for several polling intervals / repeat windows (a window of 2 makes the repeat rule fire on
    the synthetic model's occasional double tokens)."""
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import RecognitionRunner
    from surya_b200.synth import rec_state_dict, rec_synthetic_crops

    dtype = torch.float16
    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    crops = [rec_synthetic_crops(1, 48, 256 + 37 * i, seed=100 + i)[0] for i in range(11)]
    eng = _engine(cfg, sd, dtype, max_slots=8, s_max=256, max_patches=4096, max_tokens=1024)
    out = {}
    for mode in ("host", "device"):
        runner = RecognitionRunner(eng, batch_size=4, max_tokens=steps, poll=poll, stop_rules=mode)
        runner.MAX_REPEATS = max_repeats
        out[mode] = runner.run(crops)
    th, sh, bh = out["host"]
    td, sd_, bd = out["device"]
    assert td == th
    assert all(np.array_equal(np.asarray(a, np.float32), np.asarray(b, np.float32)) for a, b in zip(sd_, sh))
    assert np.array_equal(bd, bh)
    lens = [len(t) for t in th]
    _report(f"stop_rules_R{max_repeats}_T{steps}", {"lengths": lens})
    # a fixed-steps run right after a device-rules run must not see the rules any more (the engine state was reset)
    fixed = RecognitionRunner(eng, batch_size=4, max_tokens=steps, poll=poll).run(crops[:3], fixed_steps=True)[0]
    assert all(len(t) == steps for t in fixed)
    eng.close()
