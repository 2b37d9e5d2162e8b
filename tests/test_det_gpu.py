"""Detection path parity (GPU): kernels vs PyTorch fp32 restatements, engine vs the CPU oracle and the reference golden.
North-star tolerance: sigmoid heatmaps within 1e-3 (fp16) of the reference path on identical inputs."""
import json
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

from oracle import det_oracle as D

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
OUT = ROOT / "gpurun_out"
GOLDEN = ROOT / "tests" / "golden"


def _report(name, payload):
    OUT.mkdir(exist_ok=True)
    path = OUT / "det_parity.json"
    data = json.loads(path.read_text()) if path.exists() else {}
    data[name] = payload
    path.write_text(json.dumps(data, indent=1))


@pytest.mark.parametrize("cin,cout,stride,hw,act,res", [
    (32, 32, 1, (64, 48), "hardswish", False), (32, 512, 2, (64, 64), "hardswish", False), (64, 256, 1, (40, 56), "hardswish", False),
    (64, 1024, 2, (32, 64), "none", False), (128, 512, 1, (24, 40), "hardswish", False), (32, 32, 1, (72, 80), "none", True),
    (64, 96, 1, (17, 23), "relu", True), (32, 32, 1, (21, 37), "hardswish", True), (32, 32, 1, (200, 176), "hardswish", False),
])
def test_conv3x3_igemm(built_lib, cin, cout, stride, hw, act, res):
    from surya_b200 import ops

    dtype = torch.float16
    g = torch.Generator(device="cuda").manual_seed(cin + cout + stride)
    N, (H, W) = 3, hw
    x = torch.randn(N, H, W, cin, device="cuda", generator=g).to(dtype)
    w = (torch.randn(cout, cin, 3, 3, device="cuda", generator=g) * (cin * 9) ** -0.5).to(dtype)
    b = torch.randn(cout, device="cuda", generator=g) * 0.1
    Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
    r = torch.randn(N, Ho, Wo, cout, device="cuda", generator=g).to(dtype) if res else None
    out = ops.conv2d_nhwc(x, w.permute(0, 2, 3, 1).reshape(cout, -1).contiguous(), b, r, 3, stride, 1, act)
    torch.cuda.synchronize()
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), b, stride=stride, padding=1).to(dtype).float()
    if act == "hardswish":
        ref = F.hardswish(ref).to(dtype).float()
    elif act == "relu":
        ref = F.relu(ref)
    ref = ref.permute(0, 2, 3, 1)
    if res:
        ref = (ref + r.float()).to(dtype).float()
    err = (out.float() - ref).abs().max().item()
    assert err < 8e-3, f"conv3x3 cin={cin} cout={cout} s={stride}: max err {err}"


@pytest.mark.parametrize("ks,stride,C,hw", [(3, 1, 64, (20, 28)), (3, 2, 2048, (20, 28)), (5, 1, 1536, (20, 28)),
                                            (3, 1, 1024, (64, 64)), (3, 1, 72, (37, 45)), (3, 1, 3072, (32, 32)), (3, 1, 8, (5, 3))])
def test_dwconv(built_lib, ks, stride, C, hw):
    from surya_b200 import ops

    dtype = torch.float16
    g = torch.Generator(device="cuda").manual_seed(ks + C)
    x = torch.randn(3, hw[0], hw[1], C, device="cuda", generator=g).to(dtype)
    w = (torch.randn(C, 1, ks, ks, device="cuda", generator=g) / ks).to(dtype)
    b = torch.randn(C, device="cuda", generator=g) * 0.1
    pad = ks // 2
    out = ops.dwconv_nhwc(x, w.reshape(C, ks * ks).t().contiguous(), b, ks, stride, pad, "hardswish")
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), b, stride=stride, padding=pad, groups=C).to(dtype).float()
    ref = F.hardswish(ref).permute(0, 2, 3, 1)
    assert (out.float() - ref).abs().max().item() < 4e-3


@pytest.mark.parametrize("HW", [300, 301, 1024, 67])
def test_grouped_pw_and_lite_mla(built_lib, HW):
    from surya_b200 import ops

    dtype = torch.float16
    g = torch.Generator(device="cuda").manual_seed(0)
    B, heads, dim = 2, 16, 32
    C = 3 * heads * dim
    a = torch.randn(B * HW, C, device="cuda", generator=g).to(dtype)
    w = (torch.randn(C, 32, device="cuda", generator=g) * 32 ** -0.5).to(dtype)
    wp = torch.zeros(C, 64, device="cuda", dtype=dtype)
    wp[:, :32] = w
    out = ops.gemm_grouped(a, wp, groups=3 * heads)
    ref = F.conv2d(a.float().t().reshape(1, C, B * HW, 1), w.float().reshape(C, 32, 1, 1), groups=3 * heads).reshape(C, -1).t()
    assert (out.float() - ref).abs().max().item() < 4e-3
    qa = torch.randn(B * HW, C, device="cuda", generator=g).to(dtype)
    qb = torch.randn(B * HW, C, device="cuda", generator=g).to(dtype)
    o = ops.lite_mla(qa, qb, B, HW, heads, dim, 1e-5)
    ms = torch.cat([qa.reshape(B, HW, C), qb.reshape(B, HW, C)], -1).reshape(B, HW, 2 * heads, 3 * dim).permute(0, 2, 1, 3).float()
    q, k, v = ms.chunk(3, -1)
    q, k = F.relu(q), F.relu(k)
    v = F.pad(v, (0, 1), value=1.0)
    kv = k.transpose(-1, -2) @ v
    r = q @ kv
    r = (r[..., :-1] / (r[..., -1:] + 1e-5)).permute(0, 2, 1, 3).reshape(B * HW, 2 * heads * dim)
    assert (o.float() - r).abs().max().item() < 2e-3 * max(1.0, r.abs().max().item())


@pytest.mark.parametrize("kind,size", [("tiny", (256, 256)), ("tiny", (384, 512)), ("default", (1024, 1024))])
def test_engine_vs_oracle(built_lib, kind, size):
    from oracle import det_oracle as D
    from surya_b200.config import det_default, det_tiny
    from surya_b200.detection import DetEngine
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_tiny() if kind == "tiny" else det_default()
    sd = det_state_dict(cfg, seed=0)
    B = 2
    pages = det_synthetic_pages(B, max(size), seed=3, text_like=(kind == "default"))[:, : size[0], : size[1]]
    x = det_normalize(pages)
    eng = DetEngine(cfg, sd, torch.float16, max_batch=2, max_hw=size)
    got = eng.forward(x.cuda())
    up = eng.upsample(got, size)
    torch.cuda.synchronize()
    ref = D.forward(sd, cfg, x)
    err = (got.float().cpu() - ref).abs().max().item()
    ref_up = D.upsample_to_input(ref, size)
    err_up = (up.cpu() - ref_up).abs().max().item()
    _report(f"{kind}_{size[0]}x{size[1]}", {"max_abs_err_vs_fp32_oracle": err, "max_abs_err_upsampled": err_up,
                                            "ref_min": ref.min().item(), "ref_max": ref.max().item(), "ref_std": ref.std().item()})
    assert got.shape == ref.shape
    # fp16 engine vs fp32 oracle.  The reference's own fp16 path sits 2.2e-3 from its fp32 path on text-like pages
    # (tests/golden/det_default.pt), so 1e-3 is only reachable on the shallow config; bound stated per config.
    tol = 1e-3 if kind == "tiny" else 6e-3
    assert err < tol, f"heatmap max abs err {err}"
    assert err_up < tol
    eng.close()


def test_engine_vs_reference_golden(built_lib):
    from surya_b200.config import det_default
    from surya_b200.detection import B200EfficientViT, DetEngine
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    g = torch.load(GOLDEN / "det_default.pt")
    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    x = det_normalize(det_synthetic_pages(1, 512, seed=11, text_like=True))
    assert abs(x.double().sum().item() - g["input_checksum"].item()) < 1e-3
    eng = DetEngine(cfg, sd, torch.float16, max_batch=1, max_hw=(512, 512))
    model = B200EfficientViT(eng)
    assert model.config.num_labels == 2
    out = model(pixel_values=x.to("cuda", torch.float16)).logits
    o = out.float().cpu()
    err = (o - g["logits"]).abs().max().item()
    err16 = (o - g["logits_fp16_path"]).abs().max().item()
    ref_gap = (g["logits_fp16_path"] - g["logits"]).abs().max().item()
    _report("golden_512", {"max_abs_err_vs_reference_fp32": err, "max_abs_err_vs_reference_fp16_path": err16,
                           "reference_fp16_vs_fp32_gap": ref_gap})
    assert err16 < 5e-3, f"vs the reference's fp16 path: {err16}"
    assert err < 2.5 * ref_gap, f"engine error {err} vs the reference's own fp16-fp32 gap {ref_gap}"
    eng.close()


def test_stage_error_growth_vs_reference_fp16_path(built_lib):
    """Where does the fp16 error come from?  Per feature stage (and for the heat maps): engine vs the fp32 oracle next to the
    reference ALGORITHM evaluated in fp16 (oracle on CPU half tensors = model.half()) vs the same fp32 oracle, one 512x512
    text-like page, default config.  Written to gpurun_out/det_parity.json; the engine may not be worse than 1.5x the
    reference's own fp16 path at any stage."""
    from surya_b200.config import det_default
    from surya_b200.detection import DetEngine
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    x = det_normalize(det_synthetic_pages(1, 512, seed=11, text_like=True))
    eng = DetEngine(cfg, sd, torch.float16, max_batch=1, max_hw=(512, 512))
    got = eng.forward(x.cuda()).float().cpu()
    with torch.inference_mode():
        f32 = D.backbone(sd, cfg, x)
        h32 = torch.special.expit(D.decode_head(sd, cfg, f32))
        sd16 = {k: v.half() for k, v in sd.items()}
        f16 = D.backbone(sd16, cfg, x.half())
        h16 = torch.special.expit(D.decode_head(sd16, cfg, f16)).float()
    rep = {}
    for i, (a, b) in enumerate(zip(f32, f16)):
        C, H, W = a.shape[1:]
        e = eng.debug_buffer(f"feat{i}", 1, H, W, C).float().cpu().permute(0, 3, 1, 2)
        scale = a.abs().max().item()
        rep[f"feat{i}"] = {"engine_err": (e - a).abs().max().item(), "reference_fp16_err": (b.float() - a).abs().max().item(),
                           "engine_rel_fro": ((e - a).norm() / a.norm()).item(),
                           "reference_fp16_rel_fro": ((b.float() - a).norm() / a.norm()).item(), "absmax": scale}
    rep["heatmap"] = {"engine_err": (got - h32).abs().max().item(), "reference_fp16_err": (h16 - h32).abs().max().item(),
                      "engine_rms": (got - h32).pow(2).mean().sqrt().item(), "reference_fp16_rms": (h16 - h32).pow(2).mean().sqrt().item()}
    # decode head in isolation: the reference algorithm (fp16 and fp32) applied to the ENGINE's own stage features
    efeats = []
    for i, a in enumerate(f32):
        C, H, W = a.shape[1:]
        efeats.append(eng.debug_buffer(f"feat{i}", 1, H, W, C).cpu().permute(0, 3, 1, 2).contiguous())
    with torch.inference_mode():
        hh16 = torch.special.expit(D.decode_head(sd16, cfg, efeats)).float()
        hh32 = torch.special.expit(D.decode_head(sd, cfg, [f.float() for f in efeats]))
    rep["head_only"] = {"engine_vs_fp16_head_on_engine_feats_rms": (got - hh16).pow(2).mean().sqrt().item(),
                        "engine_vs_fp32_head_on_engine_feats_rms": (got - hh32).pow(2).mean().sqrt().item(),
                        "fp16_head_vs_fp32_head_on_engine_feats_rms": (hh16 - hh32).pow(2).mean().sqrt().item(),
                        "fp32_head_on_engine_feats_vs_truth_rms": (hh32 - h32).pow(2).mean().sqrt().item()}
    _report("stage_error_growth_512", rep)
    for k, v in rep.items():
        if k.startswith("feat"):
            assert v["engine_rel_fro"] <= 1.5 * v["reference_fp16_rel_fro"] + 1e-5, (k, v)
    assert rep["heatmap"]["engine_rms"] <= 2.5 * rep["heatmap"]["reference_fp16_rms"] + 1e-5, rep["heatmap"]
    eng.close()


def test_default_batch32_vs_oracle(built_lib):
    """BASELINE config 3 at full size: 32 pages of 1024x1024 (4 distinct text-like pages x 8 replicas) through the default
    EfficientViT in one call.  The 4 distinct pages are compared with the fp32 oracle (tolerance = 1.5x the reference's own fp16
    gap measured on one of them, floor 1e-3); replicas must be bit-identical wherever they sit in the batch."""
    from surya_b200.config import det_default
    from surya_b200.detection import DetEngine
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    base = det_normalize(det_synthetic_pages(4, 1024, seed=21, text_like=True))
    x = base.repeat(8, 1, 1, 1)
    eng = DetEngine(cfg, sd, torch.float16, max_batch=32, max_hw=(1024, 1024))
    got = eng.forward(x.half().cuda()).float().cpu()
    torch.set_num_threads(max(1, min(64, len(__import__("os").sched_getaffinity(0)))))
    ref = D.forward(sd, cfg, base)
    with torch.inference_mode():
        sd16 = {k: v.half() for k, v in sd.items()}
        ref16 = torch.special.expit(D.decode_head(sd16, cfg, D.backbone(sd16, cfg, base[:1].half()))).float()
    ref_gap = (ref16 - ref[:1]).abs().max().item()
    err = (got[:4] - ref).abs().max().item()
    rms = (got[:4] - ref).pow(2).mean().sqrt().item()
    ref_rms = (ref16 - ref[:1]).pow(2).mean().sqrt().item()
    for r in range(4, 32):
        assert torch.equal(got[r], got[r % 4]), f"page {r} differs from its replica"
    _report("default_1024_batch32", {"max_abs_err_vs_fp32_oracle": err, "reference_own_fp16_gap": ref_gap, "rms_err": rms,
                                     "reference_own_fp16_rms": ref_rms})
    assert err <= max(1e-3, 1.5 * ref_gap), f"{err} vs the reference's own fp16 gap {ref_gap}"
    assert rms <= 1.5 * ref_rms + 1e-5
    eng.close()


@pytest.mark.parametrize("kind", ["default", "tiny"])
def test_text_front_matches_numpy_reference_path(built_lib, kind):
    """SURVEY §8 f1: upsample + dynamic thresholds + binarisation on the device vs the reference's NumPy path (oracle restatement
    of surya/detection/heatmap.py:14-24, 27-107) on the fp32 maps the predictor would have copied to the host: the 16-bit map is
    bit-identical to the fp32 up-sampled text channel, thresholds agree to fp32 rounding, masks are identical, and the boxes /
    confidences produced from (map, mask, thresholds) equal detect_boxes on the fp32 map.  Also the pipelined host path."""
    import numpy as np

    from surya_b200.config import det_default, det_tiny
    from surya_b200.detection import DetEngine, detect_text_front_host, text_boxes_from_front
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg, S = (det_default(), 512) if kind == "default" else (det_tiny(), 256)
    sd = det_state_dict(cfg, seed=0)
    x = det_normalize(det_synthetic_pages(5, S, seed=31, text_like=True)).half()
    eng = DetEngine(cfg, sd, torch.float16, max_batch=5, max_hw=(S, S))
    logits = eng.forward(x.cuda())
    up = eng.upsample(logits, (S, S)).cpu()                      # what the reference ships to the host (fp32, both channels)
    front = {k: v.cpu() for k, v in eng.text_front(logits, (S, S)).items()}
    assert torch.equal(front["map"].float(), up[:, 0]), "16-bit text map is not the fp32 up-sampled channel"
    n_boxes = 0
    for b in range(5):
        line = up[b, 0].numpy()
        tt, low, avg = D.dynamic_thresholds(line)
        assert abs(front["thr"][b, 2].item() - float(avg)) <= 2e-6 * max(1.0, abs(float(avg)))
        assert abs(front["thr"][b, 0].item() - float(tt)) <= 2e-6 and abs(front["thr"][b, 1].item() - float(low)) <= 2e-6
        assert np.array_equal(front["mask"][b].numpy(), (line > np.float32(front["thr"][b, 1].item())).astype(np.uint8))
        assert np.array_equal(front["mask"][b].numpy(), (line > low).astype(np.uint8)), "mask differs from the NumPy path"
        ref_boxes, ref_conf = D.detect_boxes(line)
        boxes, conf = text_boxes_from_front(front["map"][b].numpy(), front["mask"][b].numpy(), front["thr"][b, 0].item(),
                                            front["thr"][b, 1].item())
        assert len(boxes) == len(ref_boxes)
        for p, q in zip(boxes, ref_boxes):
            assert np.array_equal(p, q)
        assert np.allclose(conf, ref_conf, rtol=0, atol=1e-6)
        n_boxes += len(boxes)
    host = detect_text_front_host(eng, x.pin_memory(), chunk=2)
    for k in ("map", "mask", "thr"):
        assert torch.equal(host[k], front[k]), k
    _report(f"text_front_{kind}", {"pages": 5, "boxes": n_boxes, "bytes_per_pixel_to_host": 3,
                                   "top10_mean": [round(v, 4) for v in front["thr"][:, 2].tolist()]})
    eng.close()


def test_pipelined_host_path_equals_single_shot(built_lib):
    """detect_pages_host (chunks over three streams, host in / host out) == forward + upsample of the whole batch, bit for bit
    (also exercises batch invariance: 5 pages in chunks of 2 vs all at once)."""
    from surya_b200.config import det_tiny
    from surya_b200.detection import DetEngine, detect_heatmaps, detect_pages_host
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_tiny()
    eng = DetEngine(cfg, det_state_dict(cfg, seed=0), torch.float16, max_batch=5, max_hw=(256, 256))
    x = det_normalize(det_synthetic_pages(5, 256, seed=5)).half().pin_memory()
    ref = detect_heatmaps(eng, x.cuda()).cpu()
    for _ in range(2):      # second call reuses the staging buffers
        got = detect_pages_host(eng, x, chunk=2)
        torch.cuda.synchronize()
        assert got.is_pinned() and torch.equal(got, ref)
    eng.close()


def test_ocr_pipeline_end_to_end_tiny(built_lib):
    """BASELINE config 5 data flow on small engines: uint8 pages -> device normalisation + detection + post-processing front half
    -> host boxes -> polygon crops -> width-sorted recognition.  Stage by stage against independent computations: polygons from
    the oracle's detect_boxes on the engine's own fp32 maps, crops re-sliced here, tokens from a separate runner call per crop."""
    import numpy as np

    from surya_b200.config import det_tiny, tiny_rec
    from surya_b200.detection import DetEngine
    from surya_b200.pipeline import OcrPipeline, page_polygons, slice_polygon
    from surya_b200.recognition import RecEngine, RecognitionRunner
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages, rec_state_dict

    S = 256
    dcfg, rcfg = det_tiny(), tiny_rec()
    det = DetEngine(dcfg, det_state_dict(dcfg, 0), torch.float16, max_batch=4, max_hw=(S, S))
    rec = RecEngine(rcfg, rec_state_dict(rcfg, 0), dtype=torch.float16, max_slots=9, s_max=256, max_patches=8192, max_tokens=2048)
    pages = det_synthetic_pages(5, S, seed=77, text_like=True)
    pipe = OcrPipeline(det, rec, rec_batch=8, max_tokens=6, det_chunk=2, workers=2)
    per_page, timings = pipe.run(pages, fixed_steps=True)
    assert len(per_page) == 5 and sum(len(p) for p in per_page) >= 5
    # device normalisation == host normalisation
    xn = det.normalize_u8(torch.from_numpy(pages).cuda())
    assert torch.equal(xn.cpu(), det_normalize(pages).half())
    up = det.upsample(det.forward(xn), (S, S)).cpu()
    runner = RecognitionRunner(rec, batch_size=8, max_tokens=6)
    n_lines = 0
    for pg in range(5):
        boxes, conf = D.detect_boxes(up[pg, 0].numpy())
        polys, pconf = page_polygons(boxes, conf, (S, S), (S, S))
        assert [ln.polygon for ln in per_page[pg]] == polys
        assert np.allclose([ln.confidence for ln in per_page[pg]], pconf, atol=1e-6)
        for ln in per_page[pg]:
            crop = slice_polygon(pages[pg].astype(np.float32), ln.polygon)
            tok, sc, bb = runner.run([crop], fixed_steps=True)
            assert ln.tokens == tok[0] and np.array_equal(ln.boxes, bb[0]), (pg, ln.polygon)
            n_lines += 1
    _report("ocr_pipeline_tiny", {"pages": 5, "lines": n_lines, "timings_s": {k: round(v, 4) for k, v in timings.items()}})
    # SURVEY §8 f2: the same flow with the crop preprocessing on the device (uint8 crops up, sb_rec_preprocess): same lines, the
    # tokens of a direct runner call on the same uint8 crop; against the OpenCV flow tokens may differ on near-ties only
    pipe_dev = OcrPipeline(det, rec, rec_batch=8, max_tokens=6, det_chunk=2, workers=2, preprocess="device")
    per_page_dev, _ = pipe_dev.run(pages, fixed_steps=True)
    same = total = 0
    for pg in range(5):
        assert [ln.polygon for ln in per_page_dev[pg]] == [ln.polygon for ln in per_page[pg]]
        for ln, ln_host in zip(per_page_dev[pg], per_page[pg]):
            tok, sc, bb = runner.run([slice_polygon(pages[pg], ln.polygon)], fixed_steps=True, preprocess="device")
            assert ln.tokens == tok[0] and np.array_equal(ln.boxes, bb[0]), (pg, ln.polygon)
            same += int(ln.tokens == ln_host.tokens)
            total += 1
    assert same >= total - max(1, total // 10), f"device preprocessing changed the tokens of {total - same} of {total} lines"
    rec.close()
    det.close()


def _head_logits(size, B, seed):
    from surya_b200.config import det_default
    from surya_b200.detection import DetEngine
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    cfg = det_default()
    eng = DetEngine(cfg, det_state_dict(cfg, seed=0), torch.float16, max_batch=B, max_hw=size)
    x = det_normalize(det_synthetic_pages(B, max(size), seed=seed, text_like=True)[:, : size[0], : size[1]])
    out = eng.forward(x.cuda()).float().cpu()
    eng.close()
    return out


@pytest.mark.parametrize("size", [(512, 512), (320, 448)])
@pytest.mark.parametrize("switch", ["SB_DET_FUSED_HEAD", "SB_FMB_FUSED"])
def test_fused_kernels_equal_unfused_ops(built_lib, switch, size, tmp_path):
    """The fused tcgen05 kernels against the op sequences they replace (switch = 1 / 0, read once per process, hence the subprocesses):
      SB_DET_FUSED_HEAD  det_head.cu (upsample + concat + fuse conv + ReLU + classifier + sigmoid) vs upsample_cat -> gemm ->
                         classifier: same rounding points, only the fp32 summation order of the 512-long classifier dot differs;
      SB_FMB_FUSED       conv_fmb.cu (3x3 expand + Hardswish + 1x1 project + shortcut, back-to-back GEMM) vs conv_igemm -> gemm:
                         same rounding points and the same k order.
    Heatmaps must agree to one fp16 ulp.  320x448 gives partial tiles in both directions at every stage."""
    import os
    import subprocess
    import sys

    outs = {}
    on = "1"
    for val in (on, "0"):
        path = tmp_path / f"variant{val}.pt"
        code = (f"import sys, torch; sys.path.insert(0, {str(ROOT)!r}); sys.path.insert(0, {str(ROOT / 'tests')!r});"
                f"import test_det_gpu as t; torch.save(t._head_logits({size!r}, 2, 5), {str(path)!r})")
        r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **{switch: val}), capture_output=True, text=True, timeout=240)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        outs[val] = torch.load(path)
    fused, unfused = outs[on], outs["0"]
    assert fused.shape == unfused.shape == (2, 2, size[0] // 4, size[1] // 4)
    diff = (fused - unfused).abs()
    frac_equal = (diff == 0).float().mean().item()
    print(f"{switch}={on} vs 0 at {size}: max |diff| {diff.max().item():.3g}, identical {100 * frac_equal:.2f} %")
    assert diff.max().item() <= 2 ** -10 and frac_equal > 0.98
