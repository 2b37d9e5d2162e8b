"""GPU parity tests for the layout path (SURVEY.md §8 rows a19-a22): each kernel vs a torch restatement with the same
rounding points, then the whole Swin encoder / ADETR greedy loop vs the fp32 oracle and the committed reference golden."""
import math
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
DTYPES = [torch.float16, torch.bfloat16]


def _ulp(dtype):
    return 2.0 ** -10 if dtype == torch.float16 else 2.0 ** -7


def _close(got, ref, dtype, scale=None, n_ulp=4.0):
    got, ref = got.float().cpu(), ref.float().cpu()
    mag = ref.abs() if scale is None else torch.full_like(ref, float(scale))
    tol = n_ulp * _ulp(dtype) * torch.clamp(mag, min=2.0 ** -6)
    bad = (got - ref).abs() > tol
    assert not bad.any(), f"{int(bad.sum())} / {bad.numel()} off; max err {(got - ref).abs().max().item():.4g}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_layernorm(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator().manual_seed(0)
    for rows, C in ((37, 128), (200, 512), (64, 1024), (9, 4096)):
        x = (torch.randn(rows, C, generator=g) * 2 + 0.3).to(dtype)
        w, b = (1 + 0.1 * torch.randn(C, generator=g)).to(dtype), (0.1 * torch.randn(C, generator=g)).to(dtype)
        ref = F.layer_norm(x.float(), (C,), w.float(), b.float(), 1e-5)
        got = ops.layernorm(x.cuda(), w.cuda(), b.cuda(), 1e-5)
        _close(got, ref, dtype, n_ulp=2.0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_rmsnorm_adetr(built_lib, dtype):
    from oracle.layout_oracle import adetr_rmsnorm
    from surya_b200 import ops

    g = torch.Generator().manual_seed(1)
    x = (torch.randn(33, 1024, generator=g) * 3).to(dtype)
    x[5] *= 200.0          # exercises the variance clamp
    w = (0.1 * torch.randn(1024, generator=g)).to(dtype)
    ref = adetr_rmsnorm(x, w, 1e-6)
    got = ops.rmsnorm_adetr(x.cuda(), w.cuda(), 1e-6)
    _close(got, ref, dtype, n_ulp=2.0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_patch_gather_and_merge(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator().manual_seed(2)
    px = torch.randn(2, 3, 32, 48, generator=g)
    got = ops.patch_gather(px.cuda(), 4, 64, dtype).cpu()
    ref = px.to(dtype).reshape(2, 3, 8, 4, 12, 4).permute(0, 2, 4, 1, 3, 5).reshape(2 * 8 * 12, 48)
    assert torch.equal(got[:, :48], ref) and (got[:, 48:] == 0).all()
    x = torch.randn(2 * 8 * 12, 128, generator=g).to(dtype)
    m = ops.patch_merge_gather(x.cuda(), 2, 8, 12).cpu()
    v = x.view(2, 8, 12, 128)
    ref = torch.cat([v[:, 0::2, 0::2], v[:, 1::2, 0::2], v[:, 0::2, 1::2], v[:, 1::2, 1::2]], -1).reshape(-1, 512)
    assert torch.equal(m, ref)
    tab = torch.randn(8 * 12, 128, generator=g).to(dtype)
    y = ops.add_bcast_rows_(x.cuda().clone(), tab.cuda()).cpu()
    assert torch.equal(y, (x.view(2, 96, 128) + tab).view(-1, 128))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shift", [0, 4])
@pytest.mark.parametrize("nh,H,W", [(4, 16, 24), (8, 8, 16), (32, 8, 8)])
def test_swin_window_attn(built_lib, dtype, shift, nh, H, W):
    """vs DonutSwinSelfAttention + window partition / shift / mask (surya/common/donut/encoder.py:321-398, 560-640)."""
    from oracle.layout_oracle import relative_position_index, shift_attn_mask, window_partition, window_reverse
    from surya_b200 import ops

    g = torch.Generator().manual_seed(3)
    B, hd, ws = 2, 32, 8
    C = nh * hd
    qkv = torch.randn(B * H * W, 3 * C, generator=g).to(dtype)
    table = (0.5 * torch.randn((2 * ws - 1) ** 2, nh, generator=g)).to(dtype)
    got = ops.swin_window_attn(qkv.cuda(), table.cuda(), B, H, W, nh, shift)
    # torch restatement with the reference's rounding points (scores, +bias, +mask, softmax, context all rounded to dtype)
    x = qkv.view(B, H, W, 3 * C)
    if shift:
        x = torch.roll(x, (-shift, -shift), (1, 2))
    win = window_partition(x, ws).view(-1, ws * ws, 3, nh, hd)
    q, k, v = (win[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    s = (q.float() @ k.float().transpose(-1, -2)).to(dtype)
    s = (s.float() / math.sqrt(hd)).to(dtype)
    bias = table[relative_position_index(ws).view(-1)].view(ws * ws, ws * ws, nh).permute(2, 0, 1)
    s = (s.float() + bias.float()).to(dtype)
    if shift:
        mask = shift_attn_mask(H, W, ws, shift, dtype)
        s = (s.view(B, -1, nh, 64, 64).float() + mask.float()[None, :, None]).to(dtype).view(-1, nh, 64, 64)
    p = torch.softmax(s.float(), -1).to(dtype)
    ctx = (p.float() @ v.float()).to(dtype).permute(0, 2, 1, 3).reshape(-1, ws, ws, C)
    ref = window_reverse(ctx, ws, H, W)
    if shift:
        ref = torch.roll(ref, (shift, shift), (1, 2))
    _close(got, ref.reshape(B * H * W, C), dtype, scale=1.0, n_ulp=6.0)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shift,H,W", [(0, 9, 11), (4, 18, 22), (4, 12, 40), (0, 36, 44)])
def test_swin_window_attn_zero_padded_windows(built_lib, dtype, shift, H, W):
    """DonutSwinLayer.maybe_pad (donut/encoder.py:591-596) + crop (:657-659): grids that are not multiples of the window run on a
    zero-padded grid — pad tokens are Linear(0) = the QKV bias, the shift mask is the padded grid's, pad query rows are dropped."""
    from oracle.layout_oracle import relative_position_index, shift_attn_mask, window_partition, window_reverse
    from surya_b200 import ops

    g = torch.Generator().manual_seed(5)
    B, nh, hd, ws = 2, 8, 32, 8
    C = nh * hd
    qkv = torch.randn(B * H * W, 3 * C, generator=g).to(dtype)
    qb = (0.3 * torch.randn(3 * C, generator=g)).to(dtype).float()
    table = (0.5 * torch.randn((2 * ws - 1) ** 2, nh, generator=g)).to(dtype)
    got = ops.swin_window_attn(qkv.cuda(), table.cuda(), B, H, W, nh, shift, qkv_bias=qb.cuda())
    Hp, Wp = (H + 7) // 8 * 8, (W + 7) // 8 * 8
    x = qb.to(dtype).expand(B, Hp, Wp, 3 * C).clone()
    x[:, :H, :W] = qkv.view(B, H, W, 3 * C)
    if shift:
        x = torch.roll(x, (-shift, -shift), (1, 2))
    win = window_partition(x, ws).view(-1, ws * ws, 3, nh, hd)
    q, k, v = (win[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    s = (q.float() @ k.float().transpose(-1, -2)).to(dtype)
    s = (s.float() / math.sqrt(hd)).to(dtype)
    bias = table[relative_position_index(ws).view(-1)].view(ws * ws, ws * ws, nh).permute(2, 0, 1)
    s = (s.float() + bias.float()).to(dtype)
    if shift:
        mask = shift_attn_mask(Hp, Wp, ws, shift, dtype)
        s = (s.view(B, -1, nh, 64, 64).float() + mask.float()[None, :, None]).to(dtype).view(-1, nh, 64, 64)
    p = torch.softmax(s.float(), -1).to(dtype)
    ctx = (p.float() @ v.float()).to(dtype).permute(0, 2, 1, 3).reshape(-1, ws, ws, C)
    ref = window_reverse(ctx, ws, Hp, Wp)
    if shift:
        ref = torch.roll(ref, (shift, shift), (1, 2))
    ref = ref[:, :H, :W].reshape(B * H * W, C)
    _close(got, ref, dtype, scale=1.0, n_ulp=6.0)
    with pytest.raises(Exception, match="QKV bias"):
        ops.swin_window_attn(qkv.cuda(), table.cuda(), B, H, W, nh, shift)
    with pytest.raises(Exception, match="smaller than the 8x8 window"):
        ops.swin_window_attn(qkv[: B * 6 * 16].cuda(), table.cuda(), B, 6, 16, nh, 0, qkv_bias=qb.cuda())


@pytest.mark.parametrize("dtype", DTYPES)
def test_bbox_embed_sum(built_lib, dtype):
    from oracle.layout_oracle import bbox_embedding
    from surya_b200 import ops
    from surya_b200.config import AdetrConfig
    from surya_b200.synth import LAYOUT_EMBED_TABLES, adetr_layout_state_dict

    d = AdetrConfig(num_hidden_layers=1)
    sd = {k: v.to(dtype) for k, v in adetr_layout_state_dict(d, 0).items() if "embed_tokens" in k}
    g = torch.Generator().manual_seed(4)
    boxes = torch.randint(0, 1025, (19, 7), generator=g)
    boxes[:, 6] = torch.randint(0, d.label_count, (19,), generator=g)
    boxes[0] = d.bos_token_id
    ref = bbox_embedding(sd, d, boxes.unsqueeze(1))[:, 0]
    tables = [sd[f"model.embed_tokens.{t}_embed.weight"].cuda() for t in list(LAYOUT_EMBED_TABLES) + ["label"]]
    got = ops.bbox_embed_sum(boxes.cuda(), tables, d.hidden_size, d.bbox_size, dtype)
    _close(got, ref, dtype, scale=ref.abs().max().item(), n_ulp=4.0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_attn_single_query(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator().manual_seed(5)
    B, nh, nkv, hd, Lk = 3, 16, 4, 64, 200
    q = torch.randn(B, nh * hd, generator=g).to(dtype)
    kv = torch.randn(B * Lk, 2 * nkv * hd, generator=g).to(dtype)
    got = ops.attn_single_query(q.cuda(), kv.cuda(), Lk, nh, nkv, hd, hd ** -0.5)
    K = kv.view(B, Lk, 2, nkv, hd)[:, :, 0].permute(0, 2, 1, 3).repeat_interleave(nh // nkv, 1).float()
    V = kv.view(B, Lk, 2, nkv, hd)[:, :, 1].permute(0, 2, 1, 3).repeat_interleave(nh // nkv, 1).float()
    ref = F.scaled_dot_product_attention(q.view(B, nh, 1, hd).float(), K, V, scale=hd ** -0.5).reshape(B, nh * hd)
    _close(got, ref, dtype, scale=1.0, n_ulp=3.0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_geglu_gemm(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator().manual_seed(6)
    M, K, I = 24, 1024, 4096
    x = torch.randn(M, K, generator=g).to(dtype)
    gate, up = (0.03 * torch.randn(I, K, generator=g)).to(dtype), (0.03 * torch.randn(I, K, generator=g)).to(dtype)
    w = torch.stack([gate, up], 1).reshape(2 * I, K)
    got = ops.gemm(x.cuda(), w.cuda(), act="gelu_tanh", swiglu=True)
    gg = (x.float() @ gate.float().T).to(dtype)
    uu = (x.float() @ up.float().T).to(dtype)
    ref = (F.gelu(gg.float(), approximate="tanh").to(dtype).float() * uu.float()).to(dtype)
    _close(got, ref, dtype, scale=1.0, n_ulp=4.0)


def _tiny():
    from surya_b200.config import layout_tiny
    from surya_b200.synth import adetr_layout_state_dict, layout_synthetic_pages, swin_state_dict

    cfg = layout_tiny()
    g = torch.load(GOLDEN / "layout_tiny.pt")
    sde, sdd = swin_state_dict(cfg.encoder, 0), adetr_layout_state_dict(cfg.decoder, 0)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=g["meta"]["page_seed"])
    return cfg, g, sde, sdd, x


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 2e-2), (torch.bfloat16, 1.5e-1)])
def test_swin_encoder_vs_reference_golden(built_lib, dtype, tol):
    from surya_b200.layout import LayoutEngine

    cfg, g, sde, sdd, x = _tiny()
    eng = LayoutEngine(cfg, sde, sdd, dtype=dtype)
    enc = eng.encode(x.cuda()).float().cpu()
    ref = g["encoder"]
    err = (enc - ref).abs().max().item()
    rel = ((enc - ref).norm() / ref.norm()).item()
    print(f"swin encoder {dtype}: max abs err {err:.4g} (ref max {ref.abs().max():.3g}), rel fro {rel:.3g}")
    assert err < tol * ref.abs().max().item() and rel < tol / 4


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-2), (torch.bfloat16, 6e-2)])
def test_swin_encoder_window_padding_vs_reference_golden(built_lib, dtype, tol):
    """288x352 input: token grids 36x44, 18x22 and 9x11 are not multiples of the 8x8 window, so the reference pads them
    (donut/encoder.py:591-596).  Engine (C++ loop) and the op-by-op path vs the reference's own output, and bit-identical to each
    other."""
    from surya_b200.config import LayoutConfig, SwinConfig, table_decoder
    from surya_b200.layout import LayoutEngine
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict

    g = torch.load(GOLDEN / "swin_window_padding.pt")
    enc_cfg = SwinConfig(image_size=tuple(g["meta"]["image_size"]), depths=(2, 2, 2, 2), encoder_length=99)
    cfg = LayoutConfig(encoder=enc_cfg, decoder=table_decoder(2))
    sde, sdd = swin_state_dict(enc_cfg, g["meta"]["seed"]), adetr_table_state_dict(cfg.decoder, g["meta"]["seed"])
    x = layout_synthetic_pages(1, enc_cfg.image_size, seed=g["meta"]["page_seed"])
    assert abs(float(x.double().sum()) - float(g["input_checksum"])) < 1e-6
    ref = g["encoder"]
    outs = []
    for impl in ("native", "ops"):
        eng = LayoutEngine(cfg, sde, sdd, dtype=dtype, impl=impl)
        enc = eng.encode(x.cuda())
        outs.append(enc)
        encf = enc.float().cpu()
        err = (encf - ref).abs().max().item()
        rel = ((encf - ref).norm() / ref.norm()).item()
        print(f"swin encoder with window padding, {impl}, {dtype}: max abs err {err:.4g} (ref max {ref.abs().max():.3g}), rel fro {rel:.3g}")
        assert enc.shape == (1, 99, 1024)
        assert err < tol * ref.abs().max().item() and rel < tol / 4
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-2), (torch.bfloat16, 6e-2)])
def test_adetr_decoder_teacher_forced_vs_golden(built_lib, dtype, tol):
    """Feed the reference's own box tokens and encoder states; bbox / class outputs must match per step."""
    from surya_b200.layout import LayoutEngine

    cfg, g, sde, sdd, x = _tiny()
    d = cfg.decoder
    eng = LayoutEngine(cfg, sde, sdd, dtype=dtype)
    enc = g["encoder"].to(dtype).cuda()
    eng.setup_cache(2)
    boxes = torch.full((2, 7), d.bos_token_id, dtype=torch.int64, device="cuda")
    worst_b = worst_c = 0.0
    for s in range(g["meta"]["steps"]):
        bbox, cls = eng.decode_step(boxes, enc, s)
        worst_b = max(worst_b, (bbox.cpu() - g["bbox"][:, s]).abs().max().item())
        worst_c = max(worst_c, (cls.cpu() - g["class_logits"][:, s]).abs().max().item())
        boxes = g["tokens"][:, s].cuda()
    print(f"adetr decoder {dtype}: bbox err {worst_b:.4g}, class-logit err {worst_c:.4g} (scale {g['class_logits'].abs().max():.3g})")
    assert worst_b < tol and worst_c < tol * max(1.0, g["class_logits"].abs().max().item())


def test_layout_greedy_matches_oracle_in_same_dtype(built_lib):
    """Free-running greedy decode (encoder on the GPU too).  Box tokens are trunc(sigmoid * 1024), so a 1e-3 difference
    moves a pixel and the two trajectories part; the check is therefore step-wise: the fp32 oracle is teacher-forced with
    the tokens the engine actually chose (and the engine's encoder states) and must agree with every step's outputs, and
    the engine's tokens must be exactly what its own outputs imply."""
    from oracle import layout_oracle as L
    from surya_b200.layout import B200LayoutModel, LayoutEngine, layout_greedy

    cfg, g, sde, sdd, x = _tiny()
    d = cfg.decoder
    eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16)
    steps = g["meta"]["steps"]
    tok, bbox, cls, enc = layout_greedy(eng, x.cuda(), steps)
    tok, bbox_c, cls_c = tok.cpu(), bbox.cpu(), cls.cpu()
    assert torch.equal(tok[..., :6], (bbox_c * d.bbox_size).to(torch.long)) and torch.equal(tok[..., 6], cls_c.argmax(-1))
    st = L.AdetrState(d.num_hidden_layers)
    sd32 = {k: v.to(torch.float16).float() for k, v in sdd.items()}
    boxes = torch.full((2, 1, 7), d.bos_token_id, dtype=torch.long)
    with torch.inference_mode():
        for s in range(steps):
            rb, rc = L.adetr_forward(sd32, d, boxes, enc.float().cpu(), torch.tensor([s]), st)
            assert (rb[:, -1] - bbox_c[:, s]).abs().max().item() < 5e-3, s
            assert (rc[:, -1] - cls_c[:, s]).abs().max().item() < 2e-2, s
            boxes = tok[:, s].unsqueeze(1)
    # first step has no trajectory dependence: compare with the reference golden directly
    assert (tok[:, 0, :6] - g["tokens"][:, 0, :6]).abs().max().item() <= 3 and torch.equal(tok[:, 0, 6], g["tokens"][:, 0, 6])
    # the mirror of LayoutPredictor's model surface drives the same engine
    model = B200LayoutModel(eng)
    enc2 = model.encoder(pixel_values=x.cuda())[0]
    assert torch.equal(enc2, enc)
    model.decoder.model._setup_cache(model.config, 2, model.device, model.dtype)
    boxes = torch.full((2, 1, 7), d.bos_token_id, dtype=torch.long, device="cuda")
    out = model.decoder(input_boxes=boxes, encoder_hidden_states=enc2, cache_position=torch.arange(1, device="cuda"),
                        use_cache=True, prefill=True)
    assert torch.equal(out["bbox_logits"][:, 0].float(), bbox[:, 0])
    assert out["class_logits"].shape == (2, 1, d.label_count)


def test_layout_default_config_runs(built_lib):
    """BASELINE config 4 shape: batch 16 of 768x768 pages through the full-depth Swin (2,2,16,2) + 8-layer decoder; checks
    batch invariance (same page alone vs inside a batch) bit-for-bit."""
    from surya_b200.config import layout_default
    from surya_b200.layout import LayoutEngine, layout_greedy
    from surya_b200.synth import adetr_layout_state_dict, layout_synthetic_pages, swin_state_dict

    cfg = layout_default()
    eng = LayoutEngine(cfg, swin_state_dict(cfg.encoder, 0), adetr_layout_state_dict(cfg.decoder, 0), dtype=torch.float16)
    x = layout_synthetic_pages(16, cfg.encoder.image_size, seed=3).cuda()
    tok3, bb3, cl3, enc3 = layout_greedy(eng, x, 4)
    assert enc3.shape == (16, 576, 1024) and torch.isfinite(enc3.float()).all()
    tok1, bb1, cl1, enc1 = layout_greedy(eng, x[1:2], 4)
    assert torch.equal(enc1[0], enc3[1])
    assert torch.equal(tok1[0], tok3[1])


def test_layout_default_config_vs_oracle(built_lib):
    """BASELINE config 4 (layout half) against the CPU oracle at the DEFAULT config: Swin (2,2,16,2) at 768x768 + 8-layer ADETR
    decoder, 2 pages x 16 greedy steps.  Encoder states vs the fp32 oracle; decoder step-wise: the oracle (fp32 math on the
    fp16-rounded weights) is teacher-forced with the tokens the engine chose and its encoder states, and must agree with every
    step's bbox / class outputs; the engine's tokens must be what its own outputs imply."""
    from oracle import layout_oracle as L
    from surya_b200.config import layout_default
    from surya_b200.layout import LayoutEngine, layout_greedy
    from surya_b200.synth import adetr_layout_state_dict, layout_synthetic_pages, swin_state_dict

    cfg = layout_default()
    d = cfg.decoder
    sde, sdd = swin_state_dict(cfg.encoder, 0), adetr_layout_state_dict(d, 0)
    eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=5)
    steps = 16
    tok, bbox, cls, enc = layout_greedy(eng, x.cuda(), steps)
    tok, bbox_c, cls_c = tok.cpu(), bbox.cpu(), cls.cpu()
    torch.set_num_threads(max(1, min(64, len(__import__("os").sched_getaffinity(0)))))
    with torch.inference_mode():
        ref_enc = L.swin_forward(sde, cfg.encoder, x)
    rel = ((enc.float().cpu() - ref_enc).norm() / ref_enc.norm()).item()
    mx = (enc.float().cpu() - ref_enc).abs().max().item() / ref_enc.abs().max().item()
    assert rel < 5e-3 and mx < 2e-2, (rel, mx)
    assert torch.equal(tok[..., :6], (bbox_c * d.bbox_size).to(torch.long)) and torch.equal(tok[..., 6], cls_c.argmax(-1))
    st = L.AdetrState(d.num_hidden_layers)
    sd32 = {k: v.to(torch.float16).float() for k, v in sdd.items()}
    boxes = torch.full((2, 1, 7), d.bos_token_id, dtype=torch.long)
    worst_b = worst_c = 0.0
    with torch.inference_mode():
        for s in range(steps):
            rb, rc = L.adetr_forward(sd32, d, boxes, enc.float().cpu(), torch.tensor([s]), st)
            worst_b = max(worst_b, (rb[:, -1] - bbox_c[:, s]).abs().max().item())
            worst_c = max(worst_c, (rc[:, -1] - cls_c[:, s]).abs().max().item())
            boxes = tok[:, s].unsqueeze(1)
    print(f"layout default: encoder rel {rel:.3g} max/absmax {mx:.3g}; decoder bbox err {worst_b:.3g}, class err {worst_c:.3g}")
    assert worst_b < 5e-3 and worst_c < 3e-2, (worst_b, worst_c)


def test_table_default_config_vs_oracle(built_lib):
    """BASELINE config 4 (table_rec half), DEFAULT config: Swin (2,2,12,2) at 768x768 + 6-layer decoder, 2 pages, 3-token query
    prompt + 16 greedy steps, same step-wise protocol as the layout test (five property heads, predictor token formation)."""
    from oracle import layout_oracle as L
    from surya_b200.config import table_default
    from surya_b200.layout import LayoutEngine, table_greedy
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    cfg = table_default()
    d = cfg.decoder
    sde, sdd = swin_state_dict(cfg.encoder, 0), adetr_table_state_dict(d, 0)
    eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=6)
    prompt = table_query_tokens(d, 2)
    steps = 16
    tok, done, heads, enc = table_greedy(eng, x.cuda(), prompt, steps)
    tok_c = tok.cpu()
    torch.set_num_threads(max(1, min(64, len(__import__("os").sched_getaffinity(0)))))
    with torch.inference_mode():
        ref_enc = L.swin_forward(sde, cfg.encoder, x)
    rel = ((enc.float().cpu() - ref_enc).norm() / ref_enc.norm()).item()
    assert rel < 5e-3, rel
    sd32 = {k: v.to(torch.float16).float() for k, v in sdd.items()}
    st = L.AdetrState(d.num_hidden_layers)
    ids, pos = prompt.clone(), torch.arange(prompt.shape[1])
    worst = {}
    with torch.inference_mode():
        for s in range(steps):
            ref = L.adetr_forward(sd32, d, ids, enc.float().cpu(), pos, st)
            pos = pos[-1:] + 1
            for k in ref:
                worst[k] = max(worst.get(k, 0.0), (ref[k][:, -1] - heads[k][:, s].cpu()).abs().max().item())
            ref_tok, ref_done = L.table_next_tokens({k: heads[k][:, s:s + 1].cpu() for k in heads}, d)
            assert torch.equal(ref_tok, tok_c[:, s]) and torch.equal(ref_done, done[:, s].cpu().bool())
            ids = tok_c[:, s].unsqueeze(1)
    print("table default: encoder rel %.3g; head errs %s" % (rel, {k: round(v, 5) for k, v in worst.items()}))
    assert all(v < 3e-2 for v in worst.values()), worst


# ------------------------------------------------------------------------------------------------ table_rec
@pytest.mark.parametrize("dtype", DTYPES)
def test_label_embed(built_lib, dtype):
    from oracle.layout_oracle import label_embedding
    from surya_b200 import ops
    from surya_b200.config import table_decoder
    from surya_b200.synth import adetr_table_state_dict

    d = table_decoder(1)
    sd = {k: v.to(dtype) for k, v in adetr_table_state_dict(d, 0).items() if "embed_tokens" in k}
    g = torch.Generator().manual_seed(7)
    boxes = torch.randint(0, 1025, (21, 10), generator=g)
    boxes[:, 6] = torch.randint(0, 15, (21,), generator=g)
    boxes[:, 7] = torch.randint(0, 14, (21,), generator=g)
    boxes[0] = d.bos_token_id
    boxes[1] = d.query_end_token_id
    ref = label_embedding(sd, d, boxes.unsqueeze(1))[:, 0]
    order = ["w", "h", "cx", "cy", "xskew", "yskew", "x1", "y1", "x3", "y3", "category", "merge", "colspan"]
    tables = [sd[f"model.embed_tokens.{t}_embed.weight"].cuda() for t in order]
    got = ops.label_embed(boxes.cuda(), tables, d.box_embed_size, d.property_embed_size, d.bbox_size, d.vocab_size, dtype)
    assert torch.equal(got.cpu(), ref), (got.cpu().float() - ref.float()).abs().max()


def test_box_next_token(built_lib):
    from oracle.layout_oracle import table_next_tokens
    from surya_b200 import ops
    from surya_b200.config import table_decoder

    d = table_decoder(1)
    g = torch.Generator().manual_seed(8)
    B = 37
    out = {"bbox": torch.rand(B, 1, 6, generator=g).half().float(), "category": torch.randn(B, 1, 10, generator=g),
           "merges": torch.randn(B, 1, 9, generator=g), "colspan": (3 * torch.randn(B, 1, 1, generator=g)).half().float(),
           "is_header": torch.randn(B, 1, 7, generator=g)}
    out["bbox"][0, 0, 0] = 1.0
    out["colspan"][1, 0, 0] = 2.5     # round-half-even -> 2
    out["colspan"][2, 0, 0] = 3.5     # -> 4
    out["category"][3, 0, 1] = 50.0   # eos -> done
    out["category"][4, 0, :] = 0.25   # tie -> first index (pad) -> done
    ref_tok, ref_done = table_next_tokens(out, d)
    dev = {k: v[:, 0].contiguous().cuda() for k, v in out.items()}
    tok, done = ops.box_next_token(dev["bbox"], [dev["category"], dev["merges"], dev["colspan"], dev["is_header"]], [0, 0, 1, 0],
                                   d.bbox_size, done_head=0, eos=d.eos_token_id, pad=d.pad_token_id)
    assert torch.equal(tok.cpu(), ref_tok) and torch.equal(done.cpu().bool(), ref_done)


def _table_tiny():
    from surya_b200.config import table_tiny
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    cfg = table_tiny()
    g = torch.load(GOLDEN / "table_tiny.pt")
    sde, sdd = swin_state_dict(cfg.encoder, 1), adetr_table_state_dict(cfg.decoder, 1)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=g["meta"]["page_seed"])
    return cfg, g, sde, sdd, x, table_query_tokens(cfg.decoder, 2)


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-2), (torch.bfloat16, 6e-2)])
def test_table_decoder_teacher_forced_vs_golden(built_lib, dtype, tol):
    """Reference encoder states + reference tokens in, five property heads out, per step (prompt prefill included)."""
    from surya_b200.layout import LayoutEngine

    cfg, g, sde, sdd, x, prompt = _table_tiny()
    eng = LayoutEngine(cfg, sde, sdd, dtype=dtype)
    enc = g["encoder"].to(dtype).cuda()
    eng.setup_cache(2)
    out = eng.decode_prompt(prompt.cuda(), enc, 0)
    worst = {k: 0.0 for k in g["heads"]}
    for s in range(g["meta"]["steps"]):
        for k in worst:
            worst[k] = max(worst[k], (out[k].cpu() - g["heads"][k][:, s]).abs().max().item())
        out = eng.decode_step(g["tokens"][:, s].cuda(), enc, prompt.shape[1] + s)
    print(f"table decoder {dtype}: " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    for k, v in worst.items():
        assert v < tol * max(1.0, g["heads"][k].abs().max().item()), (k, v)


def test_table_greedy_stepwise_vs_oracle_and_model_surface(built_lib):
    from oracle import layout_oracle as L
    from surya_b200.layout import B200TableRecModel, LayoutEngine, table_greedy

    cfg, g, sde, sdd, x, prompt = _table_tiny()
    d = cfg.decoder
    eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16)
    steps = g["meta"]["steps"]
    tok, done, heads, enc = table_greedy(eng, x.cuda(), prompt, steps)
    tok_c = tok.cpu()
    enc_err = (enc.float().cpu() - g["encoder"]).abs().max().item()
    assert enc_err < 2e-2 * g["encoder"].abs().max().item()
    # oracle teacher-forced with the engine's own tokens and encoder states
    sd32 = {k: v.to(torch.float16).float() for k, v in sdd.items()}
    st = L.AdetrState(d.num_hidden_layers)
    ids, pos = prompt.clone(), torch.arange(prompt.shape[1])
    with torch.inference_mode():
        for s in range(steps):
            ref = L.adetr_forward(sd32, d, ids, enc.float().cpu(), pos, st)
            pos = pos[-1:] + 1
            for k in ref:
                assert (ref[k][:, -1] - heads[k][:, s].cpu()).abs().max().item() < 2e-2, (k, s)
            ref_tok, ref_done = L.table_next_tokens({k: heads[k][:, s:s + 1].cpu() for k in heads}, d)
            assert torch.equal(ref_tok, tok_c[:, s]) and torch.equal(ref_done, done[:, s].cpu().bool())
            ids = tok_c[:, s].unsqueeze(1)
    assert (tok_c[:, 0, :6] - g["tokens"][:, 0, :6]).abs().max().item() <= 3 and torch.equal(tok_c[:, 0, 6], g["tokens"][:, 0, 6])
    # predictor-facing surface
    model = B200TableRecModel(eng)
    e2 = model.encoder(pixel_values=x.cuda()).last_hidden_state
    assert torch.equal(e2, enc)
    model.decoder.model._setup_cache(model.config, 2, model.device, model.dtype)
    out = model.decoder(input_ids=prompt.cuda(), encoder_hidden_states=e2, cache_position=torch.arange(3, device="cuda"),
                        use_cache=True, prefill=True)["box_property_logits"]
    assert set(out) == {"bbox", "category", "merges", "colspan", "is_header"}
    assert torch.equal(out["bbox"][:, -1].float(), heads["bbox"][:, 0])


def test_table_default_config_runs(built_lib):
    """BASELINE config 4, table half: batch 16 of 768x768 through Swin (2,2,12,2) + 6-layer decoder; batch invariance."""
    from surya_b200.config import table_default
    from surya_b200.layout import LayoutEngine, table_greedy
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    cfg = table_default()
    eng = LayoutEngine(cfg, swin_state_dict(cfg.encoder, 0), adetr_table_state_dict(cfg.decoder, 0), dtype=torch.float16)
    x = layout_synthetic_pages(16, cfg.encoder.image_size, seed=4).cuda()
    tok, done, heads, enc = table_greedy(eng, x, table_query_tokens(cfg.decoder, 16), 4)
    assert enc.shape == (16, 576, 1024) and torch.isfinite(enc.float()).all() and tok.shape == (16, 4, 10)
    tok1, _, _, enc1 = table_greedy(eng, x[5:6], table_query_tokens(cfg.decoder, 1), 4)
    assert torch.equal(enc1[0], enc[5]) and torch.equal(tok1[0], tok[5])


@pytest.mark.parametrize("kind", ["layout", "table"])
def test_graph_replayed_loop_equals_eager_loop(built_lib, kind):
    """run_loop: one CUDA graph per decode step (device-side token feedback, position advance, history append) must give
    bit-identical tokens and head outputs to launching the same kernels eagerly, also when the graph is reused for a second
    batch of pages."""
    from surya_b200.layout import LayoutEngine, layout_greedy, table_greedy

    if kind == "layout":
        cfg, g, sde, sdd, x = _tiny()
        run = lambda eng, px, graph: layout_greedy(eng, px, 9, use_graph=graph)[:3]
    else:
        cfg, g, sde, sdd, x, prompt = _table_tiny()

        def run(eng, px, graph):
            tok, done, heads, _ = table_greedy(eng, px, prompt, 9, use_graph=graph)
            return (tok, done) + tuple(heads[k] for k in sorted(heads))
    eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16)
    x = x.cuda()
    x2 = torch.flip(x, dims=[0]).contiguous()
    eager = [t.clone() for t in run(eng, x, False)]
    eager2 = [t.clone() for t in run(eng, x2, False)]
    graph = [t.clone() for t in run(eng, x, True)]
    graph2 = [t.clone() for t in run(eng, x2, True)]      # replays the graph captured by the previous call
    for a, b in zip(eager + eager2, graph + graph2):
        assert torch.equal(a, b)
    assert not torch.equal(graph[0], graph2[0])


@pytest.mark.parametrize("kind", ["layout", "table"])
def test_native_engine_equals_op_by_op_path(built_lib, kind):
    """sb_layout_encode / sb_layout_decode (layer loops, caches and the decode loop in C++) vs the same kernels launched op by
    op from Python: encoder states, tokens and head outputs must be bit-identical, with and without graphs."""
    from surya_b200.layout import LayoutEngine

    if kind == "layout":
        cfg, g, sde, sdd, x = _tiny()
        prompt = torch.full((2, 1, 7), cfg.decoder.bos_token_id, dtype=torch.int64, device="cuda")
    else:
        cfg, g, sde, sdd, x, prompt = _table_tiny()
        prompt = prompt.cuda()
    nat = LayoutEngine(cfg, sde, sdd, dtype=torch.float16, impl="native", max_batch=4)
    ref = LayoutEngine(cfg, sde, sdd, dtype=torch.float16, impl="ops")
    assert nat.workspace_bytes > 0
    x = x.cuda()
    enc_n, enc_p = nat.encode(x), ref.encode(x)
    assert torch.equal(enc_n, enc_p)
    # batch larger than max_batch is cut into chunks by the binding
    x6 = torch.cat([x, x, x], 0)
    assert torch.equal(nat.encode(x6), torch.cat([enc_n, enc_n, enc_n], 0))
    steps = 11
    want = [t.clone() for t in _flatten(ref.run_loop(enc_p, prompt, steps, use_graph=False))]
    for use_graph in (False, True, True):
        got = _flatten(nat.run_loop(enc_n, prompt, steps, use_graph=use_graph))
        for a, b in zip(got, want):
            assert torch.equal(a, b)
    nat.close()


def _flatten(res):
    tok, bbox, heads, done = res
    return [tok, bbox] + list(heads) + [done]


def test_nonsquare_encoder_and_cellpass_prompt_vs_reference_golden(built_lib):
    """256x512 input (non-square Swin grid) and a 7-token table_rec cell-pass prompt, both against the second reference
    fixture: encoder states, then the heads of the first generated position after the multi-token prompt."""
    from oracle import layout_oracle as L
    from surya_b200.config import LayoutConfig, SwinConfig, table_decoder
    from surya_b200.layout import LayoutEngine
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict

    g = torch.load(GOLDEN / "table_nonsquare_cellpass.pt")
    enc_cfg = SwinConfig(image_size=tuple(g["meta"]["image_size"]), depths=(2, 2, 2, 2), encoder_length=128)
    cfg = LayoutConfig(encoder=enc_cfg, decoder=table_decoder(2))
    sde, sdd = swin_state_dict(enc_cfg, g["meta"]["seed"]), adetr_table_state_dict(cfg.decoder, g["meta"]["seed"])
    x = layout_synthetic_pages(2, enc_cfg.image_size, seed=g["meta"]["page_seed"])
    rows, ref = g["encoder_rows"], g["encoder"]          # the fixture keeps a seeded half of the encoder rows
    full = L.swin_forward(sde, enc_cfg, x)               # decoder input: the oracle's states, pinned to the reference rows
    assert (full.reshape(-1, full.shape[-1])[rows] - ref).abs().max().item() < 1e-5
    for impl in ("native", "ops"):
        eng = LayoutEngine(cfg, sde, sdd, dtype=torch.float16, impl=impl, max_batch=2)
        enc = eng.encode(x.cuda())
        got = enc.float().cpu().reshape(-1, enc.shape[-1])[rows]
        rel = ((got - ref).norm() / ref.norm()).item()
        assert tuple(enc.shape) == g["encoder_shape"] and rel < 5e-3, (impl, rel)
        tok, bbox, heads, done = eng.run_loop(full.to(torch.float16).cuda(), g["prompt"].cuda(), 1, use_graph=False)
        got = {"bbox": bbox[0], "category": heads[0][0], "merges": heads[1][0], "colspan": heads[2][0], "is_header": heads[3][0]}
        for k, v in got.items():
            err = (v.cpu() - g["heads"][k][:, 0]).abs().max().item()
            assert err < 1e-2 * max(1.0, g["heads"][k].abs().max().item()), (impl, k, err)
        eng.close()
