"""CPU tests: oracle pinned to the reference goldens, host-side planning logic vs the oracle's restatement of the
reference index math, and the C-ABI library's exported surface (no compute calls without a GPU)."""
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"


def test_library_exports_every_declared_symbol(built_lib):
    from surya_b200 import _lib

    lib = _lib.load(require_cuda=False)
    names = _lib.header_symbols()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in include/surya_b200.h but not exported: {missing}"
    assert lib.sb_version() >= 1


def test_product_fails_loudly_without_gpu(built_lib):
    from surya_b200 import _lib

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.SuryaB200Error):
        _lib.load(require_cuda=True)


def test_product_never_imports_oracle():
    import re

    for f in (ROOT / "surya_b200").rglob("*.py"):
        text = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f"{f} imports the test oracle"


def _golden_crops(kind):
    from oracle.make_golden import golden_crops

    return golden_crops(kind)


def test_oracle_pinned_to_reference_golden_tiny():
    """oracle/rec_oracle.py (fp32) reproduces the reference modules' logits, boxes and tokens."""
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.synth import rec_state_dict

    g = torch.load(GOLDEN / "rec_tiny.pt")
    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    batch = O.build_batch(_golden_crops("tiny"), cfg)
    assert torch.equal(batch["input_ids"], g["input_ids"])
    assert torch.equal(torch.from_numpy(batch["grid_thw"]), g["grid_thw"])
    assert abs(batch["image_tiles"].double().sum().item() - g["tiles_checksum"].item()) < 1e-6
    tok, sc, box, logits = O.greedy_decode(sd, cfg, batch, g["meta"]["steps"], torch.float32, return_logits=True)
    assert (logits - g["logits"]).abs().max().item() < 2e-5
    assert torch.equal(tok, g["tokens"])
    # boxes are trunc(sigmoid * bbox_size): identical except where the reference's own value sits within fp32 noise of an integer
    d = box != g["boxes"]
    frac = g["bbox"] * cfg.bbox_size
    assert ((box - g["boxes"]).abs() <= 1).all() and ((frac - frac.round()).abs()[d] < 1e-3).all() and int(d.sum()) <= 2
    assert (sc - g["score"]).abs().max().item() < 1e-6


def test_oracle_pinned_to_reference_golden_synrec():
    from oracle import rec_oracle as O
    from surya_b200.config import syn_rec
    from surya_b200.synth import rec_state_dict

    g = torch.load(GOLDEN / "rec_synrec.pt")
    cfg = syn_rec()
    sd = rec_state_dict(cfg, seed=0)
    batch = O.build_batch(_golden_crops("synrec"), cfg)
    assert batch["input_ids"].shape == (2, 46) and batch["image_tiles"].shape == (320, 588)
    assert tuple(batch["grid_thw"][0]) == (1, 4, 40)
    tok, sc, box, logits = O.greedy_decode(sd, cfg, batch, g["meta"]["steps"], torch.float32, return_logits=True)
    assert (logits[..., g["logit_idx"]] - g["logit_sample"]).abs().max().item() < 5e-5
    assert torch.equal(tok, g["tokens"])
    assert torch.equal(box, g["boxes"])


def test_tiling_and_prompt_match_oracle():
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import prompt_tokens, scale_to_fit, tile_image
    from surya_b200.synth import rec_synthetic_crops

    cfg = tiny_rec()
    for hw, seed in (((48, 512), 1), ((40, 300), 2), ((64, 900), 3), ((300, 1500), 4)):
        crop = rec_synthetic_crops(1, hw[0], hw[1], seed=seed)[0]
        img = np.asarray(crop, dtype=np.float32)
        a = O.scale_to_fit(img)
        b = scale_to_fit(img)
        assert np.array_equal(a, b)
        t_ref, g_ref = O.process_and_tile(a)
        t, g = tile_image(b)
        assert g == g_ref and np.array_equal(t, t_ref.numpy())
        batch = O.build_batch([crop], cfg)
        assert np.array_equal(prompt_tokens(cfg, t.shape[0] // 4), batch["input_ids"][0].numpy())


@pytest.mark.parametrize("grids", [[(1, 4, 40)], [(1, 4, 40), (1, 6, 22), (1, 10, 66)], [(1, 2, 2), (1, 18, 74)]])
def test_prefill_plan_matches_reference_index_math(grids):
    """build_prefill_plan vs the oracle's restatement of rot_pos_emb / get_window_index / masked_scatter order."""
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import build_prefill_plan, prompt_tokens

    cfg = tiny_rec()
    e = cfg.vision_encoder
    g = np.array(grids, dtype=np.int64)
    seqs = [prompt_tokens(cfg, int(h * w) // 4) for _, h, w in grids]
    plan = build_prefill_plan(cfg, g, seqs, slots=list(range(len(grids))))
    ints = plan.ints.numpy()

    def arr(name):
        o, n = plan.off[name]
        return ints[o:o + n]

    n = int((g[:, 1] * g[:, 2]).sum())
    widx, cu_win = O.vision_window_index(g, e.window_size, e.spatial_merge_size, e.patch_size)
    pos = O.vision_rot_pos_ids(g, e.spatial_merge_size)
    rows = np.arange(n).reshape(n // 4, 4)
    assert np.array_equal(arr("patch_perm"), rows[widx].reshape(-1))
    assert np.array_equal(arr("pos_rc").reshape(-1, 2), pos.reshape(n // 4, 4, 2)[widx].reshape(-1, 2))
    assert np.array_equal(np.concatenate([arr("win_start"), [n]]), cu_win)
    assert np.array_equal(arr("win_start") + arr("win_len"), cu_win[1:])
    cu_full = np.concatenate([[0], np.cumsum(g[:, 1] * g[:, 2])])
    assert np.array_equal(arr("img_start"), cu_full[:-1]) and np.array_equal(arr("img_len"), np.diff(cu_full))
    # scatter order + learned 2-D embedding indices, checked through the reference formula on random tables
    gen = torch.Generator().manual_seed(0)
    H = cfg.hidden_size
    sd = {"img_h_embed.weight": torch.randn(1024, H, generator=gen), "img_w_embed.weight": torch.randn(1024, H, generator=gen)}
    feats_win = torch.randn(n // 4, H, generator=gen)                      # merger output, window order
    ref = feats_win[torch.argsort(torch.from_numpy(widx))] + O.learned_2d_embeddings(sd, cfg, g)
    ids = np.concatenate(seqs)
    is_img = ids == cfg.image_token_id
    fr, hi, wi = arr("feat_row")[is_img], arr("hidx")[is_img], arr("widx")[is_img]
    got = feats_win[torch.from_numpy(fr.astype(np.int64))] + (sd["img_h_embed.weight"][torch.from_numpy(hi.astype(np.int64))]
                                                              + sd["img_w_embed.weight"][torch.from_numpy(wi.astype(np.int64))])
    assert torch.allclose(got, ref, atol=1e-6)
    assert (arr("feat_row")[~is_img] == -1).all()
    # ragged token layout
    lens = np.array([len(s) for s in seqs])
    assert np.array_equal(arr("seq_len"), lens)
    assert np.array_equal(arr("last_tok"), np.cumsum(lens) - 1)
    assert np.array_equal(arr("tok_pos"), np.concatenate([np.arange(x) for x in lens]))


def test_weight_packing_layout():
    from surya_b200.config import align, tiny_rec
    from surya_b200.recognition import pack_rec_weights
    from surya_b200.synth import rec_state_dict

    cfg = tiny_rec()
    sd = rec_state_dict(cfg, seed=0)
    w = pack_rec_weights(sd, cfg, torch.bfloat16, "cpu")
    e, d = cfg.vision_encoder, cfg.decoder
    assert len(w) == 15 + 10 * e.depth + 5 * d.num_hidden_layers
    assert w[0].shape == (e.hidden_size, align(e.patch_dim, 8)) and (w[0][:, e.patch_dim:] == 0).all()
    gu = w[15 + 6]
    ip = align(e.intermediate_size, 8)
    assert gu.shape == (2 * ip, e.hidden_size)
    assert torch.equal(gu[0::2][: e.intermediate_size], sd["vision_encoder.blocks.0.mlp.gate_proj.weight"].to(torch.bfloat16))
    assert torch.equal(gu[1::2][: e.intermediate_size], sd["vision_encoder.blocks.0.mlp.up_proj.weight"].to(torch.bfloat16))
    assert (gu[2 * e.intermediate_size:] == 0).all()
    qkv = w[15 + 10 * e.depth + 0]
    assert qkv.shape == ((d.num_attention_heads + 2 * d.num_key_value_heads) * d.head_dim, d.hidden_size)
    # decoder RMSNorm weights are folded into the consuming GEMM's weight: W'[n, k] = bf16(bf16(W)[n, k] * bf16(g)[k])
    bf = torch.bfloat16
    g_in = sd["decoder.layers.0.input_layernorm.weight"].to(bf).float()
    q0 = sd["decoder.layers.0.self_attn.q_proj.weight"].to(bf).float()
    assert torch.equal(qkv[: q0.shape[0]], (q0 * g_in[None, :]).to(bf))
    g_f = sd["decoder.norm.weight"].to(bf).float()
    assert torch.equal(w[7], (sd["embedder.token_embed.weight"].to(bf).float() * g_f[None, :]).to(bf))       # SB_RW_LM_W
    assert torch.equal(w[8], sd["embedder.token_embed.weight"].to(bf))                                        # SB_RW_EMBED
    assert torch.equal(w[10], (sd["bbox_head.weight"].to(bf).float() * g_f[None, :]).to(bf))                  # SB_RW_BBOX_W


def test_detect_repeat_token_matches_oracle():
    from oracle.rec_oracle import detect_repeat_token as ref
    from surya_b200.recognition import detect_repeat_token as got

    rng = np.random.default_rng(0)
    for _ in range(200):
        n = int(rng.integers(1, 90))
        k = int(rng.integers(1, 8))
        toks = rng.integers(0, k, size=n).tolist()
        assert got(toks) == ref(toks)
    assert got([7] * 40) and not got([7] * 39)


def test_det_oracle_pinned_to_reference_golden():
    from oracle import det_oracle as D
    from surya_b200.config import det_default
    from surya_b200.synth import det_normalize, det_state_dict, det_synthetic_pages

    g = torch.load(GOLDEN / "det_default.pt")
    cfg = det_default()
    sd = det_state_dict(cfg, seed=0)
    x = det_normalize(det_synthetic_pages(1, 512, seed=11, text_like=True))
    assert abs(x.double().sum().item() - g["input_checksum"].item()) < 1e-3
    got = D.forward(sd, cfg, x)
    assert (got - g["logits"]).abs().max().item() < 1e-5


def test_det_program_structure():
    from surya_b200.config import det_default
    from surya_b200.detection import OP_CLS, OP_CONV, OP_MLA, OP_STEM, pack_det_program, plan_buffers
    from surya_b200.synth import det_state_dict

    cfg = det_default()
    prog = pack_det_program(det_state_dict(cfg, 0), cfg, torch.float16, "cpu")
    kinds = [o["op"] for o in prog.ops]
    assert kinds[0] == OP_STEM and kinds[-1] == OP_CLS
    assert kinds.count(OP_MLA) == cfg.depths[-1] and kinds.count(OP_CONV) == 6
    caps = plan_buffers(prog, 1024, 1024)
    names = prog.buf_names
    assert caps[names.index("feat0")] == 256 * 256 * 64 and caps[names.index("feat3")] == 32 * 32 * 512
    assert caps[names.index("cat")] == 256 * 256 * 512
    # BN folding is exact in fp32: folded 1x1 conv == conv + BN on random input
    import torch.nn.functional as F
    from surya_b200.detection import _fold
    from surya_b200.det_arch import det_blocks
    sd = det_state_dict(cfg, 0)
    c = det_blocks(cfg)[3].convs[1]
    w, b = _fold(sd, c)
    x = torch.randn(2, c.cin, 5, 5)
    n = f"{c.name}.norm"
    ref = F.batch_norm(F.conv2d(x, sd[c.wkey]), sd[f"{n}.running_mean"], sd[f"{n}.running_var"], sd[f"{n}.weight"], sd[f"{n}.bias"], False, 0.0, c.eps)
    assert torch.allclose(F.conv2d(x, w, b), ref, atol=1e-4)


def test_layout_oracle_pinned_to_reference_golden():
    """oracle/layout_oracle.py (fp32) reproduces the reference Swin encoder + ADETR decoder bit-for-bit on the seeded case."""
    from oracle import layout_oracle as L
    from surya_b200.config import layout_tiny
    from surya_b200.synth import adetr_layout_state_dict, layout_synthetic_pages, swin_state_dict

    g = torch.load(GOLDEN / "layout_tiny.pt")
    cfg = layout_tiny()
    sde, sdd = swin_state_dict(cfg.encoder, 0), adetr_layout_state_dict(cfg.decoder, 0)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=g["meta"]["page_seed"])
    assert abs(x.double().sum().item() - g["input_checksum"].item()) < 1e-3
    tok, enc, bl, cl = L.layout_greedy(sde, sdd, cfg, x, g["meta"]["steps"], return_logits=True)
    assert (enc - g["encoder"]).abs().max().item() < 1e-5
    assert (bl - g["bbox"]).abs().max().item() < 1e-5
    assert (cl - g["class_logits"]).abs().max().item() < 1e-4
    assert torch.equal(tok, g["tokens"])


def test_layout_weight_packing():
    from surya_b200.config import layout_tiny
    from surya_b200.layout import _sincos_table
    from oracle.layout_oracle import sincos_2d

    assert torch.equal(_sincos_table(16, 12, 256), sincos_2d(16, 12, 256)[0])
    cfg = layout_tiny()
    assert cfg.encoder.hidden_size == 1024 and cfg.encoder.grid == (64, 64)


def test_table_oracle_pinned_to_reference_golden():
    """oracle (fp32) == reference table_rec encoder + decoder on the seeded case, incl. the 3-token prompt prefill."""
    from oracle import layout_oracle as L
    from surya_b200.config import table_tiny
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict, table_query_tokens

    g = torch.load(GOLDEN / "table_tiny.pt")
    cfg = table_tiny()
    sde, sdd = swin_state_dict(cfg.encoder, 1), adetr_table_state_dict(cfg.decoder, 1)
    x = layout_synthetic_pages(2, cfg.encoder.image_size, seed=g["meta"]["page_seed"])
    tok, done, enc, heads = L.table_greedy(sde, sdd, cfg, x, table_query_tokens(cfg.decoder, 2), g["meta"]["steps"])
    assert (enc - g["encoder"]).abs().max().item() < 1e-5
    for k, v in g["heads"].items():
        assert (heads[k] - v).abs().max().item() < 1e-4, k
    assert torch.equal(tok, g["tokens"])


def test_layout_weight_table_matches_the_c_abi_layout():
    """LayoutEngine._weight_table order / count vs the SB_LW_* layout in include/surya_b200.h (what sb_layout_create checks)."""
    import re

    from surya_b200.config import layout_tiny, table_tiny
    from surya_b200.layout import LayoutEngine
    from surya_b200.synth import adetr_layout_state_dict, adetr_table_state_dict, swin_state_dict

    hdr = (ROOT / "include" / "surya_b200.h").read_text()
    def enum_size(last):      # value of the trailing enumerator = number of entries before it
        body = re.search(r"enum \{([^}]*\b%s\b)[^}]*\}" % last, hdr).group(1)
        return len([x for x in body.split(",") if x.strip()]) - 1

    n_fixed, n_layer, n_dec, n_tail = enum_size("SB_LW_ENC_FIXED"), enum_size("SB_LW_ENC_LAYER"), enum_size("SB_LW_DEC_LAYER"), enum_size("SB_LW_DEC_TAIL")
    assert (n_fixed, n_layer, n_dec, n_tail) == (5, 13, 12, 4)
    for cfg, sdd, tables, heads in ((layout_tiny(), adetr_layout_state_dict, 15, 3), (table_tiny(), adetr_table_state_dict, 13, 5)):
        eng = LayoutEngine.__new__(LayoutEngine)          # pack on the CPU without creating the CUDA engine
        import surya_b200.layout as LM
        orig = LM._lib.load
        LM._lib.load = lambda *a, **k: None
        try:
            LayoutEngine.__init__(eng, cfg, swin_state_dict(cfg.encoder, 0), sdd(cfg.decoder, 0), device="cpu", impl="ops")
        finally:
            LM._lib.load = orig
        w = eng._weight_table()
        e, d = cfg.encoder, cfg.decoder
        want = n_fixed + sum(1 + dep * n_layer for dep in e.depths) + 3 * (len(e.depths) - 1) + tables + d.num_hidden_layers * n_dec + n_tail + heads
        assert len(w) == want
        assert w[0].shape == (e.embed_dim, 64) and w[4].shape == (e.encoder_length, e.hidden_size)
        assert w[5].shape == (e.grid[0] * e.grid[1], e.embed_dim)                      # stage-0 sin-cos table
        assert w[5 + 1 + 2].shape == (3 * e.embed_dim, e.embed_dim)                     # fused qkv of the first layer
        assert w[-heads].shape[0] == 6                                                  # bbox head first


def test_prefill_plan_random_grids_property():
    """Randomised ragged batches: window permutation is a permutation, windows tile the patch range, image segments follow the
    grids, and every image token reads a distinct merged-feature row — checked against the oracle's index math."""
    from oracle import rec_oracle as O
    from surya_b200.config import tiny_rec
    from surya_b200.recognition import build_prefill_plan, prompt_tokens

    cfg = tiny_rec()
    e = cfg.vision_encoder
    rng = np.random.default_rng(7)
    for _ in range(25):
        n = int(rng.integers(1, 6))
        grids = [(1, int(2 * rng.integers(1, 10)), int(2 * rng.integers(1, 38))) for _ in range(n)]
        g = np.array(grids, dtype=np.int64)
        seqs = [prompt_tokens(cfg, int(h * w) // 4) for _, h, w in grids]
        slots = list(rng.permutation(16)[:n])
        plan = build_prefill_plan(cfg, g, seqs, slots=[int(s) for s in slots])
        ints = plan.ints.numpy()
        arr = lambda name: ints[plan.off[name][0]: plan.off[name][0] + plan.off[name][1]]
        total = int((g[:, 1] * g[:, 2]).sum())
        perm = arr("patch_perm")
        assert sorted(perm.tolist()) == list(range(total))
        widx, cu_win = O.vision_window_index(g, e.window_size, e.spatial_merge_size, e.patch_size)
        assert np.array_equal(perm, np.arange(total).reshape(total // 4, 4)[widx].reshape(-1))
        assert np.array_equal(np.concatenate([arr("win_start"), [total]]), cu_win) and (arr("win_len") > 0).all()
        assert int(arr("win_len").sum()) == total and int(arr("img_len").sum()) == total
        ids = np.concatenate(seqs)
        fr = arr("feat_row")[ids == cfg.image_token_id]
        assert sorted(fr.tolist()) == list(range(total // 4))
        lens = np.array([len(s) for s in seqs])
        assert np.array_equal(arr("tok_slot"), np.repeat(np.array(slots, dtype=np.int64), lens))


def test_pooled_preprocess_equals_serial():
    from surya_b200 import recognition as R
    from surya_b200.config import tiny_rec
    from surya_b200.synth import rec_synthetic_crops

    class _E:
        cfg = tiny_rec()

    r = R.RecognitionRunner.__new__(R.RecognitionRunner)
    r.engine = _E()
    crops = list(rec_synthetic_crops(24, 48, 512, seed=1)) + list(rec_synthetic_crops(8, 40, 300, seed=2))
    a, b = r.preprocess(crops, workers=1), r.preprocess(crops, workers=4)
    assert a[1] == b[1]
    assert all(np.array_equal(x, y) for x, y in zip(a[0], b[0])) and all(np.array_equal(x, y) for x, y in zip(a[2], b[2]))


def test_oracle_pinned_nonsquare_swin_and_cellpass_prompt():
    """Second table_rec fixture from the reference: 256x512 input (non-square windows / sin-cos order / shift masks) and a
    7-token cell-pass prompt (query + 4 column boxes) prefilled in one call."""
    from oracle import layout_oracle as L
    from surya_b200.config import LayoutConfig, SwinConfig, table_decoder
    from surya_b200.synth import adetr_table_state_dict, layout_synthetic_pages, swin_state_dict

    g = torch.load(GOLDEN / "table_nonsquare_cellpass.pt")
    enc_cfg = SwinConfig(image_size=tuple(g["meta"]["image_size"]), depths=(2, 2, 2, 2), encoder_length=128)
    cfg = LayoutConfig(encoder=enc_cfg, decoder=table_decoder(2))
    sde, sdd = swin_state_dict(enc_cfg, g["meta"]["seed"]), adetr_table_state_dict(cfg.decoder, g["meta"]["seed"])
    x = layout_synthetic_pages(2, enc_cfg.image_size, seed=g["meta"]["page_seed"])
    tok, done, enc, heads = L.table_greedy(sde, sdd, cfg, x, g["prompt"], g["meta"]["steps"])
    assert enc.shape == g["encoder_shape"] == (2, 128, 1024)
    assert (enc.reshape(2 * 128, -1)[g["encoder_rows"]] - g["encoder"]).abs().max().item() < 1e-5
    for k, v in g["heads"].items():
        assert (heads[k] - v).abs().max().item() < 1e-4, k
    assert torch.equal(tok, g["tokens"])


def test_oracle_pinned_swin_window_padding():
    """Oracle's maybe_pad branch (zero-padded windows, padded-size shift mask, crop) vs the reference's Swin encoder on a 288x352
    input whose later stages (36x44, 18x22, 9x11 tokens) are not multiples of the 8x8 window."""
    from oracle import layout_oracle as L
    from surya_b200.config import SwinConfig
    from surya_b200.synth import layout_synthetic_pages, swin_state_dict

    g = torch.load(GOLDEN / "swin_window_padding.pt")
    enc_cfg = SwinConfig(image_size=tuple(g["meta"]["image_size"]), depths=(2, 2, 2, 2), encoder_length=99)
    sde = swin_state_dict(enc_cfg, g["meta"]["seed"])
    x = layout_synthetic_pages(1, enc_cfg.image_size, seed=g["meta"]["page_seed"])
    enc = L.swin_forward(sde, enc_cfg, x)
    assert enc.shape == g["encoder"].shape == (1, 99, 1024)
    assert (enc - g["encoder"]).abs().max().item() < 1e-5


def test_committed_bench_lines_follow_the_contract():
    """The bench lines committed under profiles/ carry every key the driver's contract names (schema guard for bench.py)."""
    import json

    for name in ("r01_final_bench_n1.json", "r01_final_bench_n2.json", "r01_final_bench_n4.json", "r02_final_bench_n1.json",
                 "r02_final_bench_n2_nocpu.json", "r02_final_bench_n4_nocpu.json", "r02b_final_bench_n1.json"):
        line = [l for l in (ROOT / "profiles" / name).read_text().splitlines() if l.startswith("{")][-1]   # NCCL prints a banner first
        d = json.loads(line)
        if "nocpu" in name:
            d.setdefault("cpu_baseline", None)
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                  "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
            assert k in d, (name, k)
        assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
        assert "workload" in d["config"] and d["steps"] >= 1 and d["warmup"] >= 3 and d["gpu_launches"] > 0
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
        assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
        if d["n_gpus"] == 1:
            assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
            assert d["roofline"]["traffic"] is not None
