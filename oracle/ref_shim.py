"""ORACLE TOOLING (golden regeneration only) — import the *unmodified* reference surya from a checkout named by SURYA_REFERENCE.

The reference pins transformers ^4.51 (pyproject.toml:15); this image has 5.5.  The few names that moved are
patched *in transformers' namespace before import* (SURVEY.md §8c); no reference source is copied or edited.
The tests never import the reference: what they compare against is stored under tests/golden/ by oracle/make_golden.py.
"""
from __future__ import annotations

import os
import sys
import types
from pathlib import Path

REFERENCE = Path(os.environ.get("SURYA_REFERENCE", "")).expanduser()


def available() -> bool:
    try:
        return bool(os.environ.get("SURYA_REFERENCE")) and (REFERENCE / "surya" / "__init__.py").is_file()
    except OSError:
        return False


def install() -> None:
    if not available():
        raise RuntimeError("set SURYA_REFERENCE to a checkout of the reference surya (VikParuchuri/surya@80e9a7e) to regenerate goldens")
    if str(REFERENCE) not in sys.path:
        sys.path.insert(0, str(REFERENCE))
    import torch
    import transformers
    import transformers.cache_utils as cu
    import transformers.pytorch_utils as pu
    from transformers.modeling_rope_utils import ROPE_INIT_FUNCTIONS

    # (1) cache classes used only in isinstance checks (decoder/__init__.py:7-12, 509-510)
    for name in ("SlidingWindowCache", "StaticCache"):
        if not hasattr(cu, name):
            setattr(cu, name, type(name, (), {}))
    # (2) pruning helpers imported by donut/encoder.py:12-16 (only used by prune_heads)
    for name in ("find_pruneable_heads_and_indices", "prune_linear_layer"):
        if not hasattr(pu, name):
            setattr(pu, name, lambda *a, **k: (_ for _ in ()).throw(NotImplementedError(name)))
    # (3) classic RoPE init (decoder/__init__.py:333)
    if "default" not in ROPE_INIT_FUNCTIONS:
        def _default_rope(config, device=None, seq_len=None, **kw):
            base = config.rope_theta
            dim = getattr(config, "head_dim", None) or config.hidden_size // config.num_attention_heads
            inv = 1.0 / (base ** (torch.arange(0, dim, 2, dtype=torch.int64).to(device=device, dtype=torch.float) / dim))
            return inv, 1.0
        ROPE_INIT_FUNCTIONS["default"] = _default_rope
    # (7) surya.ocr_error (SURVEY §8 f4): config.py:5 imports transformers.onnx.OnnxConfig (removed in 5.x; only subclassed by an
    # export helper) and tokenizer.py:9 imports three unicode helpers that moved to transformers.tokenization_python
    if "transformers.onnx" not in sys.modules:
        try:
            __import__("transformers.onnx")
        except Exception:
            onnx = types.ModuleType("transformers.onnx")
            onnx.OnnxConfig = type("OnnxConfig", (), {})
            sys.modules["transformers.onnx"] = onnx
    import transformers.tokenization_utils as tu
    try:
        import transformers.tokenization_python as tp
        for name in ("_is_control", "_is_punctuation", "_is_whitespace"):
            if not hasattr(tu, name) and hasattr(tp, name):
                setattr(tu, name, getattr(tp, name))
    except Exception:
        pass
    # (6) optional host deps of surya.input that are absent in this image
    for mod in ("pypdfium2", "filetype"):
        if mod not in sys.modules:
            try:
                __import__(mod)
            except Exception:
                sys.modules[mod] = types.ModuleType(mod)


def build_reference_rec_model(cfg, state_dict, attn: str = "sdpa"):
    """Instantiate the reference SuryaModel for our RecConfig and load the synthetic weights (fp32, eval)."""
    install()
    import torch
    from surya.common.surya import SuryaModel
    from surya.common.surya.config import SuryaModelConfig

    e, d = cfg.vision_encoder, cfg.decoder
    enc = dict(depth=e.depth, hidden_size=e.hidden_size, intermediate_size=e.intermediate_size, num_heads=e.num_heads,
               in_channels=e.in_channels, patch_size=e.patch_size, spatial_merge_size=e.spatial_merge_size,
               spatial_patch_size=e.patch_size, temporal_patch_size=e.temporal_patch_size, window_size=e.window_size,
               out_hidden_size=e.out_hidden_size, fullatt_block_indexes=tuple(e.fullatt_block_indexes))
    dec = dict(vocab_size=cfg.vocab_size, hidden_size=d.hidden_size, intermediate_size=d.intermediate_size,
               num_hidden_layers=d.num_hidden_layers, num_attention_heads=d.num_attention_heads,
               num_key_value_heads=d.num_key_value_heads, rope_theta=d.rope_theta, rms_norm_eps=d.rms_norm_eps,
               pad_token_id=cfg.pad_token_id, bos_token_id=cfg.bos_token_id, eos_token_id=cfg.eos_token_id)
    mc = SuryaModelConfig(vocab_size=cfg.vocab_size, bbox_size=cfg.bbox_size, bos_token_id=cfg.bos_token_id,
                          eos_token_id=cfg.eos_token_id, pad_token_id=cfg.pad_token_id,
                          image_token_id=cfg.image_token_id, vision_encoder=enc, decoder=dec,
                          register_token_ids=tuple(cfg.register_token_ids),
                          num_register_tokens=cfg.num_register_tokens,
                          image_embed_encoding_size=cfg.image_embed_encoding_size,
                          image_embed_encoding_multiplier=cfg.image_embed_encoding_multiplier)
    mc.vision_encoder._attn_implementation = attn
    mc.decoder._attn_implementation = attn
    model = SuryaModel(mc)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    missing = [m for m in missing if "rotary" not in m and "inv_freq" not in m]
    assert not missing and not unexpected, (missing, unexpected)
    return model.eval()


def build_reference_layout_models(cfg, sd_enc, sd_dec):
    """Instantiate the reference DonutSwinLayoutModel + SuryaLayoutDecoder (surya/layout/model/{encoder,decoder}.py) for
    our LayoutConfig with the synthetic weights (fp32, eval).  Two transformers-5 incompatibilities are neutralised on the
    reference's base classes (no behaviour on the forward path): weight tying hooks and get_head_mask."""
    install()
    from surya.common.adetr.decoder import SuryaADETRDecoderPreTrainedModel
    from surya.common.donut.encoder import DonutSwinPreTrainedModel
    from surya.layout.model.config import DonutSwinLayoutConfig, SuryaLayoutDecoderConfig
    from surya.layout.model.decoder import SuryaLayoutDecoder
    from surya.layout.model.encoder import DonutSwinLayoutModel

    SuryaADETRDecoderPreTrainedModel.tie_weights = lambda self, **k: None
    SuryaADETRDecoderPreTrainedModel._tie_weights = lambda self, **k: None
    DonutSwinPreTrainedModel.get_head_mask = lambda self, head_mask, n, *a, **k: [None] * n
    e, d = cfg.encoder, cfg.decoder
    enc = DonutSwinLayoutModel(DonutSwinLayoutConfig(image_size=e.image_size, depths=list(e.depths),
                                                     encoder_length=e.encoder_length)).eval()
    miss, unexp = enc.load_state_dict(sd_enc, strict=False)
    assert not [m for m in miss if "relative_position_index" not in m] and not unexp, (miss, unexp)
    dec = SuryaLayoutDecoder(SuryaLayoutDecoderConfig(num_hidden_layers=d.num_hidden_layers)).eval()
    miss, unexp = dec.load_state_dict(sd_dec, strict=False)
    assert not miss and not unexp, (miss, unexp)
    return enc, dec


def build_reference_table_models(cfg, sd_enc, sd_dec):
    """Reference DonutSwinModel + SuryaTableRecDecoder (surya/table_rec/model/{encoder,decoder}.py) with synthetic weights."""
    install()
    from surya.common.adetr.decoder import SuryaADETRDecoderPreTrainedModel
    from surya.common.donut.encoder import DonutSwinPreTrainedModel
    from surya.table_rec.model.config import DonutSwinTableRecConfig, SuryaTableRecDecoderConfig
    from surya.table_rec.model.decoder import SuryaTableRecDecoder
    from surya.table_rec.model.encoder import DonutSwinModel

    SuryaADETRDecoderPreTrainedModel.tie_weights = lambda self, **k: None
    SuryaADETRDecoderPreTrainedModel._tie_weights = lambda self, **k: None
    DonutSwinPreTrainedModel.get_head_mask = lambda self, head_mask, n, *a, **k: [None] * n
    e, d = cfg.encoder, cfg.decoder
    enc = DonutSwinModel(DonutSwinTableRecConfig(image_size=e.image_size, depths=list(e.depths),
                                                 encoder_length=e.encoder_length)).eval()
    miss, unexp = enc.load_state_dict(sd_enc, strict=False)
    assert not [m for m in miss if "relative_position_index" not in m] and not unexp, (miss, unexp)
    dec = SuryaTableRecDecoder(SuryaTableRecDecoderConfig(num_hidden_layers=d.num_hidden_layers)).eval()
    miss, unexp = dec.load_state_dict(sd_dec, strict=False)
    assert not miss and not unexp, (miss, unexp)
    return enc, dec


def build_reference_det_model(cfg, state_dict):
    """Reference EfficientViTForSemanticSegmentation (surya/detection/model/encoderdecoder.py) with the synthetic weights."""
    install()
    from surya.detection.model.config import EfficientViTConfig
    from surya.detection.model.encoderdecoder import EfficientViTForSemanticSegmentation

    m = EfficientViTForSemanticSegmentation(EfficientViTConfig()).eval()
    missing, unexpected = m.load_state_dict(state_dict, strict=False)
    assert not [k for k in missing if "num_batches_tracked" not in k] and not unexpected, (missing, unexpected)
    return m


def build_reference_ocr_error_model(cfg, state_dict):
    """Reference DistilBertForSequenceClassification (surya/ocr_error/model/encoder.py:697) with the synthetic weights, eager
    attention (the reference's CPU path).  get_head_mask left transformers' PreTrainedModel in 5.x: neutralised on the reference's
    base class like for Donut-Swin (the predictor never passes a head mask; None entries skip the multiply, encoder.py:182-183)."""
    install()
    from surya.ocr_error.model.config import DistilBertConfig
    from surya.ocr_error.model.encoder import DistilBertForSequenceClassification, DistilBertPreTrainedModel

    DistilBertPreTrainedModel.get_head_mask = lambda self, head_mask, n, *a, **k: [None] * n
    c = DistilBertConfig(vocab_size=cfg.vocab_size, max_position_embeddings=cfg.max_position_embeddings, n_layers=cfg.n_layers,
                         n_heads=cfg.n_heads, dim=cfg.dim, hidden_dim=cfg.hidden_dim, pad_token_id=cfg.pad_token_id,
                         num_labels=cfg.num_labels)
    c._attn_implementation = "eager"
    m = DistilBertForSequenceClassification(c).eval()
    missing, unexpected = m.load_state_dict(state_dict, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    return m
