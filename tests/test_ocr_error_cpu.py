"""ocr_error (SURVEY §8 f4), CPU side: the oracle against the reference's own DistilBertForSequenceClassification (golden fixture
written by oracle/make_golden.py), the host pack plan, and the op sequence of surya_b200/ocr_error.py replayed over torch stand-ins
for the C-ABI ops (wiring / index check only — the kernels themselves are compared on the GPU in test_ocr_error_gpu.py)."""
import math
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ocr_error_oracle as E
from surya_b200 import _lib
from surya_b200 import ocr_error as OE
from surya_b200.config import ocr_error_default, ocr_error_tiny
from surya_b200.synth import ocr_error_state_dict, ocr_error_synthetic_batch

GOLDEN = Path(__file__).parent / "golden"


@pytest.mark.parametrize("kind", ["tiny", "default"])
def test_ocr_error_oracle_pinned_to_reference_golden(kind):
    g = torch.load(GOLDEN / f"ocr_error_{kind}.pt")
    cfg = ocr_error_tiny() if kind == "tiny" else ocr_error_default()
    sd = ocr_error_state_dict(cfg, seed=0)
    ids, mask = ocr_error_synthetic_batch(cfg, g["meta"]["n"], g["meta"]["max_len"], seed=g["meta"]["seed"])
    assert torch.equal(ids, g["input_ids"]) and torch.equal(mask, g["attention_mask"])
    logits, hidden = E.forward(sd, cfg, ids, mask, return_hidden=True)
    assert (logits - g["logits"]).abs().max().item() < 2e-5
    assert (hidden[:, 0] - g["cls_hidden"]).abs().max().item() < 2e-5
    assert torch.equal(logits.argmax(1), g["labels"])
    assert 0 < int(g["labels"].sum()) < g["labels"].numel()          # both labels occur: the label check is not vacuous


def test_pack_plan():
    cfg = ocr_error_tiny()
    ids, mask = ocr_error_synthetic_batch(cfg, 7, 33, seed=5)
    plan = OE.build_pack_plan(ids.numpy(), mask.numpy(), cfg)
    lens = mask.sum(1).numpy()
    assert plan["n_tok"] == lens.sum() and plan["max_len"] == 33 and plan["batch"] == 7
    assert np.array_equal(plan["seq_len"], lens) and np.array_equal(plan["seq_start"], np.concatenate([[0], np.cumsum(lens)[:-1]]))
    for b in range(7):
        s, n = plan["seq_start"][b], lens[b]
        assert np.array_equal(plan["ids"][s:s + n], ids[b, :n].numpy()) and np.array_equal(plan["pos"][s:s + n], np.arange(n))
    assert OE.build_pack_plan(np.zeros((0, 5), np.int64), None, cfg)["n_tok"] == 0
    no_mask = OE.build_pack_plan(ids.numpy(), None, cfg)
    assert no_mask["n_tok"] == ids.numel()
    bad = mask.clone(); bad[2, 1] = 0                                    # a hole
    with pytest.raises(_lib.SuryaB200Error, match="right-padded prefix"):
        OE.build_pack_plan(ids.numpy(), bad.numpy(), cfg)
    empty = mask.clone(); empty[3] = 0
    with pytest.raises(_lib.SuryaB200Error, match="all-zero attention_mask"):
        OE.build_pack_plan(ids.numpy(), empty.numpy(), cfg)
    big = ids.clone(); big[0, 1] = cfg.vocab_size
    with pytest.raises(_lib.SuryaB200Error, match="token id"):
        OE.build_pack_plan(big.numpy(), mask.numpy(), cfg)
    with pytest.raises(_lib.SuryaB200Error, match="max_position_embeddings"):
        OE.build_pack_plan(np.ones((1, cfg.max_position_embeddings + 1), np.int64), None, cfg)


class _TorchOps:
    """fp32 torch stand-ins with the call signatures of surya_b200.ops (test infrastructure)."""

    @staticmethod
    def embed_pos_layernorm(ids, pos, word, ptab, w, b, eps):
        return F.layer_norm(word[ids.long()] + ptab[pos.long()], (word.shape[1],), w, b, eps)

    @staticmethod
    def gemm(a, w, bias=None, residual=None, act="none"):
        y = F.linear(a, w, bias)
        y = {"none": lambda t: t, "gelu": F.gelu, "relu": F.relu}[act](y)
        return y + residual if residual is not None else y

    @staticmethod
    def attn_varlen(q, k, v, seq_start, seq_len, max_len, nh, nkv, hd, causal, scale):
        assert not causal and nh == nkv and int(seq_len.max()) <= max_len
        out = torch.zeros(q.shape[0], nh * hd)
        for s, n in zip(seq_start.tolist(), seq_len.tolist()):
            qs, ks, vs = (t[s:s + n].reshape(n, nh, hd).transpose(0, 1) for t in (q, k, v))
            p = torch.softmax(qs @ ks.transpose(1, 2) * scale, dim=-1)
            out[s:s + n] = (p @ vs).transpose(0, 1).reshape(n, nh * hd)
        return out

    @staticmethod
    def layernorm(x, w, b, eps):
        return F.layer_norm(x, (x.shape[1],), w, b, eps)

    @staticmethod
    def gather_pad_rows(src, perm, Kp, dtype):
        assert Kp == src.shape[1]
        return src[perm.long()]

    @staticmethod
    def small_head(x, w, b, sigmoid=True, box_scale=None):
        assert not sigmoid
        return F.linear(x, w, b), None


def test_op_sequence_matches_oracle_over_torch_standins(monkeypatch):
    cfg = ocr_error_tiny()
    sd = ocr_error_state_dict(cfg, seed=0)
    ids, mask = ocr_error_synthetic_batch(cfg, 6, 40, seed=3)
    m = object.__new__(OE.B200DistilBert)                       # no CUDA here: bypass the constructor's device checks
    m.config = m.cfg = cfg
    m.dtype, m.device = torch.float32, torch.device("cpu")
    m.w = OE.pack_ocr_error_weights(cfg, sd, torch.float32, "cpu")
    m._upload = lambda arr: torch.from_numpy(arr)
    monkeypatch.setattr(OE, "ops", _TorchOps)
    out = m(ids, attention_mask=mask).logits
    ref = E.forward(sd, cfg, ids, mask)
    assert (out - ref).abs().max().item() < 2e-5
    monkeypatch.setattr(OE.B200DistilBert, "forward_packed", lambda self, plan: E.forward(
        sd, cfg, *_unpack(plan, cfg)))
    labels = OE.detect_errors(m, ids, mask, batch_size=4)
    assert labels == [OE.ID2LABEL[int(i)] for i in ref.argmax(1)]


def _unpack(plan, cfg):
    B, L = plan["batch"], plan["max_len"]
    ids = np.full((B, L), cfg.pad_token_id, np.int64)
    mask = np.zeros((B, L), np.int64)
    for b in range(B):
        s, n = plan["seq_start"][b], plan["seq_len"][b]
        ids[b, :n], mask[b, :n] = plan["ids"][s:s + n], 1
    return torch.from_numpy(ids), torch.from_numpy(mask)


def test_reference_ocr_error_predictor_dropin_cpu():
    """Labels of the reference's UNMODIFIED OCRErrorPredictor over its own DistilBertForSequenceClassification (stored in
    tests/golden/reference_host.pt by oracle/make_golden.py) against surya_b200.ocr_error.detect_errors over the B200DistilBert
    mirror for the same texts, batches of 3 with a ragged tail (the network behind the mirror is the CPU oracle here)."""
    from oracle.make_golden import ocr_error_texts

    g = torch.load(GOLDEN / "reference_host.pt")["ocr_error"]
    cfg = ocr_error_tiny()
    sd = ocr_error_state_dict(cfg, seed=0)
    texts = ocr_error_texts()
    assert texts == g["texts"]
    mirror = object.__new__(OE.B200DistilBert)
    mirror.config = mirror.cfg = cfg
    mirror.dtype, mirror.device = torch.float32, torch.device("cpu")
    mirror.forward_packed = lambda plan: E.forward(sd, cfg, *_unpack(plan, cfg))
    tok = E.HashTokenizer(cfg)(texts)
    labels = OE.detect_errors(mirror, tok.input_ids, tok.attention_mask, batch_size=g["batch_size"])
    assert labels == g["labels"]
    assert len(set(labels)) == 2, labels
