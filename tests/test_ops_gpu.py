"""Kernel-level parity (GPU): each hand-written kernel vs a plain PyTorch fp32 restatement of the same op
with the storage-dtype roundings at the eager op boundaries.  Runs through the C ABI (ctypes)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

DT = [torch.bfloat16, torch.float16]


def _ulp(dtype):
    return 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11


def _close(got, ref, dtype, ulps=2.0, what="", scale=None):
    """|got - ref| <= ulps * ulp(max(|ref|, |scale|, 1)) elementwise; `scale` = magnitude of the largest rounded
    intermediate (a 1-ulp flip of an intermediate survives a cancelling residual add)."""
    got = got.float()
    ref = ref.float()
    mag = ref.abs().clamp(min=1.0)
    if scale is not None:
        mag = torch.maximum(mag, scale.float().abs())
    tol = ulps * 2.0 * _ulp(dtype) * torch.exp2(torch.floor(torch.log2(mag)))
    bad = (got - ref).abs() > tol
    frac = bad.float().mean().item()
    assert frac == 0.0, f"{what}: {bad.sum().item()} / {bad.numel()} beyond {ulps} ulp, max abs err {(got - ref).abs().max().item():.4g}"


def _act_ref(x, act):
    if act == "none":
        return x
    if act == "gelu":
        return torch.nn.functional.gelu(x)
    if act == "silu":
        return torch.nn.functional.silu(x)
    if act == "hardswish":
        return torch.nn.functional.hardswish(x)
    if act == "relu":
        return torch.relu(x)
    if act == "gelu_tanh":
        return torch.nn.functional.gelu(x, approximate="tanh")
    raise ValueError(act)


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize(
    "M,N,K,bn",
    [
        (128, 256, 64, 256), (128, 128, 128, 128), (256, 64, 1280, 64), (200, 96, 592, 32),
        (1000, 1280, 592, 0), (640, 3840, 1280, 0), (256, 1280, 3456, 0), (333, 520, 1280, 128),
        (4096, 1280, 1280, 256),
    ],
)
def test_gemm_plain(built_lib, dtype, M, N, K, bn):
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(dtype)
    out = ops.gemm(a, w, force_bn=bn)
    torch.cuda.synchronize()
    ref = (a.float() @ w.float().t()).to(dtype)
    _close(out, ref, dtype, what=f"gemm {M}x{N}x{K} bn={bn}")


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("act", ["none", "gelu", "silu", "hardswish", "relu", "gelu_tanh"])
def test_gemm_epilogue(built_lib, dtype, act):
    from surya_b200 import ops

    M, N, K = 300, 392, 320
    g = torch.Generator(device="cuda").manual_seed(11)
    a = (torch.randn(M, K, device="cuda", generator=g)).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.08).to(dtype)
    bias = torch.randn(N, device="cuda", generator=g).to(dtype).float()
    res = torch.randn(M, N, device="cuda", generator=g).to(dtype)
    out = ops.gemm(a, w, bias=bias, residual=res, act=act)
    torch.cuda.synchronize()
    lin = (a.float() @ w.float().t() + bias).to(dtype)
    y = _act_ref(lin.float(), act).to(dtype) if act != "none" else lin
    ref = (y.float() + res.float()).to(dtype)
    _close(out, ref, dtype, ulps=3.0, what=f"gemm epilogue {act}", scale=torch.maximum(lin.float().abs(), res.float().abs()))


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("M,N,K,act,res", [(80000, 1024, 256, "hardswish", False), (75011, 512, 128, "gelu", True),
                                           (76800, 256, 192, "relu", False)])
def test_gemm_short_k_activation_default_tile_equals_forced(built_lib, dtype, M, N, K, act, res):
    """Short-K GEMMs with an activation over many rows (detection's 1x1 expand convs): the default tile heuristic must give,
    bit for bit, what a forced 128 x 256 tile gives (same per-element arithmetic, same k order), and be right against the fp32
    restatement on a sample of rows."""
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M % 97 + N + K)
    a = torch.randn(M, K, device="cuda", generator=g).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.08).to(dtype)
    bias = torch.randn(N, device="cuda", generator=g).to(dtype).float()
    r = torch.randn(M, N, device="cuda", generator=g).to(dtype) if res else None
    out = ops.gemm(a, w, bias=bias, residual=r, act=act)
    forced = ops.gemm(a, w, bias=bias, residual=r, act=act, force_bn=256)
    torch.cuda.synchronize()
    assert torch.equal(out, forced)
    rows = torch.randint(0, M, (2048,), device="cuda", generator=g)
    lin = (a[rows].float() @ w.float().t() + bias).to(dtype)
    y = _act_ref(lin.float(), act).to(dtype)
    ref = (y.float() + r[rows].float()).to(dtype) if res else y
    _close(out[rows], ref, dtype, ulps=3.0, what=f"short-K gemm {act}", scale=lin.float().abs() if not res else torch.maximum(lin.float().abs(), r[rows].float().abs()))


@pytest.mark.parametrize("dtype", DT)
def test_gemm_swiglu(built_lib, dtype):
    from surya_b200 import ops

    M, I, K = 260, 216, 256  # N = 2*I interleaved
    g = torch.Generator(device="cuda").manual_seed(5)
    a = torch.randn(M, K, device="cuda", generator=g).to(dtype)
    wg = (torch.randn(I, K, device="cuda", generator=g) * 0.08).to(dtype)
    wu = (torch.randn(I, K, device="cuda", generator=g) * 0.08).to(dtype)
    bg = torch.randn(I, device="cuda", generator=g).to(dtype).float()
    bu = torch.randn(I, device="cuda", generator=g).to(dtype).float()
    w = torch.stack([wg, wu], dim=1).reshape(2 * I, K).contiguous()
    b = torch.stack([bg, bu], dim=1).reshape(2 * I).contiguous()
    out = ops.gemm(a, w, bias=b, act="silu", swiglu=True)
    torch.cuda.synchronize()
    gate = (a.float() @ wg.float().t() + bg).to(dtype)
    up = (a.float() @ wu.float().t() + bu).to(dtype)
    ref = (torch.nn.functional.silu(gate.float()).to(dtype).float() * up.float()).to(dtype)
    _close(out, ref, dtype, ulps=3.0, what="swiglu")


@pytest.mark.parametrize("dtype", DT)
def test_gemm_f32_out(built_lib, dtype):
    from surya_b200 import ops

    M, N, K = 130, 200, 192
    g = torch.Generator(device="cuda").manual_seed(9)
    a = torch.randn(M, K, device="cuda", generator=g).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.1).to(dtype)
    out = ops.gemm(a, w, out_f32=True)
    torch.cuda.synchronize()
    ref = a.float() @ w.float().t()
    assert (out - ref).abs().max().item() < 1e-3


@pytest.mark.parametrize("dtype", DT)
def test_rmsnorm(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(3)
    x = (torch.randn(77, 1280, device="cuda", generator=g) * 3).to(dtype)
    w = (1 + 0.1 * torch.randn(1280, device="cuda", generator=g)).to(dtype)
    out = ops.rmsnorm(x, w, eps=1e-6)
    xf = x.float()
    n = (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-6)).to(dtype)
    ref = w * n
    _close(out, ref, dtype, ulps=2.0, what="rmsnorm")
    rows = torch.tensor([5, 0, 76, 5], device="cuda", dtype=torch.int32)
    out2 = ops.rmsnorm(x, w, eps=1e-6, src_rows=rows)
    _close(out2, ref[rows.long()], dtype, ulps=2.0, what="rmsnorm gather")


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("M,N,K,swiglu,bias,res", [(256, 1920, 1280, False, True, False), (256, 6848, 1280, True, False, False),
                                                   (200, 1280, 592, False, False, True), (1000, 1920, 1280, False, True, False),
                                                   (37, 640, 320, False, True, False)])
def test_gemm_folded_rmsnorm(built_lib, dtype, M, N, K, swiglu, bias, res):
    """RMSNorm folded into the GEMM (sb_gemm_rmsnorm): C = epi(rs[m] * (x W'^T) + b).  (a) against the fp32 restatement with
    the output roundings; (b) the in-kernel 1/rms (decode path) and the row_rstd + rowscale path (prefill) must agree BIT FOR
    BIT, and both with an fp32 torch rsqrt to 2 ulp of fp32; (c) tiles wider / narrower than the default give the same bits."""
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M * 11 + N + K)
    x = (torch.randn(M, K, device="cuda", generator=g) * 1.5).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.03).to(dtype)
    b = (torch.randn(N, device="cuda", generator=g) * 0.1).to(dtype).float() if bias else None
    r = (torch.randn(M, N, device="cuda", generator=g) * 0.5).to(dtype) if res else None
    eps = 1e-6
    rs = ops.row_rstd(x, eps)
    rs_ref = torch.rsqrt(x.float().pow(2).mean(-1) + eps)
    assert ((rs - rs_ref).abs() <= 2e-6 * rs_ref.abs()).all()      # rsqrt.approx (2 ulp) + a different summation order
    got_inline = ops.gemm(x, w, bias=b, residual=r, act="silu" if swiglu else "none", swiglu=swiglu, rms_eps=eps)
    got_scale = ops.gemm(x, w, bias=b, residual=r, act="silu" if swiglu else "none", swiglu=swiglu, rowscale=rs)
    assert torch.equal(got_inline, got_scale), "in-kernel 1/rms and row_rstd path differ"
    if not swiglu and N % 128 == 0:
        assert torch.equal(ops.gemm(x, w, bias=b, residual=r, rowscale=rs, force_bn=128), got_scale)
        assert torch.equal(ops.gemm(x, w, bias=b, residual=r, rms_eps=eps, force_bn=64), got_scale)
    acc = (x.float() @ w.float().t()) * rs_ref[:, None]
    if b is not None:
        acc = acc + b
    lin = acc.to(dtype).float()
    if swiglu:
        gt, up = lin[:, 0::2], lin[:, 1::2]
        ref = (torch.nn.functional.silu(gt).to(dtype).float() * up).to(dtype)
    else:
        ref = lin if r is None else (lin + r.float())
        ref = ref.to(dtype)
    _close(got_inline, ref, dtype, ulps=2.0, what="folded rmsnorm gemm", scale=lin if r is not None else None)


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("M,N,K", [(256, 65792, 1280), (5, 1000, 320), (130, 4104, 640)])
def test_gemm_argmax_epilogue(built_lib, dtype, M, N, K):
    """lm_head with the online argmax epilogue: per-tile (max, first argmax, sum exp) partials reduce to exactly the argmax /
    max-softmax of the 16-bit logits the plain path writes (surya/recognition/__init__.py:294-324), ties resolved to the
    lowest index like torch.argmax; argmax_only must not touch C."""
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(N + K)
    x = (torch.randn(M, K, device="cuda", generator=g)).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.02).to(dtype)
    w[N // 3] = w[N // 7]                      # force exact ties between two columns
    b = (torch.randn(N, device="cuda", generator=g) * 0.02).to(dtype).float()
    b[N // 3] = b[N // 7]
    eps = 1e-6
    am = {}
    logits = ops.gemm(x, w, bias=b, rms_eps=eps, argmax=am)
    ref_logits = ops.gemm(x, w, bias=b, rms_eps=eps)
    assert torch.equal(logits, ref_logits)
    val, idx, ssum = am["val"], am["idx"].long(), am["sum"]
    m = val.max(-1).values
    cand = torch.where(val == m[:, None], idx, torch.full_like(idx, 1 << 40))
    tok = cand.min(-1).values
    lf = ref_logits.float()
    assert torch.equal(tok, lf.argmax(-1)), "argmax of the partials differs from torch.argmax of the logits"
    denom = (ssum * torch.exp(val - m[:, None])).sum(-1)
    score = 1.0 / denom
    ref_score = torch.softmax(lf, -1).max(-1).values
    assert ((score - ref_score).abs() <= 2e-5 + 1e-4 * ref_score).all()
    canary = torch.full((M, N), 7.0, device="cuda", dtype=dtype)
    am2 = {}
    ops.gemm(x, w, bias=b, rms_eps=eps, argmax=am2, argmax_only=True, out=canary)
    assert (canary == 7.0).all() and torch.equal(am2["idx"], am["idx"]) and torch.equal(am2["val"], am["val"])


@pytest.mark.parametrize("dtype", DT)
def test_gather_pad(built_lib, dtype):
    from surya_b200 import ops

    src = torch.randn(64, 588, device="cuda")
    perm = torch.randperm(64, device="cuda").to(torch.int32)
    out = ops.gather_pad_rows(src, perm, 592, dtype)
    ref = torch.zeros(64, 592, device="cuda", dtype=dtype)
    ref[:, :588] = src[perm.long()].to(dtype)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("dtype", DT)
def test_rope_vision(built_lib, dtype):
    from surya_b200 import ops

    nh, d, n = 4, 80, 50
    g = torch.Generator(device="cuda").manual_seed(2)
    qkv = torch.randn(n, 3 * nh * d, device="cuda", generator=g).to(dtype)
    pos = torch.stack([torch.arange(n, device="cuda") % 7, torch.arange(n, device="cuda") % 13], 1).to(torch.int32).contiguous()
    inv_freq = 1.0 / (10000.0 ** (torch.arange(0, d // 2, 2, dtype=torch.float) / (d // 2)))
    inv_freq = inv_freq.cuda()
    ref_in = qkv.clone()
    ops.rope_vision_(qkv, pos, inv_freq, nh, d)
    freqs = torch.cat([pos[:, 0:1].float() * inv_freq[None], pos[:, 1:2].float() * inv_freq[None]], -1)  # [n, d/2]
    emb = torch.cat([freqs, freqs], -1)
    cos, sin = emb.cos()[:, None, :], emb.sin()[:, None, :]

    def rot(x):
        x1, x2 = x[..., : d // 2], x[..., d // 2:]
        return torch.cat([-x2, x1], -1)

    qk = ref_in[:, : 2 * nh * d].reshape(n, 2 * nh, d).float()
    ref_qk = (qk * cos + rot(qk) * sin).to(dtype).reshape(n, -1)
    _close(qkv[:, : 2 * nh * d], ref_qk, dtype, ulps=1.01, what="rope_vision")
    assert torch.equal(qkv[:, 2 * nh * d:], ref_in[:, 2 * nh * d:])


def _attn_ref(q, k, v, lens, causal, scale, group):
    # q [T, nh, d], k/v [T, nkv, d] fp32; block-diagonal by lens
    outs = []
    s = 0
    for L in lens:
        qq, kk, vv = q[s:s + L], k[s:s + L], v[s:s + L]
        kk = kk.repeat_interleave(group, dim=1)
        vv = vv.repeat_interleave(group, dim=1)
        sc = torch.einsum("qhd,khd->hqk", qq, kk) * scale
        if causal:
            mask = torch.ones(L, L, device=q.device, dtype=torch.bool).tril()
            sc = sc.masked_fill(~mask, float("-inf"))
        p = sc.softmax(-1)
        outs.append(torch.einsum("hqk,khd->qhd", p, vv))
        s += L
    return torch.cat(outs, 0)


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("d,nh,nkv,causal,lens", [
    (80, 4, 4, False, [32, 32, 64, 17, 160, 1]),
    (80, 8, 2, True, [46, 46, 5, 130, 64]),
    (64, 4, 1, True, [100, 3]),
    (128, 2, 2, False, [70, 200]),
    (32, 4, 4, False, [64, 64, 9]),
])
def test_attn_varlen(built_lib, dtype, d, nh, nkv, causal, lens):
    from surya_b200 import ops

    T = sum(lens)
    g = torch.Generator(device="cuda").manual_seed(d + nh)
    width = (nh + 2 * nkv) * d
    qkv = torch.randn(T, width, device="cuda", generator=g).to(dtype)
    q, k, v = qkv[:, : nh * d], qkv[:, nh * d: (nh + nkv) * d], qkv[:, (nh + nkv) * d:]
    starts = torch.tensor([sum(lens[:i]) for i in range(len(lens))], device="cuda", dtype=torch.int32)
    lens_t = torch.tensor(lens, device="cuda", dtype=torch.int32)
    scale = d ** -0.5
    out = ops.attn_varlen(q, k, v, starts, lens_t, max(lens), nh, nkv, d, causal, scale)
    torch.cuda.synchronize()
    ref = _attn_ref(q.float().reshape(T, nh, d), k.float().reshape(T, nkv, d), v.float().reshape(T, nkv, d), lens,
                    causal, scale, nh // nkv).reshape(T, nh * d)
    err = (out.float() - ref).abs().max().item()
    assert err < (0.03 if dtype == torch.bfloat16 else 0.005), f"attn_varlen max err {err}"


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("d,nh,nkv", [(80, 16, 4), (64, 8, 8), (128, 8, 1)])
def test_decode_attn_and_rope_append(built_lib, dtype, d, nh, nkv):
    from surya_b200 import ops

    B, slots, s_max = 5, 8, 256
    g = torch.Generator(device="cuda").manual_seed(d)
    kc = torch.zeros(slots, nkv, s_max, d, device="cuda", dtype=dtype)
    vc = torch.zeros_like(kc)
    inv_freq = (1.0 / (10000.0 ** (torch.arange(0, d, 2, dtype=torch.float) / d))).cuda()
    width = (nh + 2 * nkv) * d
    # prefill: sequences with different lengths in slots 1..B via rope_kv_append
    lens = [46, 7, 100, 1, 63]
    slot_ids = [1, 3, 0, 7, 5]
    tok_pos = torch.tensor([p for L in lens for p in range(L)], device="cuda", dtype=torch.int32)
    tok_slot = torch.tensor([s for L, s in zip(lens, slot_ids) for _ in range(L)], device="cuda", dtype=torch.int32)
    Tn = sum(lens)
    qkv = torch.randn(Tn, width, device="cuda", generator=g).to(dtype)
    raw = qkv.clone()
    ops.rope_kv_append_(qkv, tok_pos, tok_slot, inv_freq, kc, vc, nh, nkv, d)

    def rope_T(x, pos):  # x [n, heads, d] in dtype; 3-rounding reference
        freqs = pos[:, None].float() * inv_freq[None]
        emb = torch.cat([freqs, freqs], -1)
        cos, sin = emb.cos().to(dtype)[:, None, :], emb.sin().to(dtype)[:, None, :]
        x1, x2 = x[..., : d // 2], x[..., d // 2:]
        rot = torch.cat([-x2, x1], -1)
        return (x * cos) + (rot * sin)

    qk_ref = rope_T(raw[:, : (nh + nkv) * d].reshape(Tn, nh + nkv, d), tok_pos)
    _close(qkv[:, : (nh + nkv) * d], qk_ref.reshape(Tn, -1), dtype, ulps=1.01, what="rope_kv_append q,k")
    # cache contents
    off = 0
    for L, s in zip(lens, slot_ids):
        kref = qk_ref[off:off + L, nh:, :].permute(1, 0, 2)
        vref = raw[off:off + L, (nh + nkv) * d:].reshape(L, nkv, d).permute(1, 0, 2)
        _close(kc[s, :, :L], kref, dtype, ulps=1.01, what="kcache")
        assert torch.equal(vc[s, :, :L], vref)
        off += L
    # decode step
    slot = torch.tensor(slot_ids, device="cuda", dtype=torch.int32)
    pos = torch.tensor(lens, device="cuda", dtype=torch.int32)
    qkv1 = torch.randn(B, width, device="cuda", generator=g).to(dtype)
    out = ops.decode_attn(qkv1, kc, vc, slot, pos, inv_freq, nh, nkv, d, d ** -0.5)
    torch.cuda.synchronize()
    qk1 = rope_T(qkv1[:, : (nh + nkv) * d].reshape(B, nh + nkv, d), pos)
    group = nh // nkv
    for b in range(B):
        L, s = lens[b], slot_ids[b]
        _close(kc[s, :, L], qk1[b, nh:], dtype, ulps=1.01, what="decode k append")
        assert torch.equal(vc[s, :, L], qkv1[b, (nh + nkv) * d:].reshape(nkv, d))
        K = kc[s, :, : L + 1].float().repeat_interleave(group, 0)  # [nh, L+1, d]
        V = vc[s, :, : L + 1].float().repeat_interleave(group, 0)
        q = qk1[b, :nh].float()  # [nh, d]
        sc = torch.einsum("hd,hkd->hk", q, K) * d ** -0.5
        ref = torch.einsum("hk,hkd->hd", sc.softmax(-1), V).reshape(-1)
        err = (out[b].float() - ref).abs().max().item()
        assert err < (0.03 if dtype == torch.bfloat16 else 0.005), f"decode_attn row {b} err {err}"


@pytest.mark.parametrize("dtype", DT)
def test_embed_splice_and_heads(built_lib, dtype):
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(1)
    V, H = 1000, 256
    embed = torch.randn(V, H, device="cuda", generator=g).to(dtype)
    feat = torch.randn(20, H, device="cuda", generator=g).to(dtype)
    he = torch.randn(64, H, device="cuda", generator=g).to(dtype)
    we = torch.randn(64, H, device="cuda", generator=g).to(dtype)
    ids = torch.tensor([3, 3, 3, 10, 999, 3], device="cuda", dtype=torch.int64)
    fr = torch.tensor([4, 0, 19, -1, -1, 7], device="cuda", dtype=torch.int32)
    hi = torch.tensor([0, 63, 5, 0, 0, 9], device="cuda", dtype=torch.int32)
    wi = torch.tensor([1, 2, 3, 0, 0, 63], device="cuda", dtype=torch.int32)
    out = ops.embed_splice(ids, fr, hi, wi, embed, feat, he, we)
    ref = embed[ids].clone()
    for t in [0, 1, 2, 5]:
        ref[t] = feat[fr[t]] + (he[hi[t]] + we[wi[t]])
    assert torch.equal(out, ref)
    assert torch.equal(ops.embed_rows(ids, embed), embed[ids])

    logits = (torch.randn(9, 65792, device="cuda", generator=g) * 2).to(dtype)
    logits[2, 1] = 50.0   # eos
    logits[4, 100] = logits[4, 200] = 40.0  # tie -> first index
    tok, score, done, nxt = ops.argmax_score(logits, eos=1, pad=2)
    lf = logits.float()
    assert torch.equal(tok, lf.argmax(-1))
    ref_score = lf.softmax(-1).max(-1).values
    ref_done = (tok == 1) | (tok == 2)
    assert torch.equal(done.bool(), ref_done)
    assert torch.allclose(score, ref_score.masked_fill(ref_done, 0), rtol=1e-4, atol=1e-6)
    assert torch.equal(nxt, torch.where(ref_done, torch.full_like(tok, 2), tok))
    assert tok[4].item() == 100

    x = torch.randn(9, H, device="cuda", generator=g).to(dtype)
    w = (torch.randn(6, H, device="cuda", generator=g) * 0.1).to(dtype)
    b = torch.randn(6, device="cuda", generator=g).to(dtype)
    sig, box = ops.small_head(x, w, b, sigmoid=True, box_scale=1025.0)
    lin = (x.float() @ w.float().t() + b.float()).to(dtype)
    ref_sig = torch.sigmoid(lin.float()).to(dtype).float()
    assert (sig - ref_sig).abs().max().item() <= 2 * _ulp(dtype)
    assert (box - (sig * 1025.0).to(torch.int64)).abs().max().item() == 0


# ------------------------------------------------------------------------------------------------ split-K cluster GEMM
@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize(
    "M,N,K,pk,bn,epi",
    [
        (256, 1280, 1280, 7, 128, "res"), (256, 1920, 1280, 4, 128, "bias"), (200, 1280, 3424, 7, 128, "res"),
        (256, 1280, 1280, 2, 64, "none"), (256, 1280, 1280, 3, 64, "bias_res_gelu"), (16, 1024, 1024, 8, 128, "none"),
        (130, 1000, 640, 5, 128, "bias"), (256, 512, 1280, 8, 64, "swiglu"), (96, 4096, 1024, 2, 128, "geglu"),
        (256, 1280, 1280, 0, 0, "res"), (256, 1920, 1280, 0, 0, "bias"), (16, 512, 1024, 0, 0, "none"),
    ],
)
def test_gemm_splitk_cluster(built_lib, dtype, M, N, K, pk, bn, epi):
    """Split-K over a thread-block cluster with the DSMEM reduce-scatter (gemm_splitk.cu); pk = 0 rows exercise the automatic
    plan that decode-sized GEMMs take.  Same contract and tolerance as the plain kernel; deterministic across runs."""
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M + N + K + pk)
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(dtype)
    bias = torch.randn(N, device="cuda", generator=g).to(dtype).float() if "bias" in epi else None
    swi = epi in ("swiglu", "geglu")
    res = torch.randn(M, N, device="cuda", generator=g).to(dtype) if "res" in epi else None
    act = "silu" if epi == "swiglu" else "gelu_tanh" if epi == "geglu" else "gelu" if "gelu" in epi else "none"
    force = 1000 * pk + bn if pk else -1     # -1: the automatic plan decode steps opt into
    out = ops.gemm(a, w, bias=bias, residual=res, act=act, swiglu=swi, force_bn=force)
    out2 = ops.gemm(a, w, bias=bias, residual=res, act=act, swiglu=swi, force_bn=force)
    torch.cuda.synchronize()
    assert torch.equal(out, out2), "split-K reduction must be deterministic"
    lin = a.float() @ w.float().t()
    if bias is not None:
        lin = lin + bias
    lin = lin.to(dtype)
    if swi:
        gate, up = lin[:, 0::2], lin[:, 1::2]
        ref = (_act_ref(gate.float(), act).to(dtype).float() * up.float()).to(dtype)
        _close(out, ref, dtype, ulps=3.0, what=f"splitk {epi}")
        return
    y = _act_ref(lin.float(), act).to(dtype) if act != "none" else lin
    ref = (y.float() + res.float()).to(dtype) if res is not None else y
    scale = torch.maximum(lin.float().abs(), res.float().abs()) if res is not None else None
    _close(out, ref, dtype, ulps=3.0, what=f"splitk {M}x{N}x{K} pk={pk} bn={bn} {epi}", scale=scale)


# ------------------------------------------------------------------------------------------------ error behaviour
def test_errors_are_loud(built_lib):
    """Bad arguments come back as a negative code + message through the C ABI (raised as SuryaB200Error), never as a silent
    fallback: misaligned TMA pitch, odd SwiGLU width, unsupported head_dim / GQA group, unsupported depthwise kernel size."""
    from surya_b200 import _lib, ops

    dt = torch.bfloat16
    a = torch.randn(64, 100, device="cuda").to(dt)          # row pitch 200 B: not a multiple of 16
    w = torch.randn(32, 100, device="cuda").to(dt)
    with pytest.raises(_lib.SuryaB200Error, match="16B"):
        ops.gemm(a, w)
    a = torch.randn(64, 128, device="cuda").to(dt)
    w = torch.randn(33, 128, device="cuda").to(dt)
    with pytest.raises(_lib.SuryaB200Error, match="even N"):
        ops.gemm(a, w, act="silu", swiglu=True)
    B, nh, nkv, hd = 2, 6, 2, 72
    qkv = torch.randn(B, (nh + 2 * nkv) * hd, device="cuda").to(dt)
    kc = torch.zeros(B, nkv, 16, hd, device="cuda", dtype=dt)
    slot = torch.arange(B, dtype=torch.int32, device="cuda")
    pos = torch.zeros(B, dtype=torch.int32, device="cuda")
    inv = torch.ones(hd // 2, device="cuda")
    with pytest.raises(_lib.SuryaB200Error, match="head_dim"):
        ops.decode_attn(qkv, kc, kc.clone(), slot, pos, inv, nh, nkv, hd, 1.0)
    x = torch.randn(1, 8, 8, 16, device="cuda").half()
    with pytest.raises(_lib.SuryaB200Error, match="kernel size"):
        ops.dwconv_nhwc(x, torch.randn(49, 16, device="cuda").half(), None, 7, 1, 3, "none")
    # and the library keeps working after an error
    a = torch.randn(64, 128, device="cuda").to(dt)
    w = torch.randn(32, 128, device="cuda").to(dt)
    out = ops.gemm(a, w)
    torch.cuda.synchronize()
    _close(out, (a.float() @ w.float().t()).to(dt), dt, what="gemm after errors")


@pytest.mark.parametrize("dtype", DT)
@pytest.mark.parametrize("M,N,K,epi", [(16, 1024, 1024, "bias"), (16, 8192, 1024, "geglu"), (16, 1024, 4096, "res"), (3, 520, 320, "gelu"),
                                       (16, 1536, 1024, "none"), (1, 20, 1024, "none")])
def test_gemm_skinny_path(built_lib, dtype, M, N, K, epi):
    """M <= 16 routes to the mma.sync kernel (gemm_skinny.cu): against the fp32 restatement with the output roundings, and
    against the tcgen05 kernel (forced tile width) to a few ulp — the two paths sum in different orders."""
    from surya_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).to(dtype)
    w = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(dtype)
    bias = (torch.randn(N, device="cuda", generator=g) * 0.1).to(dtype).float() if epi in ("bias", "gelu") else None
    res = (torch.randn(M, N, device="cuda", generator=g)).to(dtype) if epi == "res" else None
    act = {"gelu": "gelu", "geglu": "gelu_tanh"}.get(epi, "none")
    got = ops.gemm(a, w, bias=bias, residual=res, act=act, swiglu=(epi == "geglu"))
    lin = a.float() @ w.float().t()
    if bias is not None:
        lin = lin + bias
    lin = lin.to(dtype).float()
    if epi == "geglu":
        gt, up = lin[:, 0::2], lin[:, 1::2]
        ref = (_act_ref(gt, "gelu_tanh").to(dtype).float() * up).to(dtype)
    else:
        y = _act_ref(lin, act).to(dtype).float() if act != "none" else lin
        ref = (y + res.float()).to(dtype) if res is not None else y.to(dtype)
    _close(got, ref, dtype, ulps=4.0 if epi == "geglu" else 2.0, what="skinny gemm", scale=lin if res is not None else None)
    if N % 8 == 0 and epi != "geglu":
        tc = ops.gemm(a, w, bias=bias, residual=res, act=act, force_bn=32)
        _close(got, tc, dtype, ulps=2.0, what="skinny vs tcgen05", scale=lin if res is not None else None)
