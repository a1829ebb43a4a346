"""The windowed-attention encoder under the bf16 precision switch (ops.set_precision("bf16"), inference):

  * mts_band_attn_fwd_bf16 against a float64 dense masked softmax over the same bf16 q/k/v;
  * the two epilogue forms of the bf16 product (bf16 output; GELU + packed operand) against mts_gemm_bf16p, bit for bit;
  * Transformer_segmenter end to end against the oracle (oracle/ref_torch.WindowedSegmenter) with the same weights;
  * bf16 embeddings in, and the switch's hygiene (the fp32 path and training are untouched).

Every test prints what it measured next to the bound it asserts.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import multimodaltopicsegmentation_b200 as m

    m.ops.device_ok()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _call(name, *args):
    from multimodaltopicsegmentation_b200 import ops

    return ops._call(name, *args)


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    from multimodaltopicsegmentation_b200 import ops

    return ops._stream()


# ------------------------------------------------------------------------------------------------------------------
# 1. attention kernel
# ------------------------------------------------------------------------------------------------------------------
def _band_ref64(q, k, v, lens, w):
    """float64 dense reference: q, k, v [B, S, h, hd] -> o [B, S, h, hd] (zeros for padded queries), lse [B, h, S] (0 there)."""
    B, S, h, hd = q.shape
    q, k, v = (t.double().permute(0, 2, 1, 3) for t in (q, k, v))
    s = (q / np.sqrt(hd)) @ k.transpose(-1, -2)
    idx = torch.arange(S, device=q.device)
    band = (idx[:, None] - idx[None, :]).abs() <= w
    o = torch.zeros_like(q)
    lse = torch.zeros(B, h, S, dtype=torch.float64, device=q.device)
    for b in range(B):
        n = int(lens[b])
        allowed = band[:n, :n]
        sb = s[b, :, :n, :n].masked_fill(~allowed, float("-inf"))
        o[b, :, :n] = torch.softmax(sb, dim=-1) @ v[b, :, :n]
        lse[b, :, :n] = torch.logsumexp(sb, dim=-1)
    return o.permute(0, 2, 1, 3), lse


def _attn_bf16(qkv, lens_t, offs, rows, B, S, h, hd, w, dev):
    d = h * hd
    out = torch.empty((rows, d), device=dev, dtype=torch.float32)
    out_lo = torch.empty((rows, d), device=dev, dtype=torch.float32)
    lse = torch.zeros((B, h, S), device=dev, dtype=torch.float32)
    _call("mts_band_attn_fwd_bf16", _ptr(qkv), 3 * d, rows, _ptr(lens_t), _ptr(offs), B, S, h, hd, w, _ptr(out), _ptr(out_lo), d,
          _ptr(lse), _stream())
    torch.cuda.synchronize()
    return out, out_lo, lse


@pytest.mark.parametrize("hd", [16, 32, 64, 112, 128])
@pytest.mark.parametrize("w", [0, 8, 48, 360])
def test_band_attention_bf16_vs_float64(dev, hd, w):
    from multimodaltopicsegmentation_b200 import ops

    torch.manual_seed(hd * 1000 + w)
    B, S, h = 4, 960, 2
    d = h * hd
    lens = [S, 1, 517, 130]
    lens_t = torch.tensor(lens, dtype=torch.int32, device=dev)
    # q scaled up so that the softmax is peaked as well as flat across the cases
    q = (2.0 * torch.randn(B, S, h, hd, device=dev)).to(torch.bfloat16)
    k = torch.randn(B, S, h, hd, device=dev).to(torch.bfloat16)
    v = torch.randn(B, S, h, hd, device=dev).to(torch.bfloat16)
    o_ref, lse_ref = _band_ref64(q, k, v, lens, w)
    vmax = float(v.float().abs().max())
    padded = torch.cat([t.reshape(B * S, d) for t in (q, k, v)], dim=1).contiguous()
    offs = torch.tensor(np.concatenate([[0], np.cumsum(lens)[:-1]]), dtype=torch.int32, device=dev)
    ragged = torch.cat([padded[b * S: b * S + n] for b, n in enumerate(lens)]).contiguous()
    for layout in ("padded", "ragged"):
        if layout == "padded":
            out, out_lo, lse = _attn_bf16(padded, lens_t, None, B * S, B, S, h, hd, w, dev)
            o = out.view(B, S, h, hd)
            # padded queries: exact zeros
            for b, n in enumerate(lens):
                assert torch.count_nonzero(out.view(B, S, d)[b, n:]) == 0
        else:
            out, out_lo, lse = _attn_bf16(ragged, lens_t, offs, sum(lens), B, S, h, hd, w, dev)
            o = torch.zeros(B, S, d, device=dev)
            for b, n in enumerate(lens):
                o[b, :n] = out[int(offs[b]): int(offs[b]) + n]
            o = o.view(B, S, h, hd)
        err = float((o.double() - o_ref).abs().max())
        lse_err = max(float((lse[b, :, :n].double() - lse_ref[b, :, :n]).abs().max()) for b, n in enumerate(lens))
        # the packed output is the side-0 operand of out: [bf16(x) | bf16(x - trunc_tf32(x))] per 16 columns
        lo_ref = ops.split_tf32(out)[1]
        assert torch.equal(out_lo.view(torch.int32), lo_ref.view(torch.int32))
        print(f"  hd {hd} w {w} {layout}: max|o - o_ref| {err:.3e} (max|v| {vmax:.2f}, bound {1e-2 * vmax:.3e}); "
              f"max|lse - lse_ref| {lse_err:.3e}")
        assert err <= 1e-2 * vmax
        assert lse_err <= 1e-2


def test_band_attention_bf16_ignores_padding_and_out_of_band_keys(dev):
    """Padded rows' q/k/v, and keys outside every query's band, never reach the output: bit-identical results."""
    torch.manual_seed(5)
    B, S, h, hd, w = 3, 700, 2, 64, 48
    d = h * hd
    lens = [700, 300, 129]
    lens_t = torch.tensor(lens, dtype=torch.int32, device=dev)
    qkv = torch.randn(B * S, 3 * d, device=dev).to(torch.bfloat16)
    out0, lo0, lse0 = _attn_bf16(qkv, lens_t, None, B * S, B, S, h, hd, w, dev)
    alt = qkv.clone().view(B, S, 3 * d)
    for b, n in enumerate(lens):
        alt[b, n:] = 1e3 * torch.randn_like(alt[b, n:].float()).to(torch.bfloat16)
    # episode 0: keys from 128 + w + 1 on lie outside the band of every query of the first query block
    alt[0, 128 + w + 1:, d:] = -7.0
    out1, lo1, lse1 = _attn_bf16(alt.view(B * S, 3 * d), lens_t, None, B * S, B, S, h, hd, w, dev)
    o0, o1 = out0.view(B, S, d), out1.view(B, S, d)
    assert torch.equal(o0[0, :128], o1[0, :128])
    assert torch.equal(o0[1:], o1[1:])
    assert torch.equal(lse0[1:], lse1[1:]) and torch.equal(lse0[0, :, :128], lse1[0, :, :128])


def test_band_attention_bf16_rejects_unsupported_head_dims(dev):
    from multimodaltopicsegmentation_b200 import _lib

    qkv = torch.zeros((8, 3 * 48), device=dev, dtype=torch.bfloat16)
    out = torch.empty((8, 48), device=dev)
    lens = torch.tensor([8], dtype=torch.int32, device=dev)
    with pytest.raises(_lib.MtsError, match="head dim"):
        _call("mts_band_attn_fwd_bf16", _ptr(qkv), 144, 8, _ptr(lens), 0, 1, 8, 1, 48, 2, _ptr(out), 0, 0, 0, _stream())


# ------------------------------------------------------------------------------------------------------------------
# 2. GEMM epilogue forms of the bf16 product
# ------------------------------------------------------------------------------------------------------------------
def _packed(x):
    from multimodaltopicsegmentation_b200 import ops

    return ops.split_tf32(x.contiguous(), side=ops.A_SIDE)[1]


@pytest.mark.parametrize("M,N,K", [(1000, 3 * 896, 896), (300, 96, 32), (777, 192, 256)])
def test_gemm_bf16p_out16_is_rounded_fp32_output(dev, M, N, K):
    torch.manual_seed(M + N)
    a_lo = _packed(torch.randn(M, K, device=dev))
    w_lo = _packed(0.05 * torch.randn(N, K, device=dev))
    bias = torch.randn(N, device=dev)
    c32 = torch.empty((M, N), device=dev)
    c16 = torch.empty((M, N), device=dev, dtype=torch.bfloat16)
    _call("mts_gemm_bf16p", _ptr(a_lo), _ptr(w_lo), _ptr(bias), _ptr(c32), M, N, K, N, 1, 0, _stream())
    _call("mts_gemm_bf16p_out16", _ptr(a_lo), _ptr(w_lo), _ptr(bias), _ptr(c16), M, N, K, N, _stream())
    torch.cuda.synchronize()
    ref = c32.to(torch.bfloat16)   # round to nearest even
    print(f"  out16 {M}x{N}x{K}: elements differing from bf16(fp32 output): {int((c16 != ref).sum())}")
    assert torch.equal(c16.view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize("M,N,K", [(1000, 256, 896), (300, 128, 256), (513, 3584, 896)])
def test_gemm_bf16p_gelu_pair_matches_epilogue_2_and_split(dev, M, N, K):
    torch.manual_seed(M + N + 1)
    a_lo = _packed(torch.randn(M, K, device=dev))
    w_lo = _packed(0.05 * torch.randn(N, K, device=dev))
    bias = torch.randn(N, device=dev)
    c_ref = torch.empty((M, N), device=dev)
    c = torch.empty((M, N), device=dev)
    c_lo = torch.empty((M, N), device=dev)
    _call("mts_gemm_bf16p", _ptr(a_lo), _ptr(w_lo), _ptr(bias), _ptr(c_ref), M, N, K, N, 2, 0, _stream())
    _call("mts_gemm_bf16p_gelu_pair", _ptr(a_lo), _ptr(w_lo), _ptr(bias), _ptr(c), _ptr(c_lo), M, N, K, _stream())
    torch.cuda.synchronize()
    assert torch.equal(c.view(torch.int32), c_ref.view(torch.int32))
    assert torch.equal(c_lo.view(torch.int32), _packed(c).view(torch.int32))


# ------------------------------------------------------------------------------------------------------------------
# 3. - 5. the encoder
# ------------------------------------------------------------------------------------------------------------------
def _pair(d, F, nl, nh, w, seed):
    from multimodaltopicsegmentation_b200.transformer import Transformer_segmenter
    from oracle import ref_torch as rt

    torch.manual_seed(seed)
    ref = rt.WindowedSegmenter(2, d, F, num_layers=nl, nheads=nh, loss_fn="BinaryCrossEntropy", window_size=w).eval()
    with torch.no_grad():
        ref.classification.weight.mul_(4.0)
    ours = Transformer_segmenter(2, d, F, num_layers=nl, nheads=nh, loss_fn="BinaryCrossEntropy", window_size=w)
    missing, unexpected = ours.load_state_dict(ref.state_dict(), strict=False)
    assert not missing, missing
    ref.th = ours.th = 0.5
    return ref, ours


@pytest.mark.parametrize("d,F,nl,nh,w,B,S", [(896, 256, 6, 8, 16, 16, 960), (256, 512, 2, 8, 16, 8, 480)])
def test_transformer_bf16_vs_oracle(dev, d, F, nl, nh, w, B, S):
    """configs[2]-like shape (d 896, hd 112) and a d 256 one (hd 32): logits within 2e-2 of the logit scale, at most 0.5 % of the
    boundary decisions differing from the oracle (the bf16 path's contract)."""
    from multimodaltopicsegmentation_b200 import ops

    ref, ours = _pair(d, F, nl, nh, w, seed=d)
    ours = ours.to(dev).eval()
    g = torch.Generator().manual_seed(S)
    x = torch.randn(B, S, d, generator=g)
    lengths = torch.randint(100, S + 1, (B,), generator=g)
    lengths[0] = S
    with torch.no_grad():
        s_ref, tags_ref = ref(x, lengths)
    s32, tags32 = ours(x.to(dev), lengths)
    ops.set_precision("bf16")
    try:
        s16, tags16 = ours(x.to(dev), lengths)
    finally:
        ops.set_precision("f32")
    s16, s32 = s16.cpu().double(), s32.cpu().double()
    scale = float(s_ref.abs().max())
    worst = max(float((s16[b, :n] - s_ref[b, :n].double()).abs().max()) for b, n in enumerate(lengths.tolist()))
    worst32 = max(float((s32[b, :n] - s_ref[b, :n].double()).abs().max()) for b, n in enumerate(lengths.tolist()))
    n_dec = int(lengths.sum())
    flips = sum(int(a != r) for ta, tr in zip(tags16, tags_ref) for a, r in zip(ta, tr))
    flips32 = sum(int(a != r) for ta, tr in zip(tags32, tags_ref) for a, r in zip(ta, tr))
    print(f"  d {d} hd {d // nh}: bf16 worst |logit error| {worst:.3e} = {worst / scale:.2e} of scale {scale:.3f} "
          f"(fp32 path {worst32:.3e}); decisions differing from the oracle: {flips} of {n_dec} (fp32 path: {flips32})")
    assert worst <= 2e-2 * scale
    assert flips <= max(2, n_dec // 200)


@pytest.mark.parametrize("layout", ["ragged", "padded"])
def test_transformer_bf16_embeddings_in(dev, layout, monkeypatch):
    """bf16 embeddings give exactly what fp32 embeddings holding the same rounded values give."""
    from multimodaltopicsegmentation_b200 import ops, transformer

    monkeypatch.setattr(transformer, "LAYOUT", layout)
    _, ours = _pair(256, 256, 2, 4, 8, seed=3)
    ours = ours.to(dev).eval()
    g = torch.Generator().manual_seed(4)
    B, S = 5, 300
    xb = torch.randn(B, S, 256, generator=g).to(torch.bfloat16).to(dev)
    lengths = torch.tensor([300, 1, 77, 250, 128])
    ops.set_precision("bf16")
    try:
        s_in, t_in = ours(xb, lengths)
        s_rounded, t_rounded = ours(xb.float(), lengths)
    finally:
        ops.set_precision("f32")
    assert torch.equal(s_in, s_rounded) and t_in == t_rounded


def test_transformer_bf16_switch_hygiene(dev):
    """The fp32 path is bit-identical before and after a bf16 interlude; under the switch loss() and its backward run the fp32
    path (exactly its results); bf16 embeddings without the switch are refused."""
    from multimodaltopicsegmentation_b200 import ops

    _, ours = _pair(256, 256, 2, 8, 8, seed=9)
    ours = ours.to(dev)
    g = torch.Generator().manual_seed(10)
    B, S = 4, 256
    x = torch.randn(B, S, 256, generator=g).to(dev)
    lengths = torch.tensor([256, 100, 31, 200])
    tags = (torch.rand(B, S, generator=g) < 0.2).float().to(dev)
    s_before, _ = ours(x, lengths)

    def loss_and_grads():
        ours.zero_grad(set_to_none=True)
        loss = ours.loss(x, lengths, tags)
        loss.backward()
        return loss.detach().clone(), [p.grad.detach().clone() if p.grad is not None else None for p in ours.parameters()]

    l32, g32 = loss_and_grads()
    l32b, g32b = loss_and_grads()
    ops.set_precision("bf16")
    try:
        s16, _ = ours(x, lengths)
        l16, g16 = loss_and_grads()
        with pytest.raises(NotImplementedError):
            ours.loss(x.to(torch.bfloat16), lengths, tags)
    finally:
        ops.set_precision("f32")
    s_after, _ = ours(x, lengths)
    assert torch.equal(s_before, s_after)
    assert not torch.equal(s16, s_before)   # the switch did take the bf16 path
    assert torch.equal(l16, l32)
    repeatable = all((a is None and b is None) or torch.equal(a, b) for a, b in zip(g32, g32b))
    for a, b in zip(g16, g32):
        assert (a is None) == (b is None)
        if a is not None:
            # weight gradients sum split-K partial products with atomics: exact when the fp32 path repeats itself exactly
            assert torch.equal(a, b) if repeatable else torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))
    with pytest.raises(TypeError):
        with torch.no_grad():
            ours(x.to(torch.bfloat16), lengths)
