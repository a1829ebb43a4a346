"""The windowed-attention kernels at head dims 129-256: the widths of early fusions with 8 heads (768-d text + 512-d x-vectors ->
d 1280, hd 160; + 768-d wav2vec -> 1536 / 192; + 1024-d openl3 -> 1792 / 224; two openl3 streams -> 2048 / 256).

  * the fp32 forward (CUDA-core kernel, two float4 head columns per thread) against the numpy oracle;
  * the fp32 backward, with and without dropout on the probabilities, against float64 autograd;
  * the bf16 tcgen05 forward at HD 144 .. 256 against a float64 dense softmax over the same bf16 q/k/v;
  * Transformer_segmenter at d 1280 / 2048 against the HF twin (inference, training), and under the bf16 switch;
  * the user entry (TextSegmenter) and a BiLSTMRestrictedMHA block with hd 160.

Every test prints what it measured next to the bound it asserts.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BF16_WIDE = list(range(144, 257, 16))


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


def close(a, b, rtol, atol, msg=""):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=msg)


def _to_ragged(t, lens, B, S):
    return torch.cat([t.view(B, S, -1)[b, :n] for b, n in enumerate(lens)], dim=0).contiguous()


def _to_padded(t, lens, B, S):
    out = torch.zeros(B, S, t.shape[1], dtype=t.dtype, device=t.device)
    o = 0
    for b, n in enumerate(lens):
        out[b, :n] = t[o:o + n]
        o += n
    return out.view(B * S, -1)


def check_operand_pair(hi, lo, x):
    """(hi, lo) of an A operand: hi = x; lo per 16-wide K block [bf16(x) | bf16(x - trunc_tf32(x))]."""
    rows, K = x.shape
    assert torch.equal(hi, x)
    rest = x - (x.view(torch.int32) & ~0x1FFF).view(torch.float32)
    blocks = lo.contiguous().view(torch.bfloat16).view(rows, K // 16, 2, 16)
    assert torch.equal(blocks[:, :, 0], x.to(torch.bfloat16).view(rows, K // 16, 16))
    assert torch.equal(blocks[:, :, 1], rest.to(torch.bfloat16).view(rows, K // 16, 16))


# ------------------------------------------------------------------------------------------------------------------
# 1. fp32 forward
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["padded", "ragged"])
@pytest.mark.parametrize("entry", ["mts_band_attn_fwd", "mts_band_attn_fwd_simt"])
@pytest.mark.parametrize("hd", [132, 160, 200, 256])
@pytest.mark.parametrize("w", [0, 8, 48, 360])
def test_band_attention_forward_wide(dev, hd, w, entry, layout):
    """Lengths 1 .. S with 32-query block edges on both sides, a guard row behind the output, the fused operand pair."""
    from multimodaltopicsegmentation_b200 import ops
    from oracle import ref_numpy as rn

    B, S, h = 6, 300, 2
    lens = [300, 1, 32, 33, 129, 64]
    g = torch.Generator().manual_seed(S + hd + w)
    d = h * hd
    qkv = torch.randn(B * S, 3 * d, generator=g)
    L = ops.Lengths(lens, dev, S)
    ragged = layout == "ragged"
    offs = L.offs.data_ptr() if ragged else 0
    qkv_d = (_to_ragged(qkv, lens, B, S) if ragged else qkv).to(dev)
    rows = qkv_d.shape[0]
    out = torch.full((rows + 1, d), 7.0, device=dev)
    lse = torch.empty(B, h, S, device=dev)
    _call(entry, qkv_d.data_ptr(), 3 * d, L.dev.data_ptr(), offs, B, S, h, hd, w, out.data_ptr(), 0, 0, 0, lse.data_ptr(), _stream())
    assert float((out[rows] - 7.0).abs().max()) == 0.0
    out = out[:rows]
    split = lambda t: t.view(B, S, h, hd).permute(0, 2, 1, 3).numpy()
    q = split(qkv[:, :d]) / np.float32(np.sqrt(hd))
    ref = rn.banded_attention(q.astype(np.float32), split(qkv[:, d:2 * d]), split(qkv[:, 2 * d:]), lens, w)
    full = _to_padded(out, lens, B, S) if ragged else out
    got = full.view(B, S, h, hd).permute(0, 2, 1, 3)
    err = float((got.cpu().double() - torch.from_numpy(np.asarray(ref, dtype=np.float64))).abs().max())
    print(f"  hd {hd} w {w} {entry} {layout}: max|o - ref| {err:.3e}")
    close(got, ref, rtol=1e-4, atol=1e-5)
    if not ragged:
        for b, n in enumerate(lens):
            assert float(out.view(B, S, d)[b, n:].abs().max() if n < S else 0.0) == 0.0
    if d % 32 == 0:
        hl = torch.full((2, rows + 1, d), 7.0, device=dev)
        _call(entry, qkv_d.data_ptr(), 3 * d, L.dev.data_ptr(), offs, B, S, h, hd, w, 0, hl[0].data_ptr(), hl[1].data_ptr(), d, 0,
              _stream())
        assert float((hl[:, rows] - 7.0).abs().max()) == 0.0
        check_operand_pair(hl[0, :rows], hl[1, :rows], out)


def test_band_attention_fwd_rejects_head_dims_past_256(dev):
    from multimodaltopicsegmentation_b200 import _lib

    qkv = torch.zeros((8, 3 * 260), device=dev)
    out = torch.empty((8, 260), device=dev)
    lens = torch.tensor([8], dtype=torch.int32, device=dev)
    for entry in ("mts_band_attn_fwd", "mts_band_attn_fwd_simt"):
        with pytest.raises(_lib.MtsError, match="head dim"):
            _call(entry, _ptr(qkv), 3 * 260, _ptr(lens), 0, 1, 8, 1, 260, 2, _ptr(out), 0, 0, 0, 0, _stream())


# ------------------------------------------------------------------------------------------------------------------
# 2. fp32 backward
# ------------------------------------------------------------------------------------------------------------------
def _dense_band_attention_torch(qkv, lens, B, S, h, hd, w, prob_scale=None):
    """float64 autograd reference: dense scores with the band / length mask, zero rows for padded queries."""
    d = h * hd
    q, k, v = [t.view(B, S, h, hd).permute(0, 2, 1, 3) for t in (qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:])]
    s = (q / np.sqrt(hd)) @ k.transpose(-1, -2)
    idx = torch.arange(S)
    band = (idx[:, None] - idx[None, :]).abs() <= w
    outs = []
    for b in range(B):
        n = lens[b]
        allowed = band & (idx[None, :] < n)
        sb = s[b].masked_fill(~allowed, float("-inf"))
        sb = torch.where(allowed.any(-1, keepdim=True), sb, torch.zeros_like(sb))
        p = torch.softmax(sb, dim=-1) * (idx < n)[None, :, None]
        if prob_scale is not None:
            p = p * prob_scale[b]
        outs.append(p @ v[b])
    return torch.stack(outs).permute(0, 2, 1, 3).reshape(B * S, d)


@pytest.mark.parametrize("B,S,h,hd,w,lens,p", [
    (2, 100, 2, 132, 8, [100, 37], 0.0),    # 33 float4 columns: one thread carries a second column
    (2, 150, 2, 160, 48, [150, 61], 0.0),
    (3, 130, 1, 256, 8, [130, 31, 1], 0.0),
    (2, 150, 2, 160, 48, [150, 61], 0.1),
    (3, 130, 1, 256, 8, [130, 31, 1], 0.25),
])
@pytest.mark.parametrize("layout", ["padded", "ragged"])
def test_band_attention_backward_wide(dev, B, S, h, hd, w, lens, p, layout):
    """dq / dk / dv of mts_band_attn_bwd(_dropout) against float64 autograd; with dropout the oracle regenerates the keep-mask
    from the seed (oracle/ref_numpy.py attn_dropout_keep)."""
    from multimodaltopicsegmentation_b200 import ops
    from oracle import ref_numpy as rn

    g = torch.Generator().manual_seed(S + hd + w + 7)
    seed = 0x1234_5678_9ABC_DEF0 ^ (S * 7919 + hd)
    d = h * hd
    scale_mask = None
    if p > 0:
        keep = rn.attn_dropout_keep(seed, B, h, S, p)
        scale_mask = torch.from_numpy(keep.astype(np.float64)) / (1.0 - float(np.float32(p)))
    qkv = torch.randn(B * S, 3 * d, generator=g, dtype=torch.float64).requires_grad_(True)
    do = torch.randn(B * S, d, generator=g, dtype=torch.float64)
    ragged = layout == "ragged"
    if ragged:
        for b, n in enumerate(lens):
            do.view(B, S, d)[b, n:] = 0
    ref = _dense_band_attention_torch(qkv, lens, B, S, h, hd, w, prob_scale=scale_mask)
    ref.backward(do)
    L = ops.Lengths(lens, dev, S)
    offs = L.offs.data_ptr() if ragged else 0
    pack = (lambda t: _to_ragged(t, lens, B, S)) if ragged else (lambda t: t)
    qkv_d = pack(qkv.detach().float()).to(dev)
    rows = qkv_d.shape[0]
    out = torch.empty(rows, d, device=dev)
    lse = torch.empty(B, h, S, device=dev)
    _call("mts_band_attn_fwd_dropout", qkv_d.data_ptr(), 3 * d, L.dev.data_ptr(), offs, B, S, h, hd, w, out.data_ptr(), 0, 0, 0,
          lse.data_ptr(), p, seed, _stream())
    o_err = float((out.cpu().double() - pack(ref.detach())).abs().max())
    close(out, pack(ref.detach().float()), rtol=1e-4, atol=2e-5)
    dqkv = torch.full((rows + 1, 3 * d), float("nan"), device=dev)
    delta = torch.empty(B, h, S, device=dev)
    do_d = pack(do.float()).to(dev)
    _call("mts_band_attn_bwd_dropout", qkv_d.data_ptr(), 3 * d, out.data_ptr(), do_d.data_ptr(), lse.data_ptr(), L.dev.data_ptr(), offs,
          B, S, h, hd, w, dqkv.data_ptr(), delta.data_ptr(), p, seed, _stream())
    assert bool(torch.isnan(dqkv[rows]).all())
    scale = float(qkv.grad.abs().max())
    err = float((dqkv[:rows].cpu().double() - pack(qkv.grad)).abs().max())
    print(f"  hd {hd} p {p} {layout}: max|o - ref| {o_err:.3e}; max|dqkv - ref| {err:.3e} = {err / scale:.2e} of scale {scale:.3f}")
    close(dqkv[:rows], pack(qkv.grad.float()), rtol=1e-4, atol=2e-5 * scale)


# ------------------------------------------------------------------------------------------------------------------
# 3. bf16 tcgen05 forward
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
        sb = s[b, :, :n, :n].masked_fill(~band[:n, :n], float("-inf"))
        o[b, :, :n] = torch.softmax(sb, dim=-1) @ v[b, :, :n]
        lse[b, :, :n] = torch.logsumexp(sb, dim=-1)
    return o.permute(0, 2, 1, 3), lse


def _attn_bf16(qkv, lens_t, offs, rows, B, S, h, hd, w, dev):
    d = h * hd
    out = torch.full((rows + 1, d), 7.0, device=dev, dtype=torch.float32)
    out_lo = torch.full((rows + 1, d), 7.0, device=dev, dtype=torch.float32)
    lse = torch.zeros((B, h, S), device=dev, dtype=torch.float32)
    _call("mts_band_attn_fwd_bf16", _ptr(qkv), 3 * d, rows, _ptr(lens_t), _ptr(offs), B, S, h, hd, w, _ptr(out), _ptr(out_lo), d,
          _ptr(lse), _stream())
    torch.cuda.synchronize()
    assert float((out[rows] - 7.0).abs().max()) == 0.0 and float((out_lo[rows] - 7.0).abs().max()) == 0.0
    return out[:rows], out_lo[:rows], lse


@pytest.mark.parametrize("hd", BF16_WIDE)
@pytest.mark.parametrize("w", [0, 8, 48, 360])
def test_band_attention_bf16_wide_vs_float64(dev, hd, w):
    from multimodaltopicsegmentation_b200 import ops

    torch.manual_seed(hd * 1000 + w)
    B, S, h = 4, 960, 2
    d = h * hd
    lens = [S, 1, 517, 130]
    lens_t = torch.tensor(lens, dtype=torch.int32, device=dev)
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
        lo_ref = ops.split_tf32(out)[1]
        assert torch.equal(out_lo.view(torch.int32), lo_ref.view(torch.int32))
        print(f"  hd {hd} w {w} {layout}: max|o - o_ref| {err:.3e} = {err / vmax:.2e} of max|v| {vmax:.2f}; "
              f"max|lse - lse_ref| {lse_err:.3e}")
        assert err <= 1e-2 * vmax
        assert lse_err <= 1e-2


def test_band_attention_bf16_supported_set(dev):
    from multimodaltopicsegmentation_b200 import _lib

    lib = _lib.load()
    got = [hd for hd in range(1, 513) if lib.mts_band_attn_bf16_supported(hd)]
    assert got == [16, 32, 64, 112, 128] + BF16_WIDE


@pytest.mark.parametrize("hd", [136, 272])
def test_band_attention_bf16_rejects_wide_head_dims_off_the_grid(dev, hd):
    from multimodaltopicsegmentation_b200 import _lib

    d = hd
    qkv = torch.zeros((8, 3 * d), device=dev, dtype=torch.bfloat16)
    out = torch.empty((8, d), device=dev)
    lens = torch.tensor([8], dtype=torch.int32, device=dev)
    with pytest.raises(_lib.MtsError, match="head dim"):
        _call("mts_band_attn_fwd_bf16", _ptr(qkv), 3 * d, 8, _ptr(lens), 0, 1, 8, 1, hd, 2, _ptr(out), 0, 0, 0, _stream())


# ------------------------------------------------------------------------------------------------------------------
# 4. the segmenter at early-fusion widths
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(params=["ragged", "padded"])
def xf_layout(request, monkeypatch):
    from multimodaltopicsegmentation_b200 import transformer

    monkeypatch.setattr(transformer, "LAYOUT", request.param)
    return request.param


def _pair(d, F, nl, nh, w, seed, loss_fn="BinaryCrossEntropy", train=False, head_scale=1.0):
    from multimodaltopicsegmentation_b200.transformer import Transformer_segmenter
    from oracle import ref_torch as rt

    torch.manual_seed(seed)
    ref = rt.WindowedSegmenter(2, d, F, num_layers=nl, nheads=nh, loss_fn=loss_fn, window_size=w)
    ref = ref.train() if train else ref.eval()
    with torch.no_grad():
        ref.classification.weight.mul_(head_scale)
    ours = Transformer_segmenter(2, d, F, num_layers=nl, nheads=nh, loss_fn=loss_fn, window_size=w)
    missing, _ = ours.load_state_dict(ref.state_dict(), strict=False)
    assert not missing, missing
    ref.th = ours.th = 0.5
    return ref, ours


@pytest.mark.parametrize("d", [1280, 2048])
def test_transformer_wide_vs_hf_twin(dev, xf_layout, d):
    torch.manual_seed(11)
    g = torch.Generator().manual_seed(12)
    B, S, F, nl, nh, w = 3, 96, 48, 3, 8, 8
    ref, ours = _pair(d, F, nl, nh, w, seed=d)
    ours = ours.to(dev).eval()
    x = torch.randn(B, S, d, generator=g)
    lengths = torch.tensor([96, 40, 7])
    y = (torch.rand(B, S, generator=g) < 0.2).float()
    with torch.no_grad():
        s_ref, t_ref = ref(x, lengths)
        l_ref = ref.loss(x, lengths, y)
        s, t = ours(x.to(dev), lengths)
        l = ours.loss(x.to(dev), lengths, y.to(dev))
    err = max(float((s[b, :n].cpu() - s_ref[b, :n]).abs().max()) for b, n in enumerate(lengths.tolist()))
    print(f"  d {d} hd {d // nh} {xf_layout}: max|scores - HF| {err:.3e}")
    for b, n in enumerate(lengths.tolist()):
        close(s[b, :n], s_ref[b, :n], rtol=1e-4, atol=2e-5)
    assert t == t_ref
    close(l, l_ref, rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("d", [1280, 2048])
def test_transformer_wide_training_vs_hf_twin(dev, xf_layout, d):
    torch.manual_seed(21)
    g = torch.Generator().manual_seed(22)
    B, S, F, nl, nh, w = 3, 96, 48, 2, 8, 8
    ref, ours = _pair(d, F, nl, nh, w, seed=d + 1, loss_fn="FocalLoss", train=True)
    ours = ours.to(dev).train()
    x = torch.randn(B, S, d, generator=g)
    lengths = torch.tensor([96, 40, 7])
    y = (torch.rand(B, S, generator=g) < 0.2).float()
    l_ref = ref.loss(x, lengths, y)
    l_ref.backward()
    l = ours.loss(x.to(dev), lengths, y.to(dev))
    l.backward()
    close(l, l_ref, rtol=1e-4, atol=2e-5)
    ref_named = dict(ref.named_parameters())
    checked, worst = 0, 0.0
    for k, p in ours.named_parameters():
        r = ref_named[k].grad
        if r is None or float(r.abs().max()) == 0.0:
            continue
        if k.endswith("attention.self.key.bias"):
            assert float(p.grad.abs().max()) < 1e-9 and float(r.abs().max()) < 1e-9
            continue
        worst = max(worst, float((p.grad.cpu() - r).abs().max()) / float(r.abs().max()))
        close(p.grad, r, rtol=2e-4, atol=1e-4 * float(r.abs().max()), msg=k)
        checked += 1
    print(f"  d {d} {xf_layout}: loss {float(l):.7f} vs HF {float(l_ref):.7f}; worst norm-wise gradient error {worst:.2e}")
    assert checked >= 4 + 15 * nl + 2


def test_transformer_wide_attention_dropout_training(dev, monkeypatch):
    """dropout_out > 0 (HF attention_probs_dropout_prob) at hd 160: repeatable under a fixed seed function, and the gradient is
    the gradient of the dropped forward pass (central difference of the loss along the gradient, same seeds)."""
    from multimodaltopicsegmentation_b200 import transformer
    from multimodaltopicsegmentation_b200.transformer import Transformer_segmenter

    g = torch.Generator().manual_seed(5)
    B, S, d, F, nh, w = 3, 48, 1280, 16, 8, 8
    x = torch.randn(B, S, d, generator=g).to(dev)
    lengths = torch.tensor([48, 20, 33])
    y = (torch.rand(B, S, generator=g) < 0.2).float()
    for b, n in enumerate(lengths.tolist()):
        y[b, n:] = -1
    y = y.to(dev)
    torch.manual_seed(3)
    m = Transformer_segmenter(2, d, F, num_layers=2, nheads=nh, loss_fn="FocalLoss", window_size=w, dropout_out=0.3).to(dev).train()
    monkeypatch.setattr(transformer, "ATTN_SEED_FN", lambda layer: 1000 + layer)
    loss = m.loss(x, lengths, y)
    loss.backward()
    with torch.no_grad():
        # same seeds, same masks: the loss repeats up to the summation order of the split-K products
        assert abs(float(m.loss(x, lengths, y)) - float(loss)) <= 1e-6 * abs(float(loss))
        params = [q for q in m.parameters() if q.grad is not None]
        gnorm2 = sum(float((q.grad.double() ** 2).sum()) for q in params)
        eps = 1e-2 / np.sqrt(gnorm2)
        for q in params:
            q.add_(eps * q.grad)
        lp = float(m.loss(x, lengths, y).double())
        for q in params:
            q.sub_(2 * eps * q.grad)
        lm = float(m.loss(x, lengths, y).double())
        for q in params:
            q.add_(eps * q.grad)
        fd = (lp - lm) / (2 * eps)
        print(f"  hd 160, p 0.3: directional derivative {fd:.6e} vs |grad|^2 {gnorm2:.6e}")
        assert abs(fd - gnorm2) <= 2e-2 * gnorm2
        monkeypatch.setattr(transformer, "ATTN_SEED_FN", None)
        assert float(m.loss(x, lengths, y)) != float(m.loss(x, lengths, y))


@pytest.mark.parametrize("d", [1280, 1792])
def test_transformer_wide_bf16_vs_oracle(dev, d):
    """The bf16 path's contract at hd 160 / 224: logits within 2e-2 of the logit scale, at most 0.5 % of the boundary decisions
    differing from the oracle."""
    from multimodaltopicsegmentation_b200 import ops, transformer

    F, nl, nh, w, B, S = 256, 3, 8, 16, 8, 480
    ref, ours = _pair(d, F, nl, nh, w, seed=d, head_scale=4.0)
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
        assert transformer._bf16_eligible(d, nh)
        s16, tags16 = ours(x.to(dev), lengths)
    finally:
        ops.set_precision("f32")
    s16, s32 = s16.cpu().double(), s32.cpu().double()
    assert not torch.equal(s16, s32)
    scale = float(s_ref.abs().max())
    worst = max(float((s16[b, :n] - s_ref[b, :n].double()).abs().max()) for b, n in enumerate(lengths.tolist()))
    worst32 = max(float((s32[b, :n] - s_ref[b, :n].double()).abs().max()) for b, n in enumerate(lengths.tolist()))
    n_dec = int(lengths.sum())
    flips = sum(int(a != r) for ta, tr in zip(tags16, tags_ref) for a, r in zip(ta, tr))
    print(f"  d {d} hd {d // nh}: bf16 worst |logit error| {worst:.3e} = {worst / scale:.2e} of scale {scale:.3f} "
          f"(fp32 path {worst32:.3e}); decisions differing from the oracle: {flips} of {n_dec}")
    assert worst <= 2e-2 * scale
    assert flips <= max(2, n_dec // 200)


# ------------------------------------------------------------------------------------------------------------------
# 5. user entry
# ------------------------------------------------------------------------------------------------------------------
def test_text_segmenter_transformer_d1280_steps(dev):
    from multimodaltopicsegmentation_b200 import AudioPortionDataset, TextSegmenter, to_device

    g = torch.Generator().manual_seed(4)
    lines = []
    for n in (30, 12, 21, 7):
        labs = (torch.rand(n, generator=g) < 0.2).long().tolist()
        labs[-1] = 0
        lines.append((torch.randn(n, 1280, generator=g), labs, "f"))
    ds = AudioPortionDataset(lines, {"0": 0, "1": 1}, CRF=False, truncate=False)
    batch = to_device(ds.collater([ds[i] for i in range(4)]), dev)
    torch.manual_seed(0)
    seg = TextSegmenter(2, 1280, 256, architecture="Transformer", loss_fn="FocalLoss", optimizer="Adam", lr=1e-4,
                        threshold=0.4).to(dev)
    opt = seg.configure_optimizers()["optimizer"]
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss = seg.training_step(batch, 0)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(np.isfinite(losses))
    seg.eval()
    tags = seg.predict_step(batch, 0)
    assert [len(t) for t in tags] == [30, 12, 21, 7]


def test_recurrent_longformer_hd160_vs_oracle(dev):
    """BiLSTMRestrictedMHA with H 320 and 2 heads (hd 160): scores, loss and every gradient against the oracle."""
    from multimodaltopicsegmentation_b200 import RecurrentLongformer
    from oracle import ref_torch as rt

    H, nheads, D, S, window, layers = 320, 2, 40, 64, 16, 1
    torch.manual_seed(31 + H)
    g = torch.Generator().manual_seed(77 + H)
    B = 5
    ref = rt.RecurrentLongformer(2, D, H, num_layers=layers, nheads=nheads, loss_fn="FocalLoss", window_size=window)
    ours = RecurrentLongformer(2, D, H, num_layers=layers, nheads=nheads, loss_fn="FocalLoss", window_size=window)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(dev)
    for mod in ours.modules():
        if hasattr(mod, "attention_dropout"):
            mod.attention_dropout = 0.0
    x = torch.randn(B, S, D, generator=g)
    lengths = torch.randint(3, S + 1, (B,), generator=g)
    lengths[1] = S
    y = (torch.rand(B, S, generator=g) < 0.15).float()
    for b, n in enumerate(lengths.tolist()):
        y[b, n:] = -1
    s_ref, _ = ref(x, lengths)
    s, _ = ours(x.to(dev), lengths)
    err, scale = float((s.detach().cpu().double() - s_ref.detach().double()).abs().max()), float(s_ref.abs().max())
    assert err <= 1e-4 * scale + 2e-5
    loss_ref = ref.loss(x, lengths, y)
    loss_ref.backward()
    loss = ours.loss(x.to(dev), lengths, y.to(dev))
    loss.backward()
    assert abs(float(loss) - float(loss_ref)) <= 1e-4 * abs(float(loss_ref))
    ref_grads = dict(ref.named_parameters())
    worst = 0.0
    for k, prm in ours.named_parameters():
        r = ref_grads[k].grad
        if "_global" in k:
            assert prm.grad is None and r is None
            continue
        e, sc = float((prm.grad.cpu().double() - r.double()).abs().max()), float(r.abs().max())
        tol = 1e-4 * sc + 1e-7 if "key.bias" not in k else 1e-6
        assert e <= tol, (k, e, sc)
        if "key.bias" not in k and sc > 1e-6:
            worst = max(worst, e / sc)
    print(f"  scores max|err| {err:.3e} of scale {scale:.3f}; worst norm-wise gradient error {worst:.2e} (contract 1e-04)")
    assert worst <= 1e-4
