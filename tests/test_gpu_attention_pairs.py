"""Early-fusion pairs (text [B, S, D1], audio [B, S, D2]) fed to the windowed-attention segmenters: the embeddings LayerNorm
reads both sources in place instead of their concatenation.  Every check is BIT-IDENTICAL against the same computation given
torch.cat(pair, -1):

  * the three pair entry points (mts_embed_ln_fwd_pair, mts_embed_ln_fwd_f16_pair, mts_embed_ln_fwd_bf16in_pair) against the
    single-source entries, padded and ragged rows, time-cropped views, every length 1..S, and the rejected splits;
  * Transformer_segmenter: fp32 inference on the fp16-split path (d 896) and the TF32 path (d 1280), fp32 training with both
    dropouts, bf16 inference from fp32 and bf16 pairs, in both token layouts; the error paths;
  * BiLSTMRestrictedMHA (RecurrentLongformer): scores, tags, loss and gradients;
  * TextSegmenter from a keep_modalities=True loader through DevicePrefetcher, both architectures.

Sizes: the tensor-core GEMMs split long contractions (K >= 1024 with few output tiles) over atomically summed partial
products, whose order is not fixed from run to run.  The model-level checks use sizes at which no product splits, so that
the two inputs can be compared bit for bit.
"""
import json
import os
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SPLITS = [(384, 512), (768, 512), (4, 1020)]
EPS = 1e-12


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import multimodaltopicsegmentation_b200 as m

    m.ops.device_ok()
    return torch.device("cuda:0")


@pytest.fixture(params=["ragged", "padded"])
def xf_layout(request, monkeypatch):
    from multimodaltopicsegmentation_b200 import transformer

    monkeypatch.setattr(transformer, "LAYOUT", request.param)
    return request.param


@pytest.fixture
def bf16_precision():
    from multimodaltopicsegmentation_b200 import ops

    ops.set_precision("bf16")
    try:
        yield
    finally:
        ops.set_precision("f32")


@pytest.fixture
def ln_calls(monkeypatch):
    """Names of the library entries transformer.py calls (to see which embeddings LayerNorm ran)."""
    from multimodaltopicsegmentation_b200 import ops, transformer

    names = []

    def rec(name, *args):
        names.append(name)
        return ops._call(name, *args)

    monkeypatch.setattr(transformer, "_call", rec)
    return names


def _p(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    from multimodaltopicsegmentation_b200 import ops

    return ops._stream()


def _call(name, *args):
    from multimodaltopicsegmentation_b200 import ops

    return ops._call(name, *args)


def _rc(name, *args):
    """Status code of a direct call (no exception)."""
    from multimodaltopicsegmentation_b200 import _lib

    return getattr(_lib.load(), name)(*args)


def same(a, b, msg=""):
    assert a.dtype == b.dtype and a.shape == b.shape, msg
    assert torch.equal(a, b), f"{msg}: max |diff| {float((a.double() - b.double()).abs().max()):.3e}"


def split(x, D1):
    return x[..., :D1].contiguous(), x[..., D1:].contiguous()


# ------------------------------------------------------------------------------------------------------------------
# 1. kernels
# ------------------------------------------------------------------------------------------------------------------
def _kernel_case(dev, D1, D2, dtype, seed):
    """Two time-cropped sources (views [:, :S] of [B, S0, D_i]: batch stride S0 * D_i > S * D_i), their concatenation, the
    parameters, and the lengths 1..S in shuffled order."""
    from multimodaltopicsegmentation_b200 import ops

    B = S = 16
    S0 = 19
    d = D1 + D2
    g = torch.Generator().manual_seed(seed)
    x1 = torch.randn(B, S0, D1, generator=g).to(dtype).to(dev)[:, :S]
    x2 = torch.randn(B, S0, D2, generator=g).to(dtype).to(dev)[:, :S]
    assert x1.stride(0) == S0 * D1 and x2.stride(0) == S0 * D2
    xc = torch.cat((x1, x2), -1).contiguous()
    prm = [torch.randn(S + 2, d, generator=g), torch.randn(d, generator=g), 1 + 0.1 * torch.randn(d, generator=g),
           torch.randn(d, generator=g)]
    pos, typ, gamma, beta = [t.to(dev) for t in prm]
    lens = ops.Lengths(torch.randperm(S, generator=g) + 1, dev, S)
    return B, S, d, x1, x2, xc, pos, typ, gamma, beta, lens


def _rows(lens, ragged, B, S):
    return lens.N if ragged else B * S


@pytest.mark.parametrize("ragged", [False, True], ids=["padded", "ragged"])
@pytest.mark.parametrize("D1,D2", SPLITS)
def test_embed_ln_fwd_pair_fp32(dev, D1, D2, ragged):
    """fp32 pair: y, the TF32 operand pair (with and without a separate hi / K padding), the pre-LN sum and (mean, rstd)."""
    B, S, d, x1, x2, xc, pos, typ, gamma, beta, lens = _kernel_case(dev, D1, D2, torch.float32, D1 + D2)
    M = _rows(lens, ragged, B, S)
    lp, op = (_p(lens.dev), _p(lens.offs)) if ragged else (0, 0)
    for kp, with_hi in ((d, False), ((d + 31) // 32 * 32 + 32, True)):
        outs = []
        for pair in (True, False):
            y = torch.full((M, d), 7.0, device=dev)
            hi = torch.full((M, kp), 7.0, device=dev) if with_hi else None
            lo = torch.full((M, kp), 7.0, device=dev)
            pre = torch.full((M, d), 7.0, device=dev)
            st = torch.full((M, 2), 7.0, device=dev)
            if pair:
                _call("mts_embed_ln_fwd_pair", _p(x1), x1.stride(0), D1, _p(x2), x2.stride(0), D2, _p(pos), _p(typ), _p(gamma),
                      _p(beta), B, S, EPS, _p(y), _p(hi), _p(lo), kp, _p(pre), _p(st), lp, op, _stream())
            else:
                _call("mts_embed_ln_fwd", _p(xc), xc.stride(0), _p(pos), _p(typ), _p(gamma), _p(beta), B, S, d, EPS, _p(y), _p(hi),
                      _p(lo), kp, _p(pre), _p(st), lp, op, _stream())
            outs.append((y, hi, lo, pre, st))
        for name, a, b in zip(("y", "hi", "lo", "sum", "stats"), *outs):
            if a is not None:
                same(a, b, f"{name} kp {kp}")
        ref = torch.nn.functional.layer_norm(xc.double() + pos[2:S + 2].double() + typ.double(), (d,), gamma.double(),
                                             beta.double(), EPS).view(B * S, d)
        if ragged:
            ref = torch.cat([ref.view(B, S, d)[b, :n] for b, n in enumerate(lens.host)])
        assert float((outs[0][0].double() - ref).abs().max()) < 1e-4


@pytest.mark.parametrize("ragged", [False, True], ids=["padded", "ragged"])
@pytest.mark.parametrize("D1,D2", SPLITS)
def test_embed_ln_fwd_f16_pair(dev, D1, D2, ragged):
    """fp16-split form: y, the two fp16 pieces (zero beyond d) and the row scale; widths past 1024 are rejected like the
    single-source entry rejects them."""
    B, S, d, x1, x2, xc, pos, typ, gamma, beta, lens = _kernel_case(dev, D1, D2, torch.float32, 3 * D1 + D2)
    M = _rows(lens, ragged, B, S)
    lp, op = (_p(lens.dev), _p(lens.offs)) if ragged else (0, 0)
    k64 = (d + 63) // 64 * 64 + 64
    outs, rcs = [], []
    for pair in (True, False):
        y = torch.full((M, d), 7.0, device=dev)
        pieces = torch.full((M, 2, k64), 7.0, device=dev, dtype=torch.float16)
        scale = torch.full((M,), 7.0, device=dev)
        if pair:
            rcs.append(_rc("mts_embed_ln_fwd_f16_pair", _p(x1), x1.stride(0), D1, _p(x2), x2.stride(0), D2, _p(pos), _p(typ),
                           _p(gamma), _p(beta), B, S, EPS, _p(y), _p(pieces), k64, _p(scale), lp, op, _stream()))
        else:
            rcs.append(_rc("mts_embed_ln_fwd_f16", _p(xc), xc.stride(0), _p(pos), _p(typ), _p(gamma), _p(beta), B, S, d, EPS, _p(y),
                           _p(pieces), k64, _p(scale), lp, op, _stream()))
        outs.append((y, pieces, scale))
    if d > 1024:
        assert rcs == [-2, -2]
        return
    assert rcs == [0, 0]
    for name, a, b in zip(("y", "pieces", "scale"), *outs):
        same(a, b, name)
    assert float(outs[0][1][:, :, d:].abs().max()) == 0.0


@pytest.mark.parametrize("ragged", [False, True], ids=["padded", "ragged"])
@pytest.mark.parametrize("D1,D2", SPLITS)
def test_embed_ln_fwd_bf16in_pair(dev, D1, D2, ragged):
    """bf16 sources: y and its packed operand."""
    B, S, d, x1, x2, xc, pos, typ, gamma, beta, lens = _kernel_case(dev, D1, D2, torch.bfloat16, 5 * D1 + D2)
    M = _rows(lens, ragged, B, S)
    lp, op = (_p(lens.dev), _p(lens.offs)) if ragged else (0, 0)
    outs = []
    for pair in (True, False):
        y = torch.full((M, d), 7.0, device=dev)
        lo = torch.full((M, d), 7.0, device=dev)
        if pair:
            _call("mts_embed_ln_fwd_bf16in_pair", _p(x1), x1.stride(0), D1, _p(x2), x2.stride(0), D2, _p(pos), _p(typ), _p(gamma),
                  _p(beta), B, S, EPS, _p(y), _p(lo), d, lp, op, _stream())
        else:
            _call("mts_embed_ln_fwd_bf16in", _p(xc), xc.stride(0), _p(pos), _p(typ), _p(gamma), _p(beta), B, S, d, EPS, _p(y), _p(lo),
                  d, lp, op, _stream())
        outs.append((y, lo))
    same(outs[0][0], outs[1][0], "y")
    same(outs[0][1], outs[1][1], "lo")


def test_embed_ln_fwd_pair_rejects_unsupported_splits(dev):
    """MTS_E_UNSUPPORTED (-2): a width that is not a multiple of 4, a source off its load width, a batch stride that is not a
    multiple of 4.  Nothing is launched."""
    B, S, d = 2, 8, 896
    pos = torch.zeros(S + 2, d, device=dev)
    vec = torch.zeros(d, device=dev)
    y = torch.zeros(B * S, d, device=dev)
    lo = torch.zeros(B * S, d, device=dev)
    pieces = torch.zeros(B * S, 2, 896, device=dev, dtype=torch.float16)
    scale = torch.zeros(B * S, device=dev)
    buf32 = torch.zeros(B * S * d + 8, device=dev)
    buf16 = torch.zeros(B * S * d + 8, device=dev, dtype=torch.bfloat16)

    def fp32(src1, bs1, D1, src2, bs2, D2):
        return (_rc("mts_embed_ln_fwd_pair", src1, bs1, D1, src2, bs2, D2, _p(pos), _p(vec), _p(vec), _p(vec), B, S, EPS, _p(y), 0,
                    _p(lo), d, 0, 0, 0, 0, _stream()),
                _rc("mts_embed_ln_fwd_f16_pair", src1, bs1, D1, src2, bs2, D2, _p(pos), _p(vec), _p(vec), _p(vec), B, S, EPS, _p(y),
                    _p(pieces), 896, _p(scale), 0, 0, _stream()))

    def bf16(src1, bs1, D1, src2, bs2, D2):
        return (_rc("mts_embed_ln_fwd_bf16in_pair", src1, bs1, D1, src2, bs2, D2, _p(pos), _p(vec), _p(vec), _p(vec), B, S, EPS,
                    _p(y), _p(lo), d, 0, 0, _stream()),)

    a32, a16 = buf32.data_ptr(), buf16.data_ptr()
    b32, b16 = a32 + 4 * S * 384 * B, a16 + 2 * S * 384 * B
    assert fp32(a32, S * 384, 384, b32, S * 512, 512) == (0, 0)
    assert bf16(a16, S * 384, 384, b16, S * 512, 512) == (0,)
    torch.cuda.synchronize()
    assert fp32(a32, S * 382, 382, b32, S * 514, 514) == (-2, -2)              # D1 % 4 != 0
    assert bf16(a16, S * 382, 382, b16, S * 514, 514) == (-2,)
    assert fp32(a32 + 4, S * 384, 384, b32, S * 512, 512) == (-2, -2)          # first source on 4 bytes
    assert fp32(a32, S * 384, 384, b32 + 8, S * 512, 512) == (-2, -2)          # second source on 8 bytes
    assert bf16(a16 + 2, S * 384, 384, b16, S * 512, 512) == (-2,)             # bf16 source on 2 bytes
    assert bf16(a16, S * 384, 384, b16 + 4, S * 512, 512) == (-2,)             # bf16 source on 4 bytes
    assert fp32(a32, S * 384 + 2, 384, b32, S * 512, 512) == (-2, -2)          # batch stride % 4 != 0
    assert bf16(a16, S * 384, 384, b16, S * 512 + 2, 512) == (-2,)
    assert fp32(a32, S * 384, 384, 0, S * 512, 512) == (-1, -1)                # no second source: a bad argument


# ------------------------------------------------------------------------------------------------------------------
# 2. Transformer_segmenter
# ------------------------------------------------------------------------------------------------------------------
def _segmenter(dev, d, F, nl, nh, w, seed, loss_fn="FocalLoss", **kw):
    from multimodaltopicsegmentation_b200.transformer import Transformer_segmenter

    torch.manual_seed(seed)
    m = Transformer_segmenter(2, d, F, num_layers=nl, nheads=nh, loss_fn=loss_fn, window_size=w, **kw).to(dev)
    m.th = 0.5
    return m


def _batch(B, S, d, lo, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, d, generator=g)
    lengths = torch.randint(lo, S + 1, (B,), generator=g)
    lengths[0] = S
    lengths[1] = 1
    y = (torch.rand(B, S, generator=g) < 0.2).float()
    for b, n in enumerate(lengths.tolist()):
        y[b, n:] = -1
    return x.to(dev), lengths, y.to(dev)


def _inference_same(m, pair, xc, lengths, y):
    with torch.no_grad():
        s1, t1, _ = m.decode_device(pair, lengths)
        s2, t2, _ = m.decode_device(xc, lengths)
        same(s1, s2, "scores")
        same(t1, t2, "device tags")
        assert m(pair, lengths)[1] == m(xc, lengths)[1]
        same(m.loss(pair, lengths, y), m.loss(xc, lengths, y), "loss")


def test_transformer_pair_fp32_f16_path(dev, xf_layout, ln_calls):
    """d 896 (384 + 512): the fp16-split inference path, whose embeddings LayerNorm is mts_embed_ln_fwd_f16_pair."""
    from multimodaltopicsegmentation_b200 import ops, transformer

    B, S, D1, D2 = 4, 160, 384, 512
    m = _segmenter(dev, D1 + D2, 256, 2, 8, 8, seed=1).eval()
    x, lengths, y = _batch(B, S, D1 + D2, 80, 2, dev)
    M = int(lengths.sum()) if xf_layout == "ragged" else B * S
    assert transformer._f16x3_eligible(M, D1 + D2, 0, ops)
    _inference_same(m, split(x, D1), x, lengths, y)
    assert "mts_embed_ln_fwd_f16_pair" in ln_calls and "mts_embed_ln_fwd_f16" in ln_calls


def test_transformer_pair_fp32_tf32_path(dev, xf_layout, ln_calls):
    """d 1280 (768 + 512, hd 160): the TF32 path (mts_embed_ln_fwd_pair).  At least ~2 400 token rows, so that no product of the
    1280-deep contractions splits K."""
    B, S, D1, D2 = 8, 480, 768, 512
    m = _segmenter(dev, D1 + D2, 256, 2, 8, 8, seed=3).eval()
    x, lengths, y = _batch(B, S, D1 + D2, 300, 4, dev)
    lengths[1] = 300
    _inference_same(m, split(x, D1), x, lengths, y)
    assert "mts_embed_ln_fwd_pair" in ln_calls and "mts_embed_ln_fwd" in ln_calls


def test_transformer_pair_fp32_training(dev, xf_layout, monkeypatch, ln_calls):
    """Loss and every gradient with hidden-state dropout (fixed masks) and attention dropout (fixed seeds).  d 320 (128 + 192),
    fewer than 1024 tokens: no contraction of the forward or backward pass is deep enough to be split."""
    from multimodaltopicsegmentation_b200 import transformer

    def masks(site, rows, d, p, device):
        return (torch.rand((rows, d), generator=torch.Generator().manual_seed(100 + site)) >= p).to(device)

    monkeypatch.setattr(transformer, "DROPOUT_MASK_FN", masks)
    monkeypatch.setattr(transformer, "ATTN_SEED_FN", lambda layer: 1000 + layer)
    B, S, D1, D2 = 3, 96, 128, 192
    m = _segmenter(dev, D1 + D2, 96, 2, 8, 8, seed=5, dropout_in=0.1, dropout_out=0.2).train()
    x, lengths, y = _batch(B, S, D1 + D2, 20, 6, dev)
    grads = []
    for src in (split(x, D1), x):
        m.zero_grad(set_to_none=True)
        loss = m.loss(src, lengths, y)
        loss.backward()
        grads.append((loss.detach(), {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}))
    same(grads[0][0], grads[1][0], "loss")
    assert grads[0][1].keys() == grads[1][1].keys() and len(grads[0][1]) >= 4 + 16 * 2
    for k in grads[0][1]:
        same(grads[0][1][k], grads[1][1][k], k)
    assert "mts_embed_ln_fwd_pair" in ln_calls


def test_transformer_pair_bf16(dev, xf_layout, bf16_precision, ln_calls):
    """Under the bf16 switch: fp32 pair (mts_embed_ln_fwd_pair feeding the bf16 encoder), bf16 pair
    (mts_embed_ln_fwd_bf16in_pair), and a bf16 pair at a head dim the bf16 encoder does not serve (hd 48: widened to fp32)."""
    from multimodaltopicsegmentation_b200 import transformer

    B, S, D1, D2 = 4, 160, 384, 512
    m = _segmenter(dev, D1 + D2, 256, 2, 8, 8, seed=7).eval()
    assert transformer._bf16_eligible(D1 + D2, 8)
    x, lengths, y = _batch(B, S, D1 + D2, 80, 8, dev)
    _inference_same(m, split(x, D1), x, lengths, y)
    xb = x.to(torch.bfloat16)
    _inference_same(m, split(xb, D1), xb, lengths, y)
    assert "mts_embed_ln_fwd_bf16in_pair" in ln_calls and "mts_embed_ln_fwd_pair" in ln_calls
    m48 = _segmenter(dev, 384, 64, 2, 8, 8, seed=9).eval()
    assert not transformer._bf16_eligible(384, 8)
    xb = x[..., :384].to(torch.bfloat16)
    _inference_same(m48, split(xb, 192), xb, lengths, y)


def test_transformer_pair_fallbacks_and_errors(dev, ln_calls):
    """Splits the kernels reject are concatenated on the device (same results); the error paths of a malformed pair."""
    from multimodaltopicsegmentation_b200 import ops

    B, S, d = 3, 64, 896
    m = _segmenter(dev, d, 64, 1, 8, 8, seed=11).eval()
    x, lengths, y = _batch(B, S, d, 10, 12, dev)
    _inference_same(m, split(x, 382), x, lengths, y)                                 # D1 % 4 != 0
    buf = torch.empty(B * S * 384 + 1, device=dev)
    x1 = buf[1:].view(B, S, 384)                                                     # dense rows, but 4 bytes off
    x1.copy_(x[..., :384])
    _inference_same(m, (x1, x[..., 384:].contiguous()), x, lengths, y)
    assert not any(n.startswith("mts_embed_ln") and n.endswith("_pair") for n in ln_calls)
    with pytest.raises(ValueError):
        m.decode_device((x[..., :384].contiguous(), x[..., 384:-4].contiguous()), lengths)   # D1 + D2 != d_model
    with pytest.raises(ValueError):
        m.decode_device((x[:, :, :384], x[:, :32, 384:]), lengths)                          # different time axes
    with pytest.raises(TypeError):
        m.decode_device((x[..., :384].contiguous(), x[..., 384:].to(torch.bfloat16)), lengths)
    with pytest.raises(TypeError):                                                         # bf16 only under the switch
        m.decode_device(split(x.to(torch.bfloat16), 384), lengths)
    ops.set_precision("bf16")
    try:
        m.train()
        with pytest.raises(NotImplementedError):
            m.loss(split(x.to(torch.bfloat16), 384), lengths, y)
    finally:
        ops.set_precision("f32")


# ------------------------------------------------------------------------------------------------------------------
# 3. BiLSTMRestrictedMHA
# ------------------------------------------------------------------------------------------------------------------
def test_recurrent_longformer_pair(dev, monkeypatch):
    """Only the first block's RNN reads the pair; scores, tags, loss and every gradient equal those for the concatenation."""
    from multimodaltopicsegmentation_b200 import RecurrentLongformer, transformer

    monkeypatch.setattr(transformer, "ATTN_SEED_FN", lambda layer: 77 + layer)
    B, S, D1, D2, H = 4, 96, 384, 512, 64
    torch.manual_seed(13)
    m = RecurrentLongformer(2, D1 + D2, H, num_layers=2, nheads=2, loss_fn="FocalLoss", window_size=16).to(dev)
    m.th = 0.5
    x, lengths, y = _batch(B, S, D1 + D2, 10, 14, dev)
    m.eval()
    _inference_same(m, split(x, D1), x, lengths, y)
    m.train()
    grads = []
    for src in (split(x, D1), x):
        m.zero_grad(set_to_none=True)
        loss = m.loss(src, lengths, y)
        loss.backward()
        grads.append((loss.detach(), {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}))
    same(grads[0][0], grads[1][0], "loss")
    assert grads[0][1].keys() == grads[1][1].keys() and grads[0][1]
    for k in grads[0][1]:
        same(grads[0][1][k], grads[1][1][k], k)


# ------------------------------------------------------------------------------------------------------------------
# 4. TextSegmenter from a keep_modalities loader
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fusion_episodes(tmp_path_factory):
    """Five episodes of 384-d text and 512-d audio on disk, loaded as the concatenation and with keep_modalities=True."""
    from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed

    root = tmp_path_factory.mktemp("fusion")
    rng = np.random.default_rng(17)
    labs, files = {}, []
    for sub in ("text", "audio"):
        os.makedirs(root / sub)
    for i, n in enumerate((30, 12, 21, 7, 25)):
        name = f"ep{i}"
        np.save(root / "text" / f"{name}.npy", rng.standard_normal((n, 384)).astype(np.float32))
        np.save(root / "audio" / f"{name}.npy", rng.standard_normal((n, 512)).astype(np.float32))
        labs[name] = (rng.random(n) < 0.25).astype(int).tolist()
        files.append(f"{name}.npy")
    with open(root / "labs.pkl", "wb") as f:
        pickle.dump(labs, f)
    with open(root / "split.json", "w") as f:
        json.dump({"train": files, "test": [], "validation": []}, f)
    args = (str(root / "text") + "+" + str(root / "audio"), str(root / "labs.pkl"))
    cat = load_dataset_from_precomputed(*args, split=str(root / "split.json"))[0][0]
    sep = load_dataset_from_precomputed(*args, split=str(root / "split.json"), keep_modalities=True)[0][0]
    assert [e[2] for e in cat] == [e[2] for e in sep] and isinstance(sep[0][0], tuple)
    return cat, sep


def _host_batches(cat, sep):
    """The collater's batch of the concatenated episodes, and the same batch with src_tokens as the (text, audio) pair; pinned."""
    from multimodaltopicsegmentation_b200 import AudioPortionDataset
    from multimodaltopicsegmentation_b200.EncoderDataset import _pad_episodes

    ds = AudioPortionDataset(cat, {"0": 0, "1": 1}, CRF=False, truncate=False)
    cat_batch = ds.collater([ds[i] for i in range(len(ds))])
    pair_batch = dict(cat_batch)
    pair_batch["src_tokens"] = tuple(_pad_episodes([e[0][k] for e in sep], False, 0) for k in range(2))
    assert torch.equal(torch.cat(pair_batch["src_tokens"], -1), cat_batch["src_tokens"])

    def pin(b):
        return {k: (v.pin_memory() if torch.is_tensor(v) and k != "src_lengths" else
                    tuple(t.pin_memory() for t in v) if isinstance(v, tuple) else v) for k, v in b.items()}

    return pin(pair_batch), pin(cat_batch)


@pytest.mark.parametrize("arch", ["Transformer", "BiLSTMRestrictedMHA"])
def test_text_segmenter_pair_batches(dev, fusion_episodes, arch):
    from multimodaltopicsegmentation_b200 import DevicePrefetcher, TextSegmenter

    pair_host, cat_host = _host_batches(*fusion_episodes)
    torch.manual_seed(19)
    seg = TextSegmenter(2, 896, 64, architecture=arch, loss_fn="FocalLoss", optimizer="Adam", lr=1e-4, threshold=0.4,
                        attention_window=16).to(dev)
    for mod in seg.modules():   # no attention dropout: the two training-mode losses are compared bit for bit
        if hasattr(mod, "attention_dropout"):
            mod.attention_dropout = 0.0
    pair, cat = (next(iter(DevicePrefetcher([b], dev))) for b in (pair_host, cat_host))
    assert isinstance(pair["src_tokens"], tuple) and pair["src_tokens"][0].is_cuda
    seg.train()
    same(seg.training_step(pair, 0).detach(), seg.training_step(cat, 0).detach(), "training loss")
    seg.eval()
    with torch.no_grad():
        same(seg.validation_step(pair, 0), seg.validation_step(cat, 0), "validation loss")
        assert seg.test_step(pair, 0) == seg.test_step(cat, 0)
        seg.device_metrics = False
        r_pair, r_cat = seg.test_step(pair, 0), seg.test_step(cat, 0)
        seg.device_metrics = True
        assert r_pair == r_cat
        scores, _, lens = seg.model.decode_device(pair["src_tokens"], pair["src_lengths"])
        th_pair = seg.threshold_search(scores, pair["tgt_tokens"], lens)
        scores, _, lens = seg.model.decode_device(cat["src_tokens"], cat["src_lengths"])
        assert th_pair == seg.threshold_search(scores, cat["tgt_tokens"], lens)
        tags_pair = list(seg.predict_batches(DevicePrefetcher([pair_host, pair_host], dev)))
        tags_cat = list(seg.predict_batches(DevicePrefetcher([cat_host, cat_host], dev)))
    assert tags_pair == tags_cat and [len(t) for t in tags_pair[0]] == pair_host["src_lengths"].tolist()
