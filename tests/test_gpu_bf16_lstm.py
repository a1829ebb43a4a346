"""The BiLSTM path under the bf16 precision switch (ops.set_precision("bf16"), inference), kernel by kernel:

  1. mts_gemm_bf16p against the float64 product of the packed operands it reads (the exact value its MMAs compute), at a
     shape for every dispatch branch: split K, the 1-SM BN = 128 kernel, a single CTA, the 224-wide 2-SM tile;
  2. mts_lstm_rec_fwd_tc_bf16 against a float64 recurrence that rounds W_hh and h to bf16 as the kernels do (and one that
     does not), for the single-pipeline, two-pipeline and CTA-pair kernels and, in child processes, the launch choices
     read from the environment;
  3. mts_pack_rows_bf16in bit for bit against the layout rule of the packed operand;
  4. the models under the switch against the oracle (BiLSTM early fusion from two bf16 modalities, BiLSTMLateFusion,
     BiRnnCrf), and embeddings of any width.

Every test prints what it measured next to the bound it asserts.  `python tests/test_gpu_bf16_lstm.py B T n_enc ...` runs
the recurrence check of part 2 in a process of its own.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H = 256


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import multimodaltopicsegmentation_b200 as m

    m.ops.device_ok()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _ops():
    from multimodaltopicsegmentation_b200 import ops

    return ops


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _packed_bits(x, kp):
    """The packed operand of fp32 rows x [rows, K] (include/mts_b200.h, "Operand preparation", A side) as int16 [rows, 2 kp]:
    per 16 columns [bf16(x) | bf16(x - trunc_tf32(x))], zeros beyond K."""
    rows, K = x.shape
    xp = torch.zeros((rows, kp), device=x.device, dtype=torch.float32)
    xp[:, :K] = x
    rest = xp - (xp.view(torch.int32) & ~0x1FFF).view(torch.float32)
    out = torch.empty((rows, kp // 16, 2, 16), device=x.device, dtype=torch.bfloat16)
    out[:, :, 0] = xp.to(torch.bfloat16).view(rows, kp // 16, 16)
    out[:, :, 1] = rest.to(torch.bfloat16).view(rows, kp // 16, 16)
    return out.view(torch.int16).view(rows, 2 * kp)


def _halves(lo):
    """packed operand [rows, kp] -> its two halves (bf16(x) and bf16(rest)) as float64 [rows, kp]"""
    rows, kp = lo.shape
    blocks = lo.contiguous().view(torch.bfloat16).view(rows, kp // 16, 2, 16).double()
    return blocks[:, :, 0].reshape(rows, kp), blocks[:, :, 1].reshape(rows, kp)


# ------------------------------------------------------------------------------------------------------------------
# 1. mts_gemm_bf16p
# ------------------------------------------------------------------------------------------------------------------
# (M, N, D), Kp = pad32(D); 148 SMs: 74 two-CTA clusters
GEMM_SHAPES = [
    (300, 2048, 104), (300, 2048, 896), (300, 2048, 1024),          # LSTM projections; Kp 1024 at M <= 1024: split K (few tiles)
    (4100, 2048, 104), (4100, 2048, 896), (4100, 2048, 1024),
    (19200, 2048, 104), (19200, 2048, 896), (19200, 2048, 1024),
    (1000, 2048, 1024),                                            # split K at the largest M that still has few tiles
    (600, 512, 4096),                                              # split K because Kp > 3072
    (2000, 200, 256), (300, 98, 64),                               # N < 256: BN = 128 kernel (N % 4 != 0: scalar epilogue)
    (100, 2048, 1024), (64, 136, 40),                              # M <= 128: one row tile (the first also split K)
    (129, 512, 96),                                                # a partial second row tile
    (700, 896, 896),                                               # 2-SM kernel with the 224-wide tile
    (513, 2688, 896),                                              # N = 2688 (the encoder's 3d)
]


@pytest.mark.parametrize("M,N,D", GEMM_SHAPES)
def test_gemm_bf16p_vs_float64(dev, M, N, D):
    """C = A_lo B_lo^T (+ bias) over the packed operands alone: per 16 columns [bf16(x) | bf16(rest)] for both, as
    PackedLstm.wih_packed_a packs the weights.  Their float64 product X_bf W_bf^T + R_x R_w^T is what the MMAs compute; the
    error against it is fp32 accumulation only (bound 1e-5 of |X_bf||W_bf|^T + |R_x||R_w|^T + |bias| per element).  Bias and
    plain epilogues, ldc > N (columns beyond N untouched) and accumulation onto C.  The norm-wise error against the float64
    product of the unrounded fp32 operands is the bf16 contract of the product; asserted loosely and printed."""
    ops = _ops()
    g = torch.Generator(device=dev).manual_seed(M * 7 + N + D)
    x = torch.randn((M, D), device=dev, generator=g)
    w = torch.randn((N, D), device=dev, generator=g) * 0.05
    bias = torch.randn((N,), device=dev, generator=g)
    kp = ops._pad32(D)
    a_lo = ops.split_tf32(x, side=ops.A_SIDE)[1]
    w_lo = ops.split_tf32(w, side=ops.A_SIDE)[1]
    xa, ra = _halves(a_lo)
    xw, rw = _halves(w_lo)
    prod = xa @ xw.T + ra @ rw.T
    mag = xa.abs() @ xw.abs().T + ra.abs() @ rw.abs().T
    b64 = bias.double()
    del xa, ra, xw, rw

    def run(epilogue, ldc, c=None, accumulate=False):
        c = torch.full((M, ldc), float("nan"), device=dev) if c is None else c
        ops._call("mts_gemm_bf16p", _ptr(a_lo), _ptr(w_lo), _ptr(bias), _ptr(c), M, N, kp, ldc, epilogue, int(accumulate),
                  ops._stream())
        return c

    def worst(c, ref, bound):
        return float(((c.double() - ref).abs() / bound.clamp_min(1e-30)).max())

    c1 = run(1, N)
    e_bias = worst(c1, prod + b64, mag + b64.abs())
    ldc = N + 36
    c0 = run(0, ldc)
    e_plain = worst(c0[:, :N], prod, mag)
    untouched = bool(torch.isnan(c0[:, N:]).all())
    base = torch.randn((M, N), device=dev, generator=g)
    ca = run(1, N, base.clone(), accumulate=True)
    e_acc = worst(ca, base.double() + prod + b64, base.double().abs() + mag + b64.abs())
    del prod, mag
    ref32 = x.double() @ w.double().T + b64
    contract = float((c1.double() - ref32).abs().max()) / float(ref32.abs().max())
    print(f"  gemm_bf16p {M} x {N} x Kp {kp}: worst |err| / (|a_bf||w_bf| + |r_a||r_w| + |bias|): bias {e_bias:.2e}, "
          f"plain ldc {ldc} {e_plain:.2e}, accumulate {e_acc:.2e} (bound 1e-5); vs the fp32 operands norm-wise {contract:.2e} "
          "(bound 1e-2)")
    assert e_bias < 1e-5 and e_plain < 1e-5 and e_acc < 1e-5, (e_bias, e_plain, e_acc)
    assert untouched, "columns beyond N of C were written"
    assert contract < 1e-2, contract


# ------------------------------------------------------------------------------------------------------------------
# 2. mts_lstm_rec_fwd_tc_bf16
# ------------------------------------------------------------------------------------------------------------------
# Against the float64 recurrence with the kernel's roundings (bf16(W_hh) bf16(h_{t-1}), RNE): what is left is fp32 state
# and accumulation, plus now and then a bf16 rounding of h that the fp32 h falls on the other side of (one such flip moves a
# pre-activation by |w| 2^-8).  Measured on a B200 (1000 W): 1.8e-5 .. 5.4e-4 max |err|, 1.44e-3 with the mixed-magnitude
# rows of B 70; bound 2x that.
REC_BOUND_EMULATED = 3e-3
# ... and well below the error against the unrounded recurrence: measured 0.02 .. 0.35 of it, while a kernel that rounds h
# by truncation instead lands at 0.85 .. 1.2 of it
REC_RATIO = 0.5
# against the unrounded float64 recurrence: the bf16 contract of the recurrence (h in [-1, 1]); measured 9e-4 .. 1.6e-3,
# 9.2e-3 with the mixed-magnitude rows; bound 2x that
REC_CONTRACT = 2e-2


def _rec_inputs(B, T, n_enc, dev):
    g = torch.Generator(device=dev).manual_seed(B * 1000 + T + n_enc)
    gx = torch.randn((n_enc, B * T, 8 * H), device=dev, generator=g)
    whh = torch.randn((n_enc, 2, 4 * H, H), device=dev, generator=g) * 0.06
    if B == 70:   # rows of very different magnitude, one zero row (the kernels scale every row by its own power of two)
        whh = whh * (10.0 ** (torch.rand((n_enc, 2, 4 * H, 1), device=dev, generator=g) * 5.0 - 4.0))
        whh[:, :, 5, :] = 0.0
    hg = torch.Generator().manual_seed(B + T)
    lengths = [T] + [int(v) for v in torch.randint(1, T + 1, (B - 1,), generator=hg)]
    if B > 2:
        lengths[2] = 1
    return gx, whh, lengths


def _rec_ref64(gx, whh, lengths, n_enc, B, T, emulate):
    """nn.LSTM over ragged episodes in float64, gate order i, f, g, o; the reverse direction runs over each episode's own
    length; zeros beyond it.  emulate: W_hh and every h_{t-1} rounded to bf16 (RNE) before the product."""
    d64 = torch.float64
    L = torch.tensor(lengths, device=gx.device)
    ar = torch.arange(B, device=gx.device)
    y = torch.zeros((B, T, n_enc * 2 * H), dtype=d64, device=gx.device)
    for e in range(n_enc):
        g_all = gx[e].view(B, T, 8 * H).double()
        for d in range(2):
            W = (whh[e, d].to(torch.bfloat16) if emulate else whh[e, d]).to(d64)
            g = g_all[:, :, d * 4 * H:(d + 1) * 4 * H]
            h = torch.zeros((B, H), dtype=d64, device=gx.device)
            c = torch.zeros_like(h)
            col = (e * 2 + d) * H
            for s in range(T):
                live = s < L
                t = torch.full_like(L, s) if d == 0 else (L - 1 - s).clamp_min(0)
                hin = h.float().to(torch.bfloat16).to(d64) if emulate else h
                z = g[ar, t] + hin @ W.T
                i, f, gg, o = z.split(H, dim=1)
                c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
                h2 = torch.sigmoid(o) * torch.tanh(c2)
                c = torch.where(live[:, None], c2, c)
                h = torch.where(live[:, None], h2, h)
                y[ar[live], t[live], col:col + H] = h2[live]
    return y


def _rec_check(B, T, n_enc, entry="mts_lstm_rec_fwd_tc_bf16"):
    """One recurrence call against both float64 references; asserts the bounds above, exact zeros beyond every length,
    bit-identical repeats and (n_enc = 1) y_corr == the packed operand of y."""
    ops = _ops()
    dev = torch.device("cuda:0")
    gx, whh, lengths = _rec_inputs(B, T, n_enc, dev)
    lens = ops.Lengths(lengths, dev, T)

    def run(with_corr=False):
        y = torch.full((B, T, n_enc * 2 * H), float("nan"), device=dev)
        corr = torch.full((B * T, 2 * H), float("nan"), device=dev) if with_corr else None
        ops._call(entry, _ptr(gx), _ptr(whh), _ptr(lens.dev), _ptr(lens.order), n_enc, B, T, H, _ptr(y), 0, _ptr(corr),
                  *((1,) if entry.endswith("_h3p") else ()), ops._stream())
        return y, corr

    y = run()[0]
    assert torch.equal(y, run()[0]), "two runs differ"
    assert not bool(torch.isnan(y).any()), "positions left unwritten"
    for b, n in enumerate(lengths):
        assert n == T or float(y[b, n:].abs().max()) == 0.0, f"episode {b}: nonzero output beyond its length {n}"
    ya = _rec_ref64(gx, whh, lengths, n_enc, B, T, emulate=True)
    e_emul = float((y.double() - ya).abs().max())
    del ya
    e_plain = float((y.double() - _rec_ref64(gx, whh, lengths, n_enc, B, T, emulate=False)).abs().max())
    env = " ".join(f"{k}={os.environ[k]}" for k in ("MTS_REC_TC", "MTS_REC_PAIR") if k in os.environ)
    print(f"  {entry} B {B} T {T} n_enc {n_enc} {env}: max|err| vs bf16-emulating float64 {e_emul:.2e} "
          f"(bound {REC_BOUND_EMULATED:.0e}, <= {REC_RATIO} x the next), vs plain float64 {e_plain:.2e} (bound {REC_CONTRACT:.0e})")
    if n_enc == 1:
        y2, corr = run(with_corr=True)
        assert torch.equal(y2, y)
        assert torch.equal(corr.view(torch.int16), _packed_bits(y.view(B * T, 2 * H), 2 * H)), "y_corr is not the packed operand of y"
    assert e_emul <= REC_BOUND_EMULATED, e_emul
    assert e_emul <= REC_RATIO * e_plain, (e_emul, e_plain)
    assert e_plain <= REC_CONTRACT, e_plain


# B 3 / 16 / 70: one tile pipeline per cluster (lstm_rec_h3.cu); B 300 / 1000: the CTA-pair kernel with two pipelines
# (lstm_rec_h3p.cu); B 70: weight rows spanning five decades and a zero row
@pytest.mark.parametrize("B,T,n_enc", [(3, 5, 1), (16, 40, 1), (16, 33, 2), (37, 61, 1), (70, 30, 1), (300, 50, 1),
                                       (300, 20, 2), (1000, 9, 1)])
def test_recurrence_bf16_vs_float64(dev, B, T, n_enc):
    _rec_check(B, T, n_enc)


@pytest.mark.parametrize("B,T,n_enc", [(16, 40, 1), (70, 30, 1), (20, 33, 2)])
def test_recurrence_bf16_pair_kernel_one_pipeline(dev, B, T, n_enc):
    """The CTA-pair kernel in bf16 mode where the default launch would not choose it (single pipeline per cluster)."""
    _rec_check(B, T, n_enc, entry="mts_lstm_rec_fwd_h3p")


@pytest.mark.parametrize("env,cases", [
    ({"MTS_REC_TC": "tf32"}, [(16, 40, 1), (70, 30, 1), (300, 20, 2)]),   # round 1's TF32 + bf16 kernel in its bf16 mode
    ({"MTS_REC_PAIR": "0"}, [(1000, 9, 1)]),                               # lstm_rec_h3.cu with two pipelines per cluster
])
def test_recurrence_bf16_environment_choices(dev, env, cases):
    """The library reads these launch choices once per process: the same check runs in a child process, which exits
    before the test returns."""
    args = [str(v) for case in cases for v in case]
    r = subprocess.run([sys.executable, os.path.abspath(__file__), *args], env={**os.environ, **env}, cwd=ROOT,
                       capture_output=True, text=True, timeout=1200)
    print(r.stdout)
    assert r.returncode == 0, r.stderr[-4000:]


# ------------------------------------------------------------------------------------------------------------------
# 3. mts_pack_rows_bf16in
# ------------------------------------------------------------------------------------------------------------------
# (B, T, T_in, D1, D2, misaligned): T_in > T = a time-cropped source (batch stride T_in D); 20 x 301 rows of Kp 1024 are more
# 8-column groups than the grid has threads; widths off 8 and a source 2 bytes off 16 take ops.pack_rows_packed's fallback
PACK_CASES = [(3, 50, 50, 384, 512, False), (5, 37, 45, 40, 24, False), (7, 13, 13, 104, 0, False),
              (20, 301, 310, 384, 640, False), (2, 29, 31, 100, 0, False), (4, 17, 20, 44, 60, False),
              (3, 9, 9, 5, 7, False), (3, 20, 24, 64, 32, True)]


@pytest.mark.parametrize("B,T,T_in,D1,D2,misaligned", PACK_CASES)
def test_pack_rows_bf16in_layout(dev, B, T, T_in, D1, D2, misaligned):
    """[x1[b, :T] | x2[b, :T]] from bf16 sources -> per 16 columns [bf16(x) | 0], zeros up to Kp, bit for bit; identical to
    mts_pack_rows_split (hi = NULL) on the same values widened to fp32 (a bf16 value is exact in TF32: its rest is 0)."""
    ops = _ops()
    g = torch.Generator(device=dev).manual_seed(B * T + D1 + D2)

    def src(D):
        v = torch.randn((B, T_in, D), device=dev, generator=g) * (10.0 ** (torch.rand((B, T_in, 1), device=dev, generator=g) * 6 - 3))
        if not misaligned:
            return v.to(torch.bfloat16)
        flat = torch.empty(v.numel() + 1, device=dev, dtype=torch.bfloat16)
        x = flat[1:].view(B, T_in, D)
        x.copy_(v)
        return x

    x1 = src(D1)
    x2 = src(D2) if D2 else None
    kp = ops._pad32(D1 + D2)
    rows = x1[:, :T] if x2 is None else torch.cat([x1[:, :T], x2[:, :T]], dim=2)
    want = _packed_bits(rows.reshape(B * T, D1 + D2).float(), kp)
    assert int(want.view(B * T, kp // 16, 2, 16)[:, :, 1].abs().max()) == 0      # (the rule itself: no remainder)
    got = {}
    if ops._packs_by_8(x1, x2):
        lo = torch.full((B * T, kp), float("nan"), device=dev)
        ops._call("mts_pack_rows_bf16in", _ptr(x1), x1.stride(0), D1, _ptr(x2), 0 if x2 is None else x2.stride(0), D2, B, T, kp,
                  _ptr(lo), ops._stream())
        got["mts_pack_rows_bf16in"] = lo
        f1, f2 = x1.float(), (None if x2 is None else x2.float())
        lo = torch.full((B * T, kp), float("nan"), device=dev)
        ops._call("mts_pack_rows_split", _ptr(f1), f1.stride(0), D1, _ptr(f2), 0 if f2 is None else f2.stride(0), D2, B, T, kp,
                  0, _ptr(lo), ops._stream())
        got["mts_pack_rows_split (fp32, hi = NULL)"] = lo
    got["ops.pack_rows_packed (bf16)"] = ops.pack_rows_packed(x1, x2, B, T)
    got["ops.pack_rows_packed (fp32)"] = ops.pack_rows_packed(x1.float(), None if x2 is None else x2.float(), B, T)
    for name, lo in got.items():
        bad = int((lo.view(torch.int16) != want).sum())
        print(f"  {name} B {B} T {T} (of {T_in}) D {D1} + {D2} -> Kp {kp}: {bad} of {want.numel()} halfwords differ from the layout rule")
        assert bad == 0, name


# ------------------------------------------------------------------------------------------------------------------
# 4. the models under the switch, against the oracle
# ------------------------------------------------------------------------------------------------------------------
def _vs_oracle(name, s, tags, s_ref, tags_ref, lengths):
    """The bf16 path's contract: logits within 2e-2 of the logit scale, <= 0.5 % of the boundary decisions differ."""
    s = s.detach().cpu().double()
    s_ref = s_ref.detach().cpu().double()
    worst = max(float((s[b, :n] - s_ref[b, :n]).abs().max()) for b, n in enumerate(lengths.tolist()))
    scale = float(s_ref.abs().max())
    n_dec = int(lengths.sum())
    flips = sum(int(bool(a) != bool(r)) for ta, tr in zip(tags, tags_ref) for a, r in zip(ta, tr))
    print(f"  {name}: worst |logit error| {worst:.3e} = {worst / scale:.2e} of the scale {scale:.2f} (bound 2e-2); "
          f"{flips} of {n_dec} decisions differ (bound {max(2, n_dec // 200)})")
    assert worst <= 2e-2 * scale, (worst, scale)
    assert flips <= max(2, n_dec // 200), flips


def _device_tags_equal(tags_dev, tags, lengths):
    td = tags_dev.cpu()
    for b, n in enumerate(lengths.tolist()):
        assert td[b, :n].tolist() == [int(v) for v in tags[b]], f"episode {b}: decode_device tags differ from forward's"
        assert bool((td[b, n:] == 0xFF).all())


def _segmenter_pair(D, seed):
    from multimodaltopicsegmentation_b200 import BiLSTM
    from oracle import ref_torch as rt

    torch.manual_seed(seed)
    ref = rt.Segmenter(2, D, H, num_layers=2, loss_fn="FocalLoss")
    with torch.no_grad():
        ref.classification.weight.mul_(4.0)   # logits of a few units: decisions that depend on the encoder's output
    ours = BiLSTM(2, D, H, num_layers=2, loss_fn="FocalLoss")
    ours.load_state_dict(ref.state_dict())
    ref.th = ours.th = 0.5
    return ref, ours


def test_early_fusion_two_bf16_modalities_vs_oracle(dev):
    """The bench's bf16 leg input form at a reduced batch: text and audio as two bf16 tensors (384 + 512), time-cropped
    (T_in > max length), lengths 1 .. T.  Scores bit-identical to the fp32 pair holding the rounded values and to the
    concatenated single tensor; decode_device's tags equal forward's."""
    ops = _ops()
    B, T, T_in, D1, D2 = 8, 300, 311, 384, 512
    ref, ours = _segmenter_pair(D1 + D2, 21)
    ours = ours.to(dev)
    g = torch.Generator().manual_seed(2121)
    x1 = torch.randn(B, T_in, D1, generator=g).to(torch.bfloat16)
    x2 = torch.randn(B, T_in, D2, generator=g).to(torch.bfloat16)
    lengths = torch.randint(1, T + 1, (B,), generator=g)
    lengths[0], lengths[1] = T, 1
    with torch.no_grad():
        s_ref, tags_ref = ref(torch.cat([x1, x2], dim=2).float(), lengths)
    d1, d2 = x1.to(dev), x2.to(dev)
    ops.set_precision("bf16")
    try:
        s, tags = ours((d1, d2), lengths)
        s_f32, _ = ours((d1.float(), d2.float()), lengths)
        s_cat, _ = ours(torch.cat([d1, d2], dim=2), lengths)
        s_dev, tags_dev, _ = ours.decode_device((d1, d2), lengths)
    finally:
        ops.set_precision("f32")
    assert torch.equal(s, s_f32) and torch.equal(s, s_cat) and torch.equal(s, s_dev)
    _device_tags_equal(tags_dev, tags, lengths)
    _vs_oracle(f"early fusion, bf16 (384 + 512), B {B} T {T}", s, tags, s_ref, tags_ref, lengths)


def test_late_fusion_bf16_vs_oracle(dev):
    """BiLSTMLateFusion (both encoders in one recurrence launch per layer, n_enc = 2) from bf16 embeddings (384, 512)."""
    from multimodaltopicsegmentation_b200 import BiLSTMLateFusion
    from oracle import ref_torch as rt

    ops = _ops()
    torch.manual_seed(22)
    B, T, D1, D2 = 8, 200, 384, 512
    ref = rt.LateFusion(2, (D1, D2), H, num_layers=2, loss_fn="FocalLoss")
    with torch.no_grad():
        ref.classification.weight.mul_(4.0)
    ours = BiLSTMLateFusion(2, (D1, D2), H, num_layers=2, loss_fn="FocalLoss")
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(dev)
    ref.th = ours.th = 0.5
    g = torch.Generator().manual_seed(2222)
    x1 = torch.randn(B, T, D1, generator=g).to(torch.bfloat16)
    x2 = torch.randn(B, T, D2, generator=g).to(torch.bfloat16)
    lengths = torch.randint(1, T + 1, (B,), generator=g)
    lengths[0], lengths[1] = T, 1
    with torch.no_grad():
        s_ref, tags_ref = ref(x1.float(), x2.float(), lengths)
    d1, d2 = x1.to(dev), x2.to(dev)
    ops.set_precision("bf16")
    try:
        s, tags = ours(d1, d2, lengths)
        s_f32, _ = ours(d1.float(), d2.float(), lengths)
        s_dev, tags_dev, _ = ours.decode_device(d1, d2, lengths)
    finally:
        ops.set_precision("f32")
    assert torch.equal(s, s_f32) and torch.equal(s, s_dev)
    _device_tags_equal(tags_dev, tags, lengths)
    _vs_oracle(f"late fusion, bf16 (384, 512), B {B} T {T}", s, tags, s_ref, tags_ref, lengths)


def test_birnncrf_bf16_viterbi_bit_exact_on_its_emissions(dev):
    """RNN -> CRF under the switch: emissions within the contract of the oracle's; Viterbi scores and paths bit-exact against
    the C oracle run on the device's own bf16-path emissions; decode_device equal to forward."""
    from multimodaltopicsegmentation_b200 import BiRnnCrf
    from oracle import c_oracle
    from oracle import ref_torch as rt

    ops = _ops()
    torch.manual_seed(23)
    B, T, D = 6, 150, 256
    ref = rt.EncoderCRF(2, D, H, num_layers=2)
    ours = BiRnnCrf(2, D, H, num_layers=2)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(dev)
    g = torch.Generator().manual_seed(2323)
    x = torch.randn(B, T, D, generator=g)
    lengths = torch.randint(1, T + 1, (B,), generator=g)
    lengths[0], lengths[1] = T, 1
    with torch.no_grad():
        emis_ref = ref.crf.fc(ref.model(x, lengths))
        _, paths_ref = ref(x, lengths)
    xd = x.to(dev)
    ops.set_precision("bf16")
    try:
        best, paths = ours(xd, lengths)
        with torch.no_grad():
            emis = ours.crf.emissions(ours.model(xd, lengths))
        best_dev, paths_dev, _ = ours.decode_device(xd, lengths)
    finally:
        ops.set_precision("f32")
    worst = max(float((emis[b, :n].cpu().double() - emis_ref[b, :n].double()).abs().max()) for b, n in enumerate(lengths.tolist()))
    scale = float(emis_ref.abs().max())
    e = np.ascontiguousarray(emis.cpu().numpy())
    b_c, p_c = c_oracle.crf_viterbi(e, lengths.numpy(), np.ascontiguousarray(ours.crf.transitions.detach().cpu().numpy()))
    differ = sum(int(a != r) for pa, pr in zip(paths, paths_ref) for a, r in zip(pa, pr))
    print(f"  BiRnnCrf bf16, B {B} T {T} D {D}: emissions worst |err| {worst:.3e} = {worst / scale:.2e} of the scale (bound 2e-2); "
          f"{differ} of {int(lengths.sum())} tags differ from the torch oracle's own decode")
    assert worst <= 2e-2 * scale, (worst, scale)
    assert np.array_equal(best.cpu().numpy(), b_c), "Viterbi scores must be bit-exact given identical emissions"
    assert torch.equal(best_dev, best)
    for b, n in enumerate(lengths.tolist()):
        assert [int(v) for v in paths[b]] == p_c[b, :n].tolist(), f"episode {b}: path differs from the C oracle"
        assert paths_dev[b, :n].cpu().tolist() == p_c[b, :n].tolist()


@pytest.mark.parametrize("D1,D2", [(100, 0), (44, 60)])
def test_bf16_switch_takes_any_width(dev, D1, D2):
    """Widths that are not multiples of 8 under the switch, from fp32 and from bf16 embeddings, time-cropped, against the
    oracle; bf16 embeddings give exactly what the fp32 tensors holding the rounded values give.  Mixed dtypes are refused."""
    ops = _ops()
    B, T, T_in = 6, 120, 125
    ref, ours = _segmenter_pair(D1 + D2, 24 + D1)
    ours = ours.to(dev)
    g = torch.Generator().manual_seed(D1 * 100 + D2)
    x = torch.randn(B, T_in, D1 + D2, generator=g)
    lengths = torch.randint(1, T + 1, (B,), generator=g)
    lengths[0], lengths[1] = T, 1

    def inputs(t):
        return t if not D2 else (t[:, :, :D1], t[:, :, D1:])

    xb = x.to(torch.bfloat16)
    with torch.no_grad():
        s_ref, tags_ref = ref(x, lengths)
        s_ref_b, tags_ref_b = ref(xb.float(), lengths)
    ops.set_precision("bf16")
    try:
        s32, tags32 = ours(inputs(x.to(dev)), lengths)
        s16, tags16 = ours(inputs(xb.to(dev)), lengths)
        s16r, _ = ours(inputs(xb.float().to(dev)), lengths)
        if D2:
            with pytest.raises(TypeError):
                ours((x[:, :, :D1].to(dev), xb[:, :, D1:].to(dev)), lengths)
    finally:
        ops.set_precision("f32")
    assert torch.equal(s16, s16r)
    _vs_oracle(f"D {D1} + {D2}, fp32 embeddings", s32, tags32, s_ref, tags_ref, lengths)
    _vs_oracle(f"D {D1} + {D2}, bf16 embeddings", s16, tags16, s_ref_b, tags_ref_b, lengths)


if __name__ == "__main__":
    # python tests/test_gpu_bf16_lstm.py B T n_enc [B T n_enc ...]: part 2's check in a process of its own
    sys.path.insert(0, ROOT)
    import multimodaltopicsegmentation_b200 as _m

    _m.ops.device_ok()
    _vals = [int(v) for v in sys.argv[1:]]
    for _i in range(0, len(_vals), 3):
        _rec_check(*_vals[_i:_i + 3])
