"""Pyramidal windowed-attention segmenter -- host-side mirror of

    Transformer_segmenter        <- models/CRF.py:508-610
    Longformer_Local_Attention   <- models/RestrictedTransformerLayer.py:65-133

The reference builds an HF `LongformerModel` and feeds it `inputs_embeds`; what runs is: embeddings
(+position ids starting at 2, +token-type row 0, LayerNorm eps 1e-12), then per layer q/k/v projections, banded
softmax attention with one-sided reach `attention_window // 2`, output projection + residual + LayerNorm,
GELU feed-forward + residual + LayerNorm (HF modeling_longformer.py:401-442, 481-639, 1060-1171).  Here the same
arithmetic runs in libmts_b200.so: tcgen05 3xTF32 GEMMs (ops.gemm_tf32x3) and the fused kernels of csrc/xfmr.cu.

The module tree below only carries PARAMETERS, with the HF names and shapes, so that a reference checkpoint
(`model.model.model.encoder.layer.N.attention.self.query.weight`, ...) loads key for key -- including the
tensors HF allocates but this path never reads (`word_embeddings`, `*_global` projections, `pooler`).

Superset note: HF's sliding-chunk implementation only accepts sequence lengths that are multiples of every
layer's window (SURVEY.md fact 5); the kernels here accept any S <= 4094 and agree with HF wherever HF runs.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .modules import _build_head, _head_decode, _head_decode_device, _head_loss, _lens

_ptr, _call, _stream, _pad32 = ops._ptr, ops._call, ops._stream, ops._pad32

LN_EPS = 1e-12  # the wrapper's layer_norm_eps argument never reaches the HF config (RestrictedTransformerLayer.py:72,82-92)


# --------------------------------------------------------------------------------------------------------
# parameter containers with HF's names
# --------------------------------------------------------------------------------------------------------
def _linear(i, o, std=0.02):
    lin = nn.Linear(i, o)
    nn.init.normal_(lin.weight, mean=0.0, std=std)  # HF _init_weights: normal(0, initializer_range), zero bias
    nn.init.zeros_(lin.bias)
    return lin


def _embedding(n, d, padding_idx=None):
    emb = nn.Embedding(n, d, padding_idx=padding_idx)
    nn.init.normal_(emb.weight, mean=0.0, std=0.02)
    if padding_idx is not None:
        with torch.no_grad():
            emb.weight[padding_idx].zero_()
    return emb


class _Embeddings(nn.Module):
    def __init__(self, d, vocab=30522, max_pos=4096, type_vocab=2, pad_token_id=1):
        super().__init__()
        self.word_embeddings = _embedding(vocab, d, pad_token_id)  # unused: the reference feeds inputs_embeds
        self.token_type_embeddings = _embedding(type_vocab, d)
        self.LayerNorm = nn.LayerNorm(d, eps=LN_EPS)
        self.position_embeddings = _embedding(max_pos, d, pad_token_id)


class _SelfAttention(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.query, self.key, self.value = _linear(d, d), _linear(d, d), _linear(d, d)
        # allocated by HF for global attention; the reference passes an all-zero global mask, so never read
        self.query_global, self.key_global, self.value_global = _linear(d, d), _linear(d, d), _linear(d, d)


class _DenseLN(nn.Module):
    def __init__(self, i, o):
        super().__init__()
        self.dense = _linear(i, o)
        self.LayerNorm = nn.LayerNorm(o, eps=LN_EPS)


class _Dense(nn.Module):
    def __init__(self, i, o):
        super().__init__()
        self.dense = _linear(i, o)


class _Attention(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.self = _SelfAttention(d)
        self.output = _DenseLN(d, d)


class _Layer(nn.Module):
    def __init__(self, d, f):
        super().__init__()
        self.attention = _Attention(d)
        self.intermediate = _Dense(d, f)
        self.output = _DenseLN(f, d)


class _Encoder(nn.Module):
    def __init__(self, d, f, n_layers):
        super().__init__()
        self.layer = nn.ModuleList([_Layer(d, f) for _ in range(n_layers)])


class _LongformerParams(nn.Module):
    """Parameter tree of HF LongformerModel (add_pooling_layer=True)."""

    def __init__(self, d, f, n_layers):
        super().__init__()
        self.embeddings = _Embeddings(d)
        self.encoder = _Encoder(d, f, n_layers)
        self.pooler = _Dense(d, d)  # HF computes the pooled output and the reference discards it


# --------------------------------------------------------------------------------------------------------
# GEMM-ready shadow copies of the weights (rebuilt only when a parameter changes)
# --------------------------------------------------------------------------------------------------------
class PackedEncoder:
    def __init__(self, params: _LongformerParams):
        self.params = params
        self.key = None
        self.layers = None

    def used_parameters(self):
        """Parameters that take part in the forward pass, in a fixed order (= the gradient order of EncoderFn)."""
        m = self.params
        out = [m.embeddings.token_type_embeddings.weight, m.embeddings.position_embeddings.weight,
               m.embeddings.LayerNorm.weight, m.embeddings.LayerNorm.bias]
        for lyr in m.encoder.layer:
            sa = lyr.attention.self
            out += [sa.query.weight, sa.query.bias, sa.key.weight, sa.key.bias, sa.value.weight, sa.value.bias,
                    lyr.attention.output.dense.weight, lyr.attention.output.dense.bias,
                    lyr.attention.output.LayerNorm.weight, lyr.attention.output.LayerNorm.bias,
                    lyr.intermediate.dense.weight, lyr.intermediate.dense.bias,
                    lyr.output.dense.weight, lyr.output.dense.bias,
                    lyr.output.LayerNorm.weight, lyr.output.LayerNorm.bias]
        return out

    PER_LAYER = 16

    def get(self):
        ps = self.used_parameters()
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if key == self.key:
            return self.layers
        layers = []
        with torch.no_grad():
            for lyr in self.params.encoder.layer:
                sa = lyr.attention.self
                wqkv = torch.cat([sa.query.weight, sa.key.weight, sa.value.weight], dim=0).contiguous()
                bqkv = torch.cat([sa.query.bias, sa.key.bias, sa.value.bias]).contiguous()
                B_ = ops.B_SIDE
                ent = {"wqkv": ops.split_tf32(wqkv, side=B_), "bqkv": bqkv,
                       "wo": ops.split_tf32(lyr.attention.output.dense.weight.detach().contiguous(), side=B_),
                       "bo": lyr.attention.output.dense.bias.detach().contiguous(),
                       "w1": ops.split_tf32(lyr.intermediate.dense.weight.detach().contiguous(), side=B_),
                       "b1": lyr.intermediate.dense.bias.detach().contiguous(),
                       "w2": ops.split_tf32(lyr.output.dense.weight.detach().contiguous(), side=B_),
                       "b2": lyr.output.dense.bias.detach().contiguous()}
                layers.append(ent)
        self.key, self.layers = key, layers
        return layers

    def pieces(self, l):
        """fp16-split copies of the two weights whose A operand comes from a LayerNorm (q/k/v and the intermediate dense):
        made on first use per weight version, inference only."""
        ent = self.get()[l]
        if "wqkv_p" not in ent:
            lyr = self.params.encoder.layer[l]
            sa = lyr.attention.self
            with torch.no_grad():
                wqkv = torch.cat([sa.query.weight, sa.key.weight, sa.value.weight], dim=0)
                ent["wqkv_p"] = ops.f16_pieces(wqkv.detach())
                ent["w1_p"] = ops.f16_pieces(lyr.intermediate.dense.weight.detach())
        return ent

    def packed_bf16(self, l):
        """bf16 path: the four dense weights packed like A operands (side 0, mts_split_tf32) so that the packed halves of
        activations and weights pair up x * w in mts_gemm_bf16p.  Made on first use per weight version, inference only."""
        ent = self.get()[l]
        if "wqkv_bf" not in ent:
            lyr = self.params.encoder.layer[l]
            sa = lyr.attention.self
            with torch.no_grad():
                wqkv = torch.cat([sa.query.weight, sa.key.weight, sa.value.weight], dim=0).contiguous()
                for name, w in (("wqkv_bf", wqkv), ("wo_bf", lyr.attention.output.dense.weight), ("w1_bf", lyr.intermediate.dense.weight),
                                ("w2_bf", lyr.output.dense.weight)):
                    ent[name] = ops.split_tf32(w.detach().contiguous(), side=ops.A_SIDE)[1]
        return ent

    def transposed(self, l):
        """hi/lo of W^T for the dX GEMMs of the backward pass (made on first use per weight version)."""
        ent = self.get()[l]
        if "wqkv_t" not in ent:
            lyr = self.params.encoder.layer[l]
            sa = lyr.attention.self
            with torch.no_grad():
                wqkv = torch.cat([sa.query.weight, sa.key.weight, sa.value.weight], dim=0)
                B_ = ops.B_SIDE
                ent["wqkv_t"] = ops.split_tf32(wqkv.t().contiguous(), side=B_)
                ent["wo_t"] = ops.split_tf32(lyr.attention.output.dense.weight.detach().t().contiguous(), side=B_)
                ent["w1_t"] = ops.split_tf32(lyr.intermediate.dense.weight.detach().t().contiguous(), side=B_)
                ent["w2_t"] = ops.split_tf32(lyr.output.dense.weight.detach().t().contiguous(), side=B_)
        return ent


def _split_src(x):
    """Encoder input -> (x1, x2, B, S, d): x is [B,S,d] embeddings (x2 None) or an early-fusion pair (x1 [B,S,D1], x2 [B,S,D2]),
    which the embeddings LayerNorm reads in place as [x1 | x2], d = D1 + D2."""
    if isinstance(x, tuple):
        x1, x2 = x
        return x1, x2, x1.shape[0], x1.shape[1], x1.shape[2] + x2.shape[2]
    return (x, None, *x.shape)


def _ln(mode, a, b, typ, gamma, beta, B, S, d, want_split, save, lens=None, a2=None):
    """mode 0: embeddings LN over x=a [B,S,d] with position table b (lens given: ragged output rows), or over x = [a | a2]
    when the second source a2 is given; mode 1: LN(a + b) over [M,d] rows (M = B, S = 1)."""
    M = lens.N if lens is not None else B * S
    dev = a.device
    y = torch.empty((M, d), device=dev, dtype=torch.float32)
    kp = _pad32(d)
    hi = lo = None
    if want_split:  # the GEMM's `hi` operand is the fp32 tensor itself: y stands in for it when no K padding is needed
        lo = torch.empty((M, kp), device=dev, dtype=torch.float32)
        hi = None if kp == d else torch.empty((M, kp), device=dev, dtype=torch.float32)
    pre = torch.empty((M, d), device=dev, dtype=torch.float32) if save else None
    stats = torch.empty((M, 2), device=dev, dtype=torch.float32) if save else None
    if mode == 0 and a2 is not None:
        _call("mts_embed_ln_fwd_pair", _ptr(a), a.stride(0), a.shape[2], _ptr(a2), a2.stride(0), a2.shape[2], _ptr(b), _ptr(typ),
              _ptr(gamma), _ptr(beta), B, S, LN_EPS, _ptr(y), _ptr(hi), _ptr(lo), kp, _ptr(pre), _ptr(stats),
              _ptr(lens.dev) if lens is not None else 0, _ptr(lens.offs) if lens is not None else 0, _stream())
    elif mode == 0:
        _call("mts_embed_ln_fwd", _ptr(a), a.stride(0), _ptr(b), _ptr(typ), _ptr(gamma), _ptr(beta), B, S, d, LN_EPS,
              _ptr(y), _ptr(hi), _ptr(lo), kp, _ptr(pre), _ptr(stats), _ptr(lens.dev) if lens is not None else 0,
              _ptr(lens.offs) if lens is not None else 0, _stream())
    else:
        _call("mts_add_ln_fwd", _ptr(a), _ptr(b), _ptr(gamma), _ptr(beta), M, d, LN_EPS, _ptr(y), _ptr(hi), _ptr(lo), kp,
              _ptr(pre), _ptr(stats), _stream())
    return y, (y if (want_split and hi is None) else hi), lo, pre, stats


def _ln_f16(mode, a, b, typ, gamma, beta, B, S, d, lens=None, a2=None):
    """_ln for inference with the fp16-split operand of mts_gemm_f16x3 as the second output: (y, pieces [M, 2, K64], scale [M])."""
    M = lens.N if lens is not None else B * S
    dev = a.device
    k64 = (d + 63) // 64 * 64
    y = torch.empty((M, d), device=dev, dtype=torch.float32)
    pieces = torch.empty((M, 2, k64), device=dev, dtype=torch.float16)
    scale = torch.empty((M,), device=dev, dtype=torch.float32)
    if mode == 0 and a2 is not None:
        _call("mts_embed_ln_fwd_f16_pair", _ptr(a), a.stride(0), a.shape[2], _ptr(a2), a2.stride(0), a2.shape[2], _ptr(b), _ptr(typ),
              _ptr(gamma), _ptr(beta), B, S, LN_EPS, _ptr(y), _ptr(pieces), k64, _ptr(scale), _ptr(lens.dev) if lens is not None else 0,
              _ptr(lens.offs) if lens is not None else 0, _stream())
    elif mode == 0:
        _call("mts_embed_ln_fwd_f16", _ptr(a), a.stride(0), _ptr(b), _ptr(typ), _ptr(gamma), _ptr(beta), B, S, d, LN_EPS, _ptr(y),
              _ptr(pieces), k64, _ptr(scale), _ptr(lens.dev) if lens is not None else 0, _ptr(lens.offs) if lens is not None else 0,
              _stream())
    else:
        _call("mts_add_ln_fwd_f16", _ptr(a), _ptr(b), _ptr(gamma), _ptr(beta), M, d, LN_EPS, _ptr(y), _ptr(pieces), k64, _ptr(scale),
              _stream())
    return y, pieces, scale


# The dense layers fed by a LayerNorm (q/k/v projection, intermediate dense) run over fp16-split operands in inference
# (mts_gemm_f16x3: 6 instead of 8 MMAs per 32 k, half the operand bytes; 1.27x on those products at configs[2]);
# MTS_XF_F16X3=0 keeps every product on mts_gemm_tf32x3.
F16X3 = __import__("os").environ.get("MTS_XF_F16X3", "1") != "0"


# Token layout inside the encoder: "ragged" (default) keeps rows only for the sum(len) valid sentences, so the dense
# layers, LayerNorms and GELU do no work on padding (45 % of the rows at configs[2]); "padded" is the reference's
# [B*S] layout.  Valid positions come out identical either way (padded keys are masked); with the ragged layout the
# padded positions of the returned hidden state are exact zeros instead of the reference's don't-care values.
LAYOUT = __import__("os").environ.get("MTS_XF_LAYOUT", "ragged")
# Folding the residual adds into the dense layers' epilogues (LayerNorm then reads one tensor instead of two) is
# bit-identical but NOT faster: measured at configs[2] LayerNorm 5.05 -> 4.46 ms, GEMMs 17.0 -> 17.9 ms per step -- the
# GEMM sits on the L2 throughput cap, so the residual read costs there what it saves here.  Off by default.
FOLD_RESIDUAL = __import__("os").environ.get("MTS_XF_FOLD", "0") == "1"


# Keep-masks of the hidden-state dropout: callable (site, rows, d, p, device) -> bool/uint8/float [rows, d].
# None = Bernoulli(1 - p) from torch's CUDA generator.  Tests install a function that replays recorded masks.
DROPOUT_MASK_FN = None


# Seeds of the attention-probability dropout: callable (layer) -> int below 2^63.  None = drawn from torch's CPU generator
# (so torch.manual_seed makes a training run repeatable; no device synchronisation).  The keep-mask itself is a pure
# function of the seed and the (episode, head, query, key) indices (csrc/common.cuh attn_keep_scale) and is regenerated
# by the backward kernels: no mask tensor is stored.
ATTN_SEED_FN = None


def attn_seed(layer):
    if ATTN_SEED_FN is not None:
        return int(ATTN_SEED_FN(layer))
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def band_attention(qkv, ld, lens, offs, B, S, nheads, hd, reach, out, out_hi, out_lo, kp, lse, p_attn=0.0, seed=0):
    """mts_band_attn_fwd, or its dropout form when p_attn > 0 (training)."""
    if p_attn > 0:
        _call("mts_band_attn_fwd_dropout", _ptr(qkv), ld, _ptr(lens.dev), offs, B, S, nheads, hd, reach, _ptr(out), _ptr(out_hi),
              _ptr(out_lo), kp, _ptr(lse), float(p_attn), int(seed), _stream())
    else:
        _call("mts_band_attn_fwd", _ptr(qkv), ld, _ptr(lens.dev), offs, B, S, nheads, hd, reach, _ptr(out), _ptr(out_hi),
              _ptr(out_lo), kp, _ptr(lse), _stream())


def _keep_mask(site, rows, d, p, device):
    if DROPOUT_MASK_FN is not None:
        return DROPOUT_MASK_FN(site, rows, d, p, device)
    return torch.rand((rows, d), device=device) >= p


def _drop(t, site, p, masks):
    """In-place inverted dropout of a [rows, d] activation; the keep-mask is remembered for the backward pass."""
    keep = _keep_mask(site, t.shape[0], t.shape[1], p, t.device)
    t.mul_(keep).mul_(1.0 / (1.0 - p))
    masks.append(keep)
    return t


def _f16x3_eligible(M, d, F, ops_mod):
    """mts_gemm_f16x3 is served by the 2-SM GEMM (M, N >= 256) and the fp16-pieces LayerNorm (d <= 1024); the out-proj and the
    output dense keep mts_gemm_tf32x3 (their A operands come from the attention kernel / the GELU epilogue)."""
    return (F16X3 and ops_mod.GEMM_IMPL != "simt" and ops_mod.PRECISION != "bf16" and M >= 256 and d % 4 == 0 and d <= 1024
            and 3 * d >= 256 and _pad32(d) == d)


def encoder_forward_f16(x, lens, packed: PackedEncoder, nheads, reaches):
    """Inference pass of the encoder with the LayerNorm-fed dense layers on fp16-split operands:

        emb LN -> (h, h pieces) -> QKV [f16x3] -> banded attention -> out-proj [tf32x3] -> LN(t + h) -> (y, y pieces)
               -> intermediate dense + GELU [f16x3 when F >= 256, writes (z, z_lo)] -> output dense [tf32x3] -> LN(u + y) -> ...

    Same arithmetic contract as encoder_forward (fp32-grade products: relative error ~2^-22 instead of ~2^-19)."""
    x, x2, B, S, d = _split_src(x)
    ragged = LAYOUT == "ragged"
    M = lens.N if ragged else B * S
    offs = _ptr(lens.offs) if ragged else 0
    dev = x.device
    hd = d // nheads
    m = packed.params
    emb = m.embeddings
    h, h_p, h_s = _ln_f16(0, x, emb.position_embeddings.weight.detach(), emb.token_type_embeddings.weight.detach()[0],
                          emb.LayerNorm.weight.detach(), emb.LayerNorm.bias.detach(), B, S, d, lens if ragged else None, a2=x2)
    n_layers = len(m.encoder.layer)
    for l in range(n_layers):
        lyr = m.encoder.layer[l]
        ent = packed.pieces(l)
        F = lyr.intermediate.dense.out_features
        qkv = torch.empty((M, 3 * d), device=dev, dtype=torch.float32)
        ops.gemm_f16x3(h_p, h_s, ent["wqkv_p"][0], ent["wqkv_p"][1], ent["bqkv"], qkv, M, 3 * d, epilogue=1)
        a = torch.empty((M, d), device=dev, dtype=torch.float32)
        a_lo = torch.empty((M, d), device=dev, dtype=torch.float32)
        _call("mts_band_attn_fwd", _ptr(qkv), 3 * d, _ptr(lens.dev), offs, B, S, nheads, hd, reaches[l], 0, _ptr(a), _ptr(a_lo), d,
              0, _stream())
        t = torch.empty((M, d), device=dev, dtype=torch.float32)
        ops.gemm_tf32x3(a, a_lo, ent["wo"][0], ent["wo"][1], ent["bo"], t, M, d, epilogue=1)
        ln1 = lyr.attention.output.LayerNorm
        kf = _pad32(F)
        z_hl = torch.empty((2, M, kf), device=dev, dtype=torch.float32)
        if F >= 256 and kf == F:
            y, y_p, y_s = _ln_f16(1, t, h, None, ln1.weight.detach(), ln1.bias.detach(), M, 1, d)
            ops.gemm_f16x3(y_p, y_s, ent["w1_p"][0], ent["w1_p"][1], ent["b1"], z_hl[0], M, F, epilogue=2, out_lo=z_hl[1])
        else:   # narrow feed-forward: the TF32 + bf16 product (GELU + operand pair in its epilogue when the width allows)
            y, y_hi, y_lo, _, _ = _ln(1, t, h, None, ln1.weight.detach(), ln1.bias.detach(), M, 1, d, True, False)
            if kf == F:
                _call("mts_gemm_tf32x3_gelu_pair", _ptr(y_hi), _ptr(y_lo), _ptr(ent["w1"][0]), _ptr(ent["w1"][1]), _ptr(ent["b1"]),
                      _ptr(z_hl[0]), _ptr(z_hl[1]), M, F, y_hi.shape[1], _stream())
            else:
                zp = torch.empty((M, F), device=dev, dtype=torch.float32)
                ops.gemm_tf32x3(y_hi, y_lo, ent["w1"][0], ent["w1"][1], ent["b1"], zp, M, F, epilogue=1)
                _call("mts_gelu_split", _ptr(zp), F, M, F, kf, 0, _ptr(z_hl[0]), _ptr(z_hl[1]), _stream())
        u = torch.empty((M, d), device=dev, dtype=torch.float32)
        ops.gemm_tf32x3(z_hl[0], z_hl[1], ent["w2"][0], ent["w2"][1], ent["b2"], u, M, d, epilogue=1)
        ln2 = lyr.output.LayerNorm
        if l + 1 < n_layers:
            h, h_p, h_s = _ln_f16(1, u, y, None, ln2.weight.detach(), ln2.bias.detach(), M, 1, d)
        else:
            h = _ln(1, u, y, None, ln2.weight.detach(), ln2.bias.detach(), M, 1, d, False, False)[0]
    if ragged:  # back to the caller's [B,S,d] layout, padded sentences zero
        out = torch.empty((B, S, d), device=dev, dtype=torch.float32)
        _call("mts_ragged_copy", _ptr(h), _ptr(out), _ptr(lens.dev), _ptr(lens.offs), B, S, d, 1, 0.0, _stream())
        return out
    return h.view(B, S, d)


def _bf16_eligible(d, nheads):
    """The bf16 encoder (ops.set_precision("bf16")) serves widths that are whole 32-column blocks (the packed operands carry no K
    padding) and the head dims of the bf16 attention kernel; everything else keeps the fp32 path."""
    return (ops.PRECISION == "bf16" and _pad32(d) == d and d <= 2048
            and ops._lib.load().mts_band_attn_bf16_supported(d // nheads) != 0)


def encoder_forward_bf16(x, lens, packed: PackedEncoder, nheads, reaches):
    """Inference pass of the encoder under the bf16 precision switch: every dense layer is a bf16 x bf16 product
    (mts_gemm_bf16p and its epilogue forms) over the packed operands the producers write, q/k/v are bf16 and the banded
    attention runs on bf16 operands (mts_band_attn_fwd_bf16):

        emb LN (h, h_lo) -> QKV [bf16p_out16, bf16 qkv] -> band_attn_fwd_bf16 -> a_lo -> out-proj [bf16p] -> LN(t + h) (y, y_lo)
               -> intermediate dense + GELU [bf16p_gelu_pair: z, z_lo] -> output dense [bf16p] -> LN(u + y) -> ...

    The residual stream, the LayerNorm statistics, the softmax, all accumulators and the returned hidden state are fp32.
    x may be fp32 or bfloat16 embeddings (read as they are: half the bytes), or an early-fusion pair of either."""
    x, x2, B, S, d = _split_src(x)
    ragged = LAYOUT == "ragged"
    M = lens.N if ragged else B * S
    offs = _ptr(lens.offs) if ragged else 0
    dev = x.device
    hd = d // nheads
    m = packed.params
    emb = m.embeddings
    pos, typ = emb.position_embeddings.weight.detach(), emb.token_type_embeddings.weight.detach()[0]
    if x.dtype == torch.bfloat16:
        h = torch.empty((M, d), device=dev, dtype=torch.float32)
        h_lo = torch.empty((M, d), device=dev, dtype=torch.float32)
        if x2 is not None:
            _call("mts_embed_ln_fwd_bf16in_pair", _ptr(x), x.stride(0), x.shape[2], _ptr(x2), x2.stride(0), x2.shape[2], _ptr(pos),
                  _ptr(typ), _ptr(emb.LayerNorm.weight.detach()), _ptr(emb.LayerNorm.bias.detach()), B, S, LN_EPS, _ptr(h), _ptr(h_lo),
                  d, _ptr(lens.dev) if ragged else 0, offs, _stream())
        else:
            _call("mts_embed_ln_fwd_bf16in", _ptr(x), x.stride(0), _ptr(pos), _ptr(typ), _ptr(emb.LayerNorm.weight.detach()),
                  _ptr(emb.LayerNorm.bias.detach()), B, S, d, LN_EPS, _ptr(h), _ptr(h_lo), d, _ptr(lens.dev) if ragged else 0, offs,
                  _stream())
    else:
        h, _, h_lo, _, _ = _ln(0, x, pos, typ, emb.LayerNorm.weight.detach(), emb.LayerNorm.bias.detach(), B, S, d, True, False,
                               lens if ragged else None, a2=x2)
    n_layers = len(m.encoder.layer)
    for l in range(n_layers):
        lyr = m.encoder.layer[l]
        ent = packed.packed_bf16(l)
        F = lyr.intermediate.dense.out_features
        qkv = torch.empty((M, 3 * d), device=dev, dtype=torch.bfloat16)
        _call("mts_gemm_bf16p_out16", _ptr(h_lo), _ptr(ent["wqkv_bf"]), _ptr(ent["bqkv"]), _ptr(qkv), M, 3 * d, d, 3 * d, _stream())
        a_lo = torch.empty((M, d), device=dev, dtype=torch.float32)
        _call("mts_band_attn_fwd_bf16", _ptr(qkv), 3 * d, M, _ptr(lens.dev), offs, B, S, nheads, hd, reaches[l], 0, _ptr(a_lo), d, 0,
              _stream())
        t = torch.empty((M, d), device=dev, dtype=torch.float32)
        _call("mts_gemm_bf16p", _ptr(a_lo), _ptr(ent["wo_bf"]), _ptr(ent["bo"]), _ptr(t), M, d, d, d, 1, 0, _stream())
        ln1 = lyr.attention.output.LayerNorm
        y, _, y_lo, _, _ = _ln(1, t, h, None, ln1.weight.detach(), ln1.bias.detach(), M, 1, d, True, False)
        kf = _pad32(F)
        z_hl = torch.empty((2, M, kf), device=dev, dtype=torch.float32)
        if kf == F and d <= 3072:
            _call("mts_gemm_bf16p_gelu_pair", _ptr(y_lo), _ptr(ent["w1_bf"]), _ptr(ent["b1"]), _ptr(z_hl[0]), _ptr(z_hl[1]), M, F, d,
                  _stream())
        else:
            zp = torch.empty((M, F), device=dev, dtype=torch.float32)
            _call("mts_gemm_bf16p", _ptr(y_lo), _ptr(ent["w1_bf"]), _ptr(ent["b1"]), _ptr(zp), M, F, d, F, 1, 0, _stream())
            _call("mts_gelu_split", _ptr(zp), F, M, F, kf, 0, _ptr(z_hl[0]), _ptr(z_hl[1]), _stream())
        u = torch.empty((M, d), device=dev, dtype=torch.float32)
        _call("mts_gemm_bf16p", _ptr(z_hl[1]), _ptr(ent["w2_bf"]), _ptr(ent["b2"]), _ptr(u), M, d, kf, d, 1, 0, _stream())
        ln2 = lyr.output.LayerNorm
        h, _, h_lo, _, _ = _ln(1, u, y, None, ln2.weight.detach(), ln2.bias.detach(), M, 1, d, l + 1 < n_layers, False)
    if ragged:  # back to the caller's [B,S,d] layout, padded sentences zero
        out = torch.empty((B, S, d), device=dev, dtype=torch.float32)
        _call("mts_ragged_copy", _ptr(h), _ptr(out), _ptr(lens.dev), _ptr(lens.offs), B, S, d, 1, 0.0, _stream())
        return out
    return h.view(B, S, d)


def encoder_forward(x, lens, packed: PackedEncoder, nheads, reaches, save, p_hidden=0.0, p_attn=0.0):
    """x [B,S,d] -> last hidden state [B,S,d].  `reaches[l]` = one-sided window of layer l.
    With save=True also returns what the backward pass needs.
    p_hidden > 0 applies HF's `hidden_dropout_prob` at its three sites (after the embeddings LayerNorm and on the
    two dense outputs that feed a residual LayerNorm: modeling_longformer.py LongformerEmbeddings / SelfOutput /
    Output) as plain element-wise passes -- a training-time regulariser, not part of the timed inference path.
    p_attn > 0 applies HF's `attention_probs_dropout_prob` inside the attention kernel (one seed per layer).
    x may also be an early-fusion pair (x1 [B,S,D1], x2 [B,S,D2]) of the sources the embeddings LayerNorm reads in place."""
    _, _, B, S, d = _split_src(x)
    ragged = LAYOUT == "ragged"
    M = lens.N if ragged else B * S
    if not save and p_hidden == 0 and p_attn == 0 and _bf16_eligible(d, nheads):
        return encoder_forward_bf16(x, lens, packed, nheads, reaches), None
    if not save and p_hidden == 0 and p_attn == 0 and not FOLD_RESIDUAL and _f16x3_eligible(M, d, 0, ops):
        return encoder_forward_f16(x, lens, packed, nheads, reaches), None
    x, x2 = _split_src(x)[:2]
    offs = _ptr(lens.offs) if ragged else 0
    dev = x.device
    hd = d // nheads
    m = packed.params
    layers = packed.get()
    emb = m.embeddings
    h, h_hi, h_lo, pre0, st0 = _ln(0, x, emb.position_embeddings.weight.detach(), emb.token_type_embeddings.weight.detach()[0],
                                   emb.LayerNorm.weight.detach(), emb.LayerNorm.bias.detach(), B, S, d, True, save,
                                   lens if ragged else None, a2=x2)
    masks = []
    if p_hidden > 0:
        h = _drop(h, 0, p_hidden, masks)
        h_hi, h_lo = ops.split_tf32(h)
        if _pad32(d) == d:
            h_hi = h
    saved = {"emb": (pre0, st0), "layers": [], "ragged": ragged, "masks": masks, "p_hidden": p_hidden, "p_attn": p_attn}
    # Optional (MTS_XF_FOLD=1), inference only: the two residual adds folded into the dense layers' epilogues
    # (accumulate onto the residual, which is dead as an operand by then) -- bit-identical sums, see FOLD_RESIDUAL.
    fold = FOLD_RESIDUAL and not save and p_hidden == 0 and _pad32(d) == d
    for l, ent in enumerate(layers):
        lyr = m.encoder.layer[l]
        F = lyr.intermediate.dense.out_features
        qkv = torch.empty((M, 3 * d), device=dev, dtype=torch.float32)
        ops.gemm_tf32x3(h_hi, h_lo, ent["wqkv"][0], ent["wqkv"][1], ent["bqkv"], qkv, M, 3 * d, epilogue=1)
        kp = _pad32(d)
        lse = torch.empty((B, nheads, S), device=dev, dtype=torch.float32) if save else None
        seed = attn_seed(l) if p_attn > 0 else 0
        if kp == d:  # the attention output is its own `hi` operand; the kernel adds the correction operand
            a = torch.empty((M, d), device=dev, dtype=torch.float32)
            a_lo = torch.empty((M, kp), device=dev, dtype=torch.float32)
            a_hi = a
            band_attention(qkv, 3 * d, lens, offs, B, S, nheads, hd, reaches[l], None, a_hi, a_lo, kp, lse, p_attn, seed)
        else:  # widths that are not a multiple of 32: plain output, then the generic (zero-padding) split
            a = torch.empty((M, d), device=dev, dtype=torch.float32)
            a_hl = torch.empty((2, M, kp), device=dev, dtype=torch.float32)
            a_hi, a_lo = a_hl[0], a_hl[1]
            band_attention(qkv, 3 * d, lens, offs, B, S, nheads, hd, reaches[l], a, None, None, 0, lse, p_attn, seed)
            _call("mts_split_tf32", _ptr(a), d, M, d, kp, ops.A_SIDE, _ptr(a_hi), _ptr(a_lo), _stream())
        ln1 = lyr.attention.output.LayerNorm
        if fold:  # t + h formed by the GEMM epilogue, in h (its operand role ended with the QKV product)
            ops.gemm_tf32x3(a_hi, a_lo, ent["wo"][0], ent["wo"][1], ent["bo"], h, M, d, epilogue=1, accumulate=True)
            y, y_hi, y_lo, pre1, st1 = _ln(1, h, None, None, ln1.weight.detach(), ln1.bias.detach(), M, 1, d, True, False)
        else:
            t = torch.empty((M, d), device=dev, dtype=torch.float32)
            ops.gemm_tf32x3(a_hi, a_lo, ent["wo"][0], ent["wo"][1], ent["bo"], t, M, d, epilogue=1)
            if p_hidden > 0:
                _drop(t, 1 + 2 * l, p_hidden, masks)
            y, y_hi, y_lo, pre1, st1 = _ln(1, t, h, None, ln1.weight.detach(), ln1.bias.detach(), M, 1, d, True, save)
        kf = _pad32(F)
        z_hl = torch.empty((2, M, kf), device=dev, dtype=torch.float32)
        if not save and kf == F and y_hi.shape[1] <= 3072:  # inference: GELU and the operand pair of z in the GEMM epilogue
            zp = z = None
            _call("mts_gemm_tf32x3_gelu_pair", _ptr(y_hi), _ptr(y_lo), _ptr(ent["w1"][0]), _ptr(ent["w1"][1]), _ptr(ent["b1"]),
                  _ptr(z_hl[0]), _ptr(z_hl[1]), M, F, y_hi.shape[1], _stream())
        else:
            zp = torch.empty((M, F), device=dev, dtype=torch.float32)
            ops.gemm_tf32x3(y_hi, y_lo, ent["w1"][0], ent["w1"][1], ent["b1"], zp, M, F, epilogue=1)
            z = torch.empty((M, F), device=dev, dtype=torch.float32) if save else None
            _call("mts_gelu_split", _ptr(zp), F, M, F, kf, _ptr(z), _ptr(z_hl[0]), _ptr(z_hl[1]), _stream())
        ln2 = lyr.output.LayerNorm
        h_in = h
        last = l == len(layers) - 1
        if fold:
            ops.gemm_tf32x3(z_hl[0], z_hl[1], ent["w2"][0], ent["w2"][1], ent["b2"], y, M, d, epilogue=1, accumulate=True)
            h, h_hi, h_lo, pre2, st2 = _ln(1, y, None, None, ln2.weight.detach(), ln2.bias.detach(), M, 1, d, not last, False)
        else:
            u = torch.empty((M, d), device=dev, dtype=torch.float32)
            ops.gemm_tf32x3(z_hl[0], z_hl[1], ent["w2"][0], ent["w2"][1], ent["b2"], u, M, d, epilogue=1)
            if p_hidden > 0:
                _drop(u, 2 + 2 * l, p_hidden, masks)
            h, h_hi, h_lo, pre2, st2 = _ln(1, u, y, None, ln2.weight.detach(), ln2.bias.detach(), M, 1, d, not last, save)
        if save:
            saved["layers"].append({"h_in": h_in, "qkv": qkv, "lse": lse, "a": a, "attn_seed": seed, "pre1": pre1, "st1": st1,
                                    "y": y, "zp": zp, "z": z, "pre2": pre2, "st2": st2})
    if ragged:  # back to the caller's [B,S,d] layout, padded sentences zero
        out = torch.empty((B, S, d), device=dev, dtype=torch.float32)
        _call("mts_ragged_copy", _ptr(h), _ptr(out), _ptr(lens.dev), _ptr(lens.offs), B, S, d, 1, 0.0, _stream())
        return out, saved
    return h.view(B, S, d), saved


def _encoder_input(parts):
    """[x] -> x; [x1, x2] -> the pair (x1, x2) when the embeddings LayerNorm can read it in place (widths multiples of 4, sources
    aligned to the load width: 16 bytes for fp32, 8 for bf16, batch strides multiples of 4), else its concatenation on the
    device (same values: the single-source path)."""
    if len(parts) == 1:
        return parts[0]
    align = 16 if parts[0].dtype == torch.float32 else 8
    if all(t.shape[2] % 4 == 0 and t.data_ptr() % align == 0 and t.stride(0) % 4 == 0 for t in parts):
        return tuple(parts)
    return torch.cat(parts, dim=-1)


class EncoderFn(torch.autograd.Function):
    """Differentiable w.r.t. the encoder parameters (the input embeddings, a tensor or an early-fusion pair, are data)."""

    @staticmethod
    def forward(ctx, x, lens, packed, nheads, reaches, p_hidden, p_attn, *params):
        need = any(ctx.needs_input_grad)
        out, saved = encoder_forward(x, lens, packed, nheads, reaches, save=need, p_hidden=p_hidden, p_attn=p_attn)
        if need:
            ctx.saved, ctx.lens, ctx.packed, ctx.nheads, ctx.reaches = saved, lens, packed, nheads, reaches
            ctx.shape = _split_src(x)[2:]
        return out

    @staticmethod
    def backward(ctx, dout):
        from .transformer_bwd import encoder_backward

        grads = encoder_backward(ctx, dout.contiguous())
        ctx.saved = None
        return (None, None, None, None, None, None, None, *grads)


class Longformer_Local_Attention(nn.Module):
    def __init__(self, d_model: int, nhead: int, n_layers: int, dim_feedforward: int = 2048, window_size=3,
                 dropout: float = 0.1, dropout_attention: float = 0.1, layer_norm_eps: float = 1e-5, tagset_size=2,
                 device=None, max_position_embedding=4096) -> None:
        super().__init__()
        if d_model % nhead != 0:
            raise ValueError(f"The hidden size ({d_model}) is not a multiple of the number of attention heads ({nhead})")
        windows = list(window_size) if isinstance(window_size, (list, tuple)) else [window_size] * n_layers
        assert len(windows) == n_layers, "`len(config.attention_window)` should equal `config.num_hidden_layers`"
        for i, wdw in enumerate(windows):  # HF LongformerSelfAttention.__init__ asserts
            assert wdw % 2 == 0, f"`attention_window` for layer {i} has to be an even value. Given {wdw}"
            assert wdw > 0, f"`attention_window` for layer {i} has to be positive. Given {wdw}"
        self.d_model, self.nhead, self.windows = d_model, nhead, windows
        self.reaches = [wdw // 2 for wdw in windows]
        self.hidden_dropout, self.attention_dropout = float(dropout), float(dropout_attention)
        self.max_positions = max_position_embedding
        self.model = _LongformerParams(d_model, dim_feedforward, n_layers)
        self._packed = None

    def packed(self):
        if self._packed is None:
            self._packed = PackedEncoder(self.model)
        return self._packed

    def forward(self, src, lengths):
        """src: [B, S, d_model] embeddings, or an early-fusion pair (text [B, S, D1], audio [B, S, D2]) with D1 + D2 = d_model,
        which the embeddings LayerNorm reads in place instead of their concatenation (same results, bit for bit)."""
        pair = isinstance(src, (tuple, list))
        if pair:
            if len(src) != 2 or not all(torch.is_tensor(t) for t in src):
                raise TypeError("src: an early-fusion input is a pair (text, audio) of [B, S, D_i] tensors")
            if src[0].dtype != src[1].dtype:
                raise TypeError(f"src: both members of the pair must have one dtype, got {src[0].dtype} and {src[1].dtype}")
        parts = list(src) if pair else [src]
        if torch.is_tensor(parts[0]) and parts[0].dtype == torch.bfloat16:   # bf16 embeddings: inference under ops.set_precision("bf16")
            parts = [ops._check(t, "src", torch.bfloat16) for t in parts]
            if ops.PRECISION != "bf16":
                raise TypeError("src: bfloat16 embeddings belong to the bf16 path (ops.set_precision('bf16')); the fp32 path takes fp32")
        else:
            parts = [ops._check(t, "src") for t in parts]
        x = parts[0]
        if pair:
            x2 = parts[1]
            if x.dim() != 3 or x2.dim() != 3 or x.shape[:2] != x2.shape[:2] or x.shape[2] + x2.shape[2] != self.d_model:
                raise ValueError(f"expected a pair of [B, S, D_i] embeddings with D1 + D2 = {self.d_model}, got {tuple(x.shape)} "
                                 f"and {tuple(x2.shape)}")
        elif x.dim() != 3 or x.shape[2] != self.d_model:
            raise ValueError(f"expected [B, S, {self.d_model}] embeddings, got {tuple(x.shape)}")
        if x.shape[1] + 2 > self.max_positions:
            raise IndexError(f"sequence length {x.shape[1]} exceeds the position table ({self.max_positions} rows, "
                             "position ids start at 2)")
        p_hidden = self.hidden_dropout if self.training else 0.0
        p_attn = self.attention_dropout if self.training else 0.0   # HF attention_probs_dropout_prob (RestrictedTransformerLayer.py:92)
        parts = [t if (t.stride(2) == 1 and t.stride(1) == t.shape[2]) else t.contiguous() for t in parts]
        lens = lengths if isinstance(lengths, ops.Lengths) else ops.Lengths(lengths, x.device, x.shape[1])
        packed = self.packed()
        params = packed.used_parameters()
        if not (torch.is_grad_enabled() and any(p.requires_grad for p in params)):  # inference: nothing saved
            if x.dtype == torch.bfloat16 and not (p_hidden == 0 and p_attn == 0 and _bf16_eligible(self.d_model, self.nhead)):
                # a shape or dropout setting the bf16 encoder does not serve: the fp32 path, on the same values
                parts = [t.float() for t in parts]
            return encoder_forward(_encoder_input(parts), lens, packed, self.nhead, self.reaches, save=False, p_hidden=p_hidden,
                                   p_attn=p_attn)[0]
        if x.dtype == torch.bfloat16:
            raise NotImplementedError("bfloat16 embeddings serve inference only (ops.set_precision('bf16')): train in fp32")
        return EncoderFn.apply(_encoder_input(parts), lens, packed, self.nhead, self.reaches, p_hidden, p_attn, *params)


class Transformer_segmenter(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=6, nheads=8, dropout_in=0.0, dropout_out=0.0,
                 batch_first=True, loss_fn="CrossEntropy", positional_encoding=True, threshold=None, restricted=True,
                 window_size=127, alpha=0.9, gamma=2):
        super().__init__()
        if not restricted:
            raise NotImplementedError("only the windowed (restricted) encoder is on the B200 hot path")
        self.embedding_dim, self.hidden_dim, self.tagset_size = embedding_dim, hidden_dim, tagset_size
        self.device = "cuda"
        self.no_mask = True
        windows = [win * window_size for win in range(num_layers, 0, -1)]  # pyramidal, models/CRF.py:529
        self.model = Longformer_Local_Attention(embedding_dim, nheads, num_layers, hidden_dim, window_size=windows,
                                                dropout=dropout_in, dropout_attention=dropout_out, layer_norm_eps=1e-5,
                                                tagset_size=tagset_size, device=None, max_position_embedding=4096)
        _build_head(self, embedding_dim, tagset_size, loss_fn, threshold, alpha, gamma)

    # xs: [B, S, embedding_dim] embeddings or an early-fusion pair (text, audio) of [B, S, D_i] (Longformer_Local_Attention.forward)
    def loss(self, xs, lengths, tags, segments=None, global_count=None):
        if segments is not None:
            raise NotImplementedError("the auxiliary cosine loss (segments=...) is outside the B200 hot path")
        lens = _lens(lengths, xs)
        return _head_loss(self, self.model(xs, lens), lens, tags, global_count)

    def forward(self, xs, lenghts, threshold=0.4):
        lens = _lens(lenghts, xs)
        with torch.no_grad():
            return _head_decode(self, self.model(xs, lens), lens, threshold)

    def decode_device(self, xs, lenghts, threshold=0.4):
        lens = _lens(lenghts, xs)
        with torch.no_grad():
            return (*_head_decode_device(self, self.model(xs, lens), lens, threshold), lens)
