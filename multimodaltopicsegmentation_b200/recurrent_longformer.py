"""`BiLSTMRestrictedMHA` -- host-side mirror of

    RecurrentLongformerBlock   <- models/CRF.py:636-684
    RecurrentLongformer        <- models/CRF.py:764-858
    Longformer_Local_Attention(just_mha=True) <- models/RestrictedTransformerLayer.py:65-133

One block = a one-layer bi-LSTM followed by an FFN-less windowed multi-head attention in which the FORWARD hidden states
are the queries (and values) and the BACKWARD hidden states are the keys.  The attention layer comes from the
reference's `models/longformer_noffn.py`, whose source is missing from the repository (SURVEY.md fact 7); what it does
was read from the byte code of `models/__pycache__/longformer_noffn.cpython-310.pyc`:

    LongformerLayer.__init__        only `self.attention = LongformerAttention(config, layer_id)` -- no intermediate / output
    LongformerLayer.forward         is_index_masked = attention_mask < 0; returns self.attention(...)[0] (a tensor)
    LongformerAttention.__init__    only `self.self = LongformerSelfAttention(config, layer_id)` -- no output dense / LayerNorm
    LongformerAttention.forward     returns the self-attention outputs unchanged (no residual, no LayerNorm)
    LongformerSelfAttention.forward query = Q(hidden_states); key = K(external_input) if given else K(hidden_states);
                                    value = V(hidden_states); everything after that is HF 4.24's sliding-chunk attention
                                    (query / sqrt(head_dim), one-sided window attention_window[layer_id] // 2, padded keys
                                    masked, fp32 softmax, rows of padded queries zeroed, dropout on the probabilities)

so a block's output is softmax_band(Q(h_fwd) K(h_bwd)^T / sqrt(hd)) V(h_fwd), [B, S, hidden_dim], zero at padded
positions.  Here the projections are tcgen05 GEMMs and the attention is the banded kernel of csrc/attn_tc.cu /
csrc/xfmr.cu (the same one the pyramidal encoder uses), forward and backward.

Superset notes: the reference asserts `inputs.shape[1] == 3600` and re-pads every block's LSTM output to 3600 rows
(CRF.py:660-684); here any S works -- the time axis simply stays S and rows beyond len_b stay zero, which is what the
re-padding produces.  HF's sliding chunks additionally need S to be a multiple of the window; the kernels do not.
The reference's CrossEntropy branch reads `self.tagset_size`, which `RecurrentLongformer.__init__` never sets
(AttributeError on construction); here it is set from the constructor argument.
Parity: the GPU tests compare with the torch twin of this composition (HF's own LongformerSelfAttention with the key
projection redirected as the byte code does); the reference class itself cannot be imported (source-less module) --
"parity unpinned" for this row, DESIGN.md.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .modules import RNN, _build_head, _head_decode, _head_decode_device, _head_loss, _lens
from .transformer import attn_seed, band_attention
from .transformer_bwd import _dense_param_grads

_ptr, _call, _stream, _pad32 = ops._ptr, ops._call, ops._stream, ops._pad32


# --------------------------------------------------------------------------------------------------------
# parameter containers with the reference's names: transformer.model.attention.self.{query,key,value}[_global]
# --------------------------------------------------------------------------------------------------------
class _SelfAttention(nn.Module):
    def __init__(self, d):
        super().__init__()
        # a bare LongformerLayer is not a PreTrainedModel: nn.Linear's default initialisation applies
        self.query, self.key, self.value = nn.Linear(d, d), nn.Linear(d, d), nn.Linear(d, d)
        # allocated by LongformerSelfAttention.__init__ for global attention, never read on this path
        self.query_global, self.key_global, self.value_global = nn.Linear(d, d), nn.Linear(d, d), nn.Linear(d, d)


class _Attention(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.self = _SelfAttention(d)


class _NoffnLayer(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.attention = _Attention(d)


class _PackedMha:
    """GEMM-ready copies of the three projections (rebuilt when a parameter changes)."""

    def __init__(self, sa: _SelfAttention):
        self.sa = sa
        self.key = None
        self.ent = None

    def params(self):
        sa = self.sa
        return [sa.query.weight, sa.query.bias, sa.key.weight, sa.key.bias, sa.value.weight, sa.value.bias]

    def get(self):
        ps = self.params()
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if key != self.key:
            with torch.no_grad():
                self.ent = {"w": [ops.split_tf32(ps[2 * j].detach().contiguous(), side=ops.B_SIDE) for j in range(3)],
                            "b": [ps[2 * j + 1].detach().contiguous() for j in range(3)]}
            self.key = key
        return self.ent

    def transposed(self):
        ent = self.get()
        if "wt" not in ent:
            with torch.no_grad():
                ent["wt"] = [ops.split_tf32(self.params()[2 * j].detach().t().contiguous(), side=ops.B_SIDE) for j in range(3)]
        return ent


def _mha_forward(xq, xk, lens, packed: _PackedMha, nheads, reach, save, p_attn=0.0, seed=0):
    """xq, xk [B,S,d] (views with unit inner stride are fine) -> attention output [B,S,d]."""
    B, S, d = xq.shape
    M = B * S
    hd = d // nheads
    dev = xq.device
    ent = packed.get()
    xq2 = xq.reshape(M, d) if xq.is_contiguous() else xq.as_strided((M, d), (xq.stride(1), 1), xq.storage_offset())
    xk2 = xk.reshape(M, d) if xk.is_contiguous() else xk.as_strided((M, d), (xk.stride(1), 1), xk.storage_offset())
    q_hl = ops.split_tf32(xq2, cols=d, ld=xq2.stride(0), rows=M)
    k_hl = q_hl if xk is xq else ops.split_tf32(xk2, cols=d, ld=xk2.stride(0), rows=M)
    qkv = torch.empty((M, 3 * d), device=dev, dtype=torch.float32)
    for j, src in enumerate((q_hl, k_hl, q_hl)):   # query and value read the forward states, key the backward states
        ops.gemm_tf32x3(src[0], src[1], ent["w"][j][0], ent["w"][j][1], ent["b"][j], qkv[:, j * d:(j + 1) * d], M, d,
                        epilogue=1, ldc=3 * d)
    a = torch.empty((B, S, d), device=dev, dtype=torch.float32)
    lse = torch.empty((B, nheads, S), device=dev, dtype=torch.float32) if save else None
    band_attention(qkv, 3 * d, lens, 0, B, S, nheads, hd, reach, a, None, None, 0, lse, p_attn, seed)
    return a, (xq2, xk2, qkv, lse)


class BandMhaFn(torch.autograd.Function):
    """Differentiable w.r.t. both inputs and the three projections."""

    @staticmethod
    def forward(ctx, xq, xk, lens, packed, nheads, reach, p_attn, *params):
        need = any(ctx.needs_input_grad)
        seed = attn_seed(0) if p_attn > 0 else 0
        a, saved = _mha_forward(xq, xk, lens, packed, nheads, reach, save=need, p_attn=p_attn, seed=seed)
        if need:
            ctx.saved, ctx.lens, ctx.packed, ctx.nheads, ctx.reach = saved + (a,), lens, packed, nheads, reach
            ctx.p_attn, ctx.seed = p_attn, seed
            ctx.same = xk is xq
        return a

    @staticmethod
    def backward(ctx, dout):
        xq2, xk2, qkv, lse, a = ctx.saved
        lens, packed, nheads, reach = ctx.lens, ctx.packed, ctx.nheads, ctx.reach
        B, S, d = a.shape
        M = B * S
        hd = d // nheads
        dev = dout.device
        ent = packed.transposed()
        da = dout.contiguous()
        dqkv = torch.empty((M, 3 * d), device=dev, dtype=torch.float32)
        delta = torch.empty((B, nheads, S), device=dev, dtype=torch.float32)
        _call("mts_band_attn_bwd_dropout", _ptr(qkv), 3 * d, _ptr(a), _ptr(da), _ptr(lse), _ptr(lens.dev), 0, B, S, nheads, hd, reach,
              _ptr(dqkv), _ptr(delta), float(ctx.p_attn), int(ctx.seed), _stream())
        grads = []
        for j, x in enumerate((xq2, xk2, xq2)):
            dw, db = _dense_param_grads(dqkv[:, j * d:(j + 1) * d], x, M, d, d)
            grads += [dw, db]
        dxq = torch.empty((B, S, d), device=dev, dtype=torch.float32)
        dxk = dxq if ctx.same else torch.empty((B, S, d), device=dev, dtype=torch.float32)
        for j, (dst, acc) in enumerate(((dxq, False), (dxk, ctx.same), (dxq, True))):
            hl = ops.split_tf32(dqkv[:, j * d:(j + 1) * d], cols=d, ld=3 * d, rows=M)
            ops.gemm_tf32x3(hl[0], hl[1], ent["wt"][j][0], ent["wt"][j][1], None, dst.view(M, d), M, d, accumulate=acc)
        ctx.saved = None
        return (dxq, None if ctx.same else dxk, None, None, None, None, None, *grads)


class Longformer_Local_Attention(nn.Module):
    """The `just_mha=True` form of models/RestrictedTransformerLayer.py:65-133: `self.model` is the FFN-less layer."""

    def __init__(self, d_model: int, nhead: int, n_layers: int = 1, dim_feedforward: int = 2048, window_size=(8, 4),
                 dropout: float = 0.1, dropout_attention: float = 0.1, layer_norm_eps: float = 1e-5, tagset_size: int = 2,
                 device=None, max_position_embedding: int = 4096, just_mha: bool = True) -> None:
        super().__init__()
        if not just_mha:
            raise NotImplementedError("the full encoder is transformer.Longformer_Local_Attention")
        if isinstance(window_size, (list, tuple)):   # RestrictedTransformerLayer.py:77-80
            assert all(x % 2 == 0 for x in window_size), "All window sizes must be divisible by 2!"
        else:
            assert window_size % 2 == 0, "Window size must be divisible by 2!"
            raise TypeError("'int' object is not subscriptable: the FFN-less layer indexes config.attention_window[layer_id]; "
                            "pass a list (RecurrentLongformer does)")
        if d_model % nhead != 0:
            raise ValueError(f"The hidden size ({d_model}) is not a multiple of the number of attention heads ({nhead})")
        self.d_model, self.nhead = d_model, nhead
        self.reach = window_size[0] // 2          # layer_id defaults to 0: attention_window[0] // 2
        self.attention_dropout = float(dropout_attention)
        self.model = _NoffnLayer(d_model)
        self.layer = True
        self._packed = None

    def packed(self):
        if self._packed is None:
            self._packed = _PackedMha(self.model.attention.self)
        return self._packed

    def forward(self, inputs, lengths, external_input=None):
        xq = ops._check(inputs, "inputs")
        xk = xq if external_input is None else ops._check(external_input, "external_input")
        if xq.dim() != 3 or xq.shape[2] != self.d_model or xk.shape != xq.shape:
            raise ValueError(f"expected [B, S, {self.d_model}] hidden states, got {tuple(xq.shape)} / {tuple(xk.shape)}")
        if xq.stride(2) != 1 or xk.stride(2) != 1 or xq.stride(0) != xq.shape[1] * xq.stride(1) or xk.stride(0) != xk.shape[1] * xk.stride(1):
            xq, xk = xq.contiguous(), (xq.contiguous() if xk is xq else xk.contiguous())
        p_attn = self.attention_dropout if self.training else 0.0
        lens = lengths if isinstance(lengths, ops.Lengths) else ops.Lengths(lengths, xq.device, xq.shape[1])
        packed = self.packed()
        params = packed.params()
        if not (torch.is_grad_enabled() and (any(p.requires_grad for p in params) or xq.requires_grad or xk.requires_grad)):
            return _mha_forward(xq, xk, lens, packed, self.nhead, self.reach, save=False, p_attn=p_attn,
                                seed=attn_seed(0) if p_attn > 0 else 0)[0]
        return BandMhaFn.apply(xq, xk, lens, packed, self.nhead, self.reach, p_attn, *params)


class RecurrentLongformerBlock(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, nheads=8, dropout_in=0.0, dropout_attention=0.0,
                 batch_first=True, window_size=127, separate_forward_backward=False, just_mha=True):
        super().__init__()
        self.lstm = RNN(embedding_dim, hidden_dim, 1, tagset_size, True, dropout_in, dropout_attention, batch_first=batch_first,
                        LSTM=True)
        transformer_in = hidden_dim if separate_forward_backward else hidden_dim * 2
        self.sep_fb = separate_forward_backward
        just_mha = True if separate_forward_backward else just_mha
        # The reference does not pass `dropout_attention` here (models/CRF.py:653-657), so its wrapper default (0.1) becomes
        # HF's attention_probs_dropout_prob while training: same here (mts_band_attn_fwd_dropout); evaluation is dropout-free.
        self.transformer = Longformer_Local_Attention(transformer_in, nheads, 1, transformer_in, window_size=window_size,
                                                      dropout=dropout_in, layer_norm_eps=1e-12,
                                                      tagset_size=tagset_size, device=None, max_position_embedding=4096,
                                                      just_mha=just_mha)

    def forward(self, inputs, lengths):
        lens = _lens(lengths, inputs)
        x = self.lstm(inputs, lens)                      # [B, S, 2H], zero beyond len_b (the reference re-pads to 3600 rows)
        if self.sep_fb:
            H = x.shape[2] // 2
            return self.transformer(x[:, :, :H], lens, external_input=x[:, :, H:])   # x.view(bs, sl, 2, -1)[:, :, 0 / 1, :]
        return self.transformer(x, lens)


class RecurrentLongformer(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=6, nheads=8, dropout_in=0.0, dropout_out=0.0,
                 batch_first=True, loss_fn="CrossEntropy", threshold=None, window_size=127, alpha=0.9, gamma=2,
                 separate_forward_backward=True, last_bilstm=True):
        super().__init__()
        if isinstance(window_size, int):
            window_size = [window_size]
        self.tagset_size = tagset_size
        kw = dict(nheads=nheads, dropout_in=dropout_in, dropout_attention=dropout_out, batch_first=batch_first,
                  window_size=window_size, separate_forward_backward=separate_forward_backward, just_mha=True)
        self.model = nn.ModuleList([RecurrentLongformerBlock(tagset_size, embedding_dim, hidden_dim, **kw)])
        block_out = hidden_dim if separate_forward_backward else hidden_dim * 2
        # the reference builds every later block with embedding_dim = hidden_dim (CRF.py:782), which only matches the
        # previous block's output width when separate_forward_backward is set (its default)
        self.model.extend([RecurrentLongformerBlock(tagset_size, hidden_dim, hidden_dim, **kw) for _ in range(num_layers - 1)])
        if last_bilstm:
            self.model.append(RNN(hidden_dim, hidden_dim, 1, tagset_size, True, dropout_in, dropout_out, batch_first=batch_first,
                                  LSTM=True))
        out_dim = hidden_dim * 2 if last_bilstm else block_out
        _build_head(self, out_dim, tagset_size, loss_fn, threshold, alpha, gamma)

    def _features(self, x, lens):
        """x: [B, S, embedding_dim] or an early-fusion pair (text, audio); only the first block's RNN reads the pair (in its input
        projection), later blocks get the previous block's output."""
        for block in self.model:
            x = block(x, lens)
        return x

    def loss(self, x, lengths, tags, segments=None, global_count=None):
        if segments is not None:
            raise NotImplementedError("the auxiliary cosine loss (segments=...) is outside the B200 hot path")
        lens = _lens(lengths, x)
        return _head_loss(self, self._features(x, lens), lens, tags, global_count)

    def forward(self, x, lenghts, threshold=0.4):
        lens = _lens(lenghts, x)
        with torch.no_grad():
            return _head_decode(self, self._features(x, lens), lens, threshold)

    def decode_device(self, x, lenghts, threshold=0.4):
        lens = _lens(lenghts, x)
        with torch.no_grad():
            return (*_head_decode_device(self, self._features(x, lens), lens, threshold), lens)
