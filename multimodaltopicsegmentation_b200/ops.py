"""Python face of the C ABI: thin wrappers that hand raw device pointers of torch tensors to
libmts_b200.so, plus the autograd.Function glue for training.  PyTorch is used here for device memory,
streams and autograd bookkeeping only -- every arithmetic step of the hot path is one of our kernels.

A global launch counter (`launch_count()`) records how many of OUR kernels were launched; bench.py reports it.
"""
from __future__ import annotations

import torch

from . import _lib

_LAUNCHES = 0
# kernels launched per ABI call (for the bench's gpu_launches claim)
_KERNELS_PER_CALL = {
    "mts_seg_loss_fwd": 2, "mts_head_bwd": 3, "mts_colsum": 2, "mts_ln_bwd": 3, "mts_band_attn_bwd": 2,
}


def launch_count():
    return _LAUNCHES


def reset_launch_count():
    global _LAUNCHES
    _LAUNCHES = 0


PROFILE = None  # bench.py sets this to a dict to collect CUDA-event timings per ABI entry point
# debugging aid for tests only: MTS_GEMM_IMPL=simt routes the input projections through mts_gemm_f32
GEMM_IMPL = __import__("os").environ.get("MTS_GEMM_IMPL", "tcgen05")
# recurrence for H == 256: "tc" = tcgen05 tensor-core kernel (default), "fma" = exact-fp32 packed-FMA cluster kernel
REC_IMPL = __import__("os").environ.get("MTS_REC_IMPL", "tc")


# Arithmetic of the LSTM path: "f32" (default; the parity contract: error-compensated TF32 + bf16 products, fp32-grade) or
# "bf16" (explicit switch, inference only: bf16 x bf16 products in the input projections and the recurrence, fp32 state and
# accumulation; tolerances per kernel in DESIGN.md).  MTS_PRECISION=bf16 or set_precision("bf16").
PRECISION = __import__("os").environ.get("MTS_PRECISION", "f32")


def set_precision(name):
    global PRECISION
    if name not in ("f32", "bf16"):
        raise ValueError("precision must be 'f32' or 'bf16'")
    PRECISION = name


def _call(name, *args):
    global _LAUNCHES
    _LAUNCHES += _KERNELS_PER_CALL.get(name, 1)
    if PROFILE is None:
        return _lib.call(name, *args)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    rc = _lib.call(name, *args)
    end.record()
    PROFILE.setdefault(name, []).append((start, end))
    return rc


def _stream():
    """Raw handle of torch's current CUDA stream on the current device (every launch takes it as its last argument).
    torch.cuda.current_stream() builds a Python Stream object per call (~15 us, 60+ calls per training step: a fifth of the
    host time of a configs[3] step); the raw query is a plain C call."""
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _check(t, name, dtype=torch.float32):
    if not t.is_cuda:
        raise _lib.MtsError(f"{name} must live on a CUDA device: this package has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # the C ABI launches on the CUDA runtime's current device and on torch's current stream of that device
        raise _lib.MtsError(f"{name} lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}: "
                            "wrap the call in torch.cuda.device(tensor.device)")
    return t


def _pad32(k):
    return (k + 31) // 32 * 32


def device_ok():
    return _lib.call("mts_device_ok")


# --------------------------------------------------------------------------------------------------------
# lengths: the reference consumes them on the host (lengths.data.tolist()); we keep a host list, a device
# int32 copy and the length-sorted episode order used to build the tiles of the recurrence kernels.
# --------------------------------------------------------------------------------------------------------
class Lengths:
    def __init__(self, lengths, device, T_in):
        if torch.is_tensor(lengths):
            host = [int(v) for v in lengths.detach().cpu().tolist()]
        else:
            host = [int(v) for v in lengths]
        if not host or min(host) < 1:
            raise ValueError("every episode must hold at least one sentence")
        if max(host) > T_in:
            raise ValueError(f"length {max(host)} exceeds the padded time axis {T_in}")
        self.host = host
        self.B = len(host)
        self.T = max(host)  # pad_packed_sequence crops the time axis to max(lengths) (SURVEY fact 10)
        self.N = sum(host)
        order = sorted(range(self.B), key=lambda i: -host[i])
        offs, run = [], 0
        for n in host:  # exclusive prefix sums: first row of every episode in the ragged token layout
            offs.append(run)
            run += n
        both = torch.tensor([host, order, offs], dtype=torch.int32)
        both = both.pin_memory() if torch.cuda.is_available() else both
        dev = both.to(device, non_blocking=True)
        self.dev = dev[0]
        self.order = dev[1]
        self.offs = dev[2]


# --------------------------------------------------------------------------------------------------------
# GEMMs
# --------------------------------------------------------------------------------------------------------
A_SIDE, B_SIDE = 0, 1  # which GEMM operand a split matrix will be (the correction halves are ordered per side)


def split_tf32(src2d, cols=None, ld=None, rows=None, side=A_SIDE):
    """src [rows, cols] (row stride ld) -> (hi, lo) [rows, pad32(cols)]: hi = the fp32 values (zero padded), lo = the
    packed bf16 correction operand of the same byte size (include/mts_b200.h, "Operand preparation")."""
    rows = src2d.shape[0] if rows is None else rows
    cols = src2d.shape[1] if cols is None else cols
    ld = src2d.stride(0) if ld is None else ld
    kp = _pad32(cols)
    out = torch.empty((2, rows, kp), device=src2d.device, dtype=torch.float32)
    _call("mts_split_tf32", _ptr(src2d), ld, rows, cols, kp, side, _ptr(out[0]), _ptr(out[1]), _stream())
    return out[0], out[1]


def _rows_ok(x, name, B, T):
    """The packing kernel reads src + b * bstride + t * D + k: rows of one episode must be dense (stride(1) == D,
    stride(2) == 1).  A view that is not (e.g. x[:, :, :D1] of a fused tensor) is made contiguous here."""
    if x is None:
        return None
    _check(x, name, torch.bfloat16 if x.dtype == torch.bfloat16 else torch.float32)
    if x.dtype == torch.bfloat16 and PRECISION != "bf16":
        raise TypeError(f"{name}: bfloat16 embeddings belong to the bf16 path (ops.set_precision('bf16')); the fp32 path takes fp32")
    if x.dim() != 3 or x.shape[0] < B or x.shape[1] < T:
        raise ValueError(f"{name}: expected [B >= {B}, T >= {T}, D], got {tuple(x.shape)}")
    if x.stride(2) != 1 or x.stride(1) != x.shape[2]:
        x = x.contiguous()
    return x


def _packs_by_8(x1, x2):
    """The packed-operand-only kernels move 8 elements per 16-byte access: every width a multiple of 8, every batch stride
    and source pointer on 16 bytes."""
    return all(x.shape[2] % 8 == 0 and x.stride(0) * x.element_size() % 16 == 0 and x.data_ptr() % 16 == 0
               for x in (x1, x2) if x is not None)


def pack_rows_packed(x1, x2, B, T):
    """bf16 path: [x1[b,:T] | x2[b,:T]] -> the packed operand alone [B*T, pad32(D1+D2)].  The sources may be fp32 or -- embeddings
    stored and shipped as bf16 -- bfloat16 tensors, of any width: sources the 8-wide kernels cannot take are packed by the
    element-wise kernel, bf16 ones widened to fp32 first (exact)."""
    if x2 is not None and x2.dtype != x1.dtype:
        raise TypeError("both modalities must have the same dtype")
    D1 = x1.shape[2]
    D2 = 0 if x2 is None else x2.shape[2]
    kp = _pad32(D1 + D2)
    lo = torch.empty((B * T, kp), device=x1.device, dtype=torch.float32)
    by8 = _packs_by_8(x1, x2)
    if x1.dtype == torch.bfloat16:
        if by8:
            _call("mts_pack_rows_bf16in", _ptr(x1), x1.stride(0), D1, _ptr(x2), 0 if x2 is None else x2.stride(0), D2, B, T, kp,
                  _ptr(lo), _stream())
            return lo
        x1, x2 = x1[:B, :T].float(), (None if x2 is None else x2[:B, :T].float())
        by8 = _packs_by_8(x1, x2)
    # the element-wise kernel writes the fp32 operand too: a scratch `hi`, dropped
    hi = None if by8 else torch.empty_like(lo)
    _call("mts_pack_rows_split", _ptr(x1), x1.stride(0), D1, _ptr(x2), 0 if x2 is None else x2.stride(0), D2, B, T, kp,
          _ptr(hi), _ptr(lo), _stream())
    return lo


def pack_rows_split(x1, x2, B, T):
    """[x1[b,:T] | x2[b,:T]] -> (hi, lo) [B*T, pad32(D1+D2)] (early fusion concat + crop + split, one kernel)"""
    x1, x2 = _rows_ok(x1, "input", B, T), _rows_ok(x2, "second input", B, T)
    D1 = x1.shape[2]
    D2 = 0 if x2 is None else x2.shape[2]
    kp = _pad32(D1 + D2)
    out = torch.empty((2, B * T, kp), device=x1.device, dtype=torch.float32)
    _call("mts_pack_rows_split", _ptr(x1), x1.stride(0), D1, _ptr(x2), 0 if x2 is None else x2.stride(0), D2, B, T, kp,
          _ptr(out[0]), _ptr(out[1]), _stream())
    return out[0], out[1]


# The layer-0 input projection reads the embeddings in place (two TMA maps split along K) and only the packed correction
# operand is written beforehand; MTS_PROJ_DIRECT=0 restores the concat + operand-pair packing pass.
PROJ_DIRECT = __import__("os").environ.get("MTS_PROJ_DIRECT", "1") != "0"


def _direct_sources_ok(x1, x2, B, T):
    """In-place reading needs [B*T, D_i] to be plain matrices: no time crop, dense rows, 16-byte row pitch, and -- when a second
    source follows -- a first width that is a whole number of 32-wide k-blocks."""
    for x in (x1, x2):
        if x is None:
            continue
        if x.dtype != torch.float32 or x.shape[0] != B or x.shape[1] != T or not x.is_contiguous() or x.shape[2] % 8 != 0:
            return False    # (the packed-operand-only packing kernel works on 8-element units)
        if x.data_ptr() % 16 != 0:
            return False
    return x2 is None or x1.shape[2] % 32 == 0


# The same projection over fp16-split operands (mts_pack_rows_f16 -> mts_gemm_f16x3: 6 instead of 8 MMAs per 32 k, 1.27x at
# cfg1's 19 200 x 2048 x 896); MTS_PROJ_F16X3=0 keeps the TF32 + bf16 product.
PROJ_F16X3 = __import__("os").environ.get("MTS_PROJ_F16X3", "1") != "0"


def _f16_projection_ok(x1, x2, B, T, N):
    D = x1.shape[2] + (0 if x2 is None else x2.shape[2])
    for x in (x1, x2):
        if x is not None and (x.dtype != torch.float32 or x.shape[2] % 4 != 0 or x.stride(0) % 4 != 0 or x.data_ptr() % 16 != 0):
            return False
    return PROJ_F16X3 and PRECISION != "bf16" and B * T >= 256 and N >= 256 and D <= 2048


def input_projection(x1, x2, B, T, w_hi, w_lo, bias, out, N, w_pieces=None):
    """out [B*T, N] = [x1 | x2] W^T + bias: early-fusion concat + linear projection (load_datasets_precomputed.py:158-161 +
    NeuralArchitectures.py:113).  w_pieces: callable returning the fp16-split weights (pieces, scale); with it and a large
    enough product the operand is packed as fp16 pieces and the product runs in the GEMM's fp16-split mode; otherwise the
    embeddings are read in place by the TF32 + bf16 GEMM's TMA producer."""
    x1, x2 = _rows_ok(x1, "input", B, T), _rows_ok(x2, "second input", B, T)
    if w_pieces is not None and _f16_projection_ok(x1, x2, B, T, N):
        D1 = x1.shape[2]
        D2 = 0 if x2 is None else x2.shape[2]
        k64 = (D1 + D2 + 63) // 64 * 64
        pieces = torch.empty((B * T, 2, k64), device=x1.device, dtype=torch.float16)
        scale = torch.empty((B * T,), device=x1.device, dtype=torch.float32)
        _call("mts_pack_rows_f16", _ptr(x1), x1.stride(0), D1, _ptr(x2), 0 if x2 is None else x2.stride(0), D2, B, T, k64,
              _ptr(pieces), _ptr(scale), _stream())
        wp, ws = w_pieces()
        return gemm_f16x3(pieces, scale, wp, ws, bias, out, B * T, N, epilogue=1)
    if not (PROJ_DIRECT and _direct_sources_ok(x1, x2, B, T)):
        a_hi, a_lo = pack_rows_split(x1, x2, B, T)
        return gemm_tf32x3(a_hi, a_lo, w_hi, w_lo, bias, out, B * T, N, epilogue=1, ldc=N)
    D1 = x1.shape[2]
    D2 = 0 if x2 is None else x2.shape[2]
    a_lo = pack_rows_packed(x1, x2, B, T)     # the packed correction operand alone (hi == NULL)
    _call("mts_gemm_tf32x3_srcs", _ptr(x1), D1, D1, _ptr(x2), D2, D2, _ptr(a_lo), _ptr(w_hi), _ptr(w_lo), _ptr(bias), _ptr(out),
          B * T, N, a_lo.shape[1], N, 1, 0, _stream())
    return out


def f16_pieces(w):
    """fp32 matrix [N, K] -> (pieces [N, 2, K64] fp16, scale [N]): the fp16-split operand of mts_gemm_f16x3.  Row n is scaled by the
    exact power of two 2^s that puts its largest magnitude into [2^13, 2^14); pieces = fp16(w 2^s), fp16(w 2^s - piece 1);
    scale = 2^-s.  (Weight packing: once per parameter version, plain torch ops.)"""
    N, K = w.shape
    K64 = (K + 63) // 64 * 64
    amax = w.abs().amax(dim=1)
    _, e = torch.frexp(amax)                     # amax = m 2^e, m in [0.5, 1)
    sexp = torch.where(amax > 0, 14 - e, torch.zeros_like(e)).clamp(-110, 110)
    scale = torch.ldexp(torch.ones_like(amax), sexp)
    ws = w * scale[:, None]
    pieces = torch.zeros((N, 2, K64), device=w.device, dtype=torch.float16)
    w1 = ws.half()
    pieces[:, 0, :K] = w1
    pieces[:, 1, :K] = (ws - w1.float()).half()
    return pieces.contiguous(), (1.0 / scale).contiguous()


def f16_pieces_stacked(mats):
    """f16_pieces of the row-wise concatenation of `mats` ([N_i, K] fp32 each) without forming it: one mts_pack_rows_f16
    launch per matrix (warp per row: maximum, power-of-two scale, two pieces) into slices of the outputs.  In training the
    weights change every step, so this runs once per step and LSTM layer: the torch formulation above costs ~15 small
    launches each time.  Falls back to it for matrices the kernel does not take (width not a multiple of 4, unaligned)."""
    K = mats[0].shape[1]
    ok = all(m.is_cuda and m.dtype == torch.float32 and m.dim() == 2 and m.shape[1] == K and m.is_contiguous()
             and m.data_ptr() % 16 == 0 for m in mats) and K % 4 == 0 and K <= 2048
    if not ok:
        return f16_pieces(torch.cat([m.detach() for m in mats], dim=0))
    K64 = (K + 63) // 64 * 64
    N = sum(m.shape[0] for m in mats)
    pieces = torch.empty((N, 2, K64), device=mats[0].device, dtype=torch.float16)
    scale = torch.empty((N,), device=mats[0].device, dtype=torch.float32)
    row = 0
    for m in mats:
        n = m.shape[0]
        _call("mts_pack_rows_f16", _ptr(m), n * K, K, 0, 0, 0, 1, n, K64, pieces.data_ptr() + row * 2 * K64 * 2,
              scale.data_ptr() + row * 4, _stream())
        row += n
    return pieces, scale


def gemm_f16x3(a_pieces, a_scale, b_pieces, b_scale, bias, out, M, N, epilogue=0, out_lo=None):
    """out [M, N] = A B^T (+ bias; epilogue 2: GELU) over fp16-split operands (include/mts_b200.h, mts_gemm_f16x3)."""
    K64 = a_pieces.shape[-1]
    assert b_pieces.shape[-1] == K64
    _call("mts_gemm_f16x3", _ptr(a_pieces), _ptr(b_pieces), _ptr(a_scale), _ptr(b_scale), _ptr(bias), _ptr(out), _ptr(out_lo), M, N,
          K64, out.stride(-2), epilogue if bias is not None else 0, _stream())
    return out


def transpose_split(src_ptr, bstride, ld, rows, cols, T, device, shift=0, lengths=None, side=A_SIDE):
    """(hi, lo) [cols, pad32(rows)] of the transposed (optionally time-shifted / length-masked) source: the K-major
    operand of a GEMM that contracts over tokens (weight gradients)."""
    kp = _pad32(rows)
    out = torch.empty((2, cols, kp), device=device, dtype=torch.float32)
    _call("mts_transpose_split", src_ptr, bstride, ld, rows, cols, T, shift, _ptr(lengths), kp, side, _ptr(out[0]),
          _ptr(out[1]), _stream())
    return out[0], out[1]


def weight_grad(dyT, x_ptr, x_bstride, x_ld, rows, n_in, T, out, ldc, device, shift=0, lengths=None):
    """out[n_out, n_in] (row stride ldc) = dY^T X over `rows` tokens on the tensor cores.  dyT = (hi, lo) of dY^T
    [n_out, pad32(rows)] from transpose_split; X is transposed / split here."""
    xT = transpose_split(x_ptr, x_bstride, x_ld, rows, n_in, T, device, shift=shift, lengths=lengths, side=B_SIDE)
    gemm_tf32x3(dyT[0], dyT[1], xT[0], xT[1], None, out, dyT[0].shape[0], n_in, ldc=ldc)


def gemm_tf32x3(a_hi, a_lo, b_hi, b_lo, bias, out, M, N, epilogue=0, accumulate=False, ldc=None):
    kp = a_hi.shape[1]
    assert b_hi.shape[1] == kp
    _call("mts_gemm_tf32x3", _ptr(a_hi), _ptr(a_lo), _ptr(b_hi), _ptr(b_lo), _ptr(bias), _ptr(out), M, N, kp,
          out.stride(-2) if ldc is None else ldc, epilogue if bias is not None else 0, int(accumulate), _stream())
    return out


def gemm_f32(a_ptr, lda, b_ptr, ldb, bias, c_ptr, ldc, M, N, K, layout, epilogue=0, accumulate=False, splits=1,
             shift=0, T=0, lengths=None):
    _call("mts_gemm_f32", a_ptr, lda, b_ptr, ldb, _ptr(bias), c_ptr, ldc, M, N, K, layout,
          epilogue if bias is not None else 0, int(accumulate), splits, shift, T, _ptr(lengths), _stream())


def colsum(x_ptr, ld, M, N, out, accumulate=False):
    ws = torch.empty(_lib.load().mts_colsum_ws_bytes(M, N) // 4, device=out.device, dtype=torch.float32)
    _call("mts_colsum", x_ptr, ld, M, N, _ptr(out), int(accumulate), _ptr(ws), _stream())


class LinearFn(torch.autograd.Function):
    """y = x W^T + b on the exact-fp32 GEMM (small output widths: CRF emissions)."""

    @staticmethod
    def forward(ctx, x, w, b):
        _check(x, "x"); _check(w, "weight")
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        M, K = x2.shape
        N = w.shape[0]
        wc = w.contiguous()
        y = torch.empty((M, N), device=x.device, dtype=torch.float32)
        gemm_f32(_ptr(x2), K, _ptr(wc), K, b.contiguous(), _ptr(y), N, M, N, K, layout=0, epilogue=1)
        ctx.save_for_backward(x2, wc)
        ctx.xshape = x.shape
        return y.reshape(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        x2, w = ctx.saved_tensors
        M, K = x2.shape
        N = w.shape[0]
        dy2 = dy.reshape(M, N).contiguous()
        dx = torch.empty_like(x2)
        gemm_f32(_ptr(dy2), N, _ptr(w), K, None, _ptr(dx), K, M, K, N, layout=2)
        dw = torch.empty_like(w)
        gemm_f32(_ptr(dy2), N, _ptr(x2), K, None, _ptr(dw), K, N, K, M, layout=3, splits=8 if M > 4096 else 1)
        db = torch.empty(N, device=w.device, dtype=torch.float32)
        colsum(_ptr(dy2), N, M, N, db)
        return dx.reshape(ctx.xshape), dw, db


# --------------------------------------------------------------------------------------------------------
# LSTM stack
# --------------------------------------------------------------------------------------------------------
class PackedLstm:
    """GEMM-ready shadow copies of one or two nn.LSTM parameter sets (state-dict layout untouched):
    per layer  w_ih (hi, lo) [n_enc][8H, pad32(D_l)], bias [n_enc][8H] = b_ih + b_hh, w_hh [n_enc, 2, 4H, H]."""

    def __init__(self, rnns):
        self.rnns = rnns
        self.key = None
        self.layers = None

    _NAMES = {}

    def _params(self, rnn, layer):
        # straight out of the module's parameter dict: nn.Module.__getattr__ (the fallback path every `rnn.weight_*` takes)
        # made this lookup a tenth of the host time of a training step
        names = self._NAMES.get(layer)
        if names is None:
            sfx = f"_l{layer}"
            names = self._NAMES[layer] = ("weight_ih" + sfx, "weight_hh" + sfx, "bias_ih" + sfx, "bias_hh" + sfx,
                                          "weight_ih" + sfx + "_reverse", "weight_hh" + sfx + "_reverse",
                                          "bias_ih" + sfx + "_reverse", "bias_hh" + sfx + "_reverse")
        prm = rnn._parameters
        return [prm[n] for n in names]

    def flat_params(self):
        out = []
        for rnn in self.rnns:
            for layer in range(rnn.num_layers):
                out.extend(self._params(rnn, layer))
        return out

    def wih_pieces(self, layer, e):
        """fp16-split copy of W_ih of (layer, encoder e), both directions stacked: (pieces [8H, 2, K64], scale [8H]) for
        mts_gemm_f16x3.  Made on first use per weight version."""
        ent = self.get()[layer]
        cache = ent.setdefault("wih_p", {})
        if e not in cache:
            w_f, _, _, _, w_r = self._params(self.rnns[e], layer)[:5]
            with torch.no_grad():
                cache[e] = f16_pieces_stacked([w_f.detach(), w_r.detach()])
        return cache[e]

    def wih_packed_a(self, layer, e):
        """bf16 path: W_ih of (layer, encoder e), both directions stacked, packed like an A operand (side 0) so that the
        packed halves of activations and weights pair up x * w.  Made on first use per weight version."""
        ent = self.get()[layer]
        cache = ent.setdefault("wih_bf", {})
        if e not in cache:
            w_f, _, _, _, w_r = self._params(self.rnns[e], layer)[:5]
            D = w_f.shape[1]
            kp = _pad32(D)
            H4 = w_f.shape[0]
            bf = torch.empty((2, 2 * H4, kp), device=w_f.device, dtype=torch.float32)
            with torch.no_grad():
                for d, w in enumerate((w_f, w_r)):
                    wc = w.detach().contiguous()
                    _call("mts_split_tf32", _ptr(wc), D, H4, D, kp, A_SIDE, _ptr(bf[0, d * H4:]), _ptr(bf[1, d * H4:]), _stream())
            cache[e] = bf[1]
        return cache[e]

    def get(self):
        key = tuple((p.data_ptr(), p._version) for p in self.flat_params())
        if key == self.key:
            return self.layers
        rnn0 = self.rnns[0]
        H, L = rnn0.hidden_size, rnn0.num_layers
        dev = rnn0.weight_hh_l0.device
        layers = []
        with torch.no_grad():
            for layer in range(L):
                wih, bias = [], []
                whh = torch.empty((len(self.rnns), 2, 4 * H, H), device=dev, dtype=torch.float32)
                for e, rnn in enumerate(self.rnns):
                    w_f, h_f, bi_f, bh_f, w_r, h_r, bi_r, bh_r = self._params(rnn, layer)
                    D = w_f.shape[1]
                    kp = _pad32(D)
                    pair = torch.empty((2, 8 * H, kp), device=dev, dtype=torch.float32)
                    for d, w in enumerate((w_f, w_r)):
                        wc = w.detach().contiguous()
                        _call("mts_split_tf32", _ptr(wc), D, 4 * H, D, kp, B_SIDE, _ptr(pair[0, d * 4 * H:]),
                              _ptr(pair[1, d * 4 * H:]), _stream())
                    wih.append((pair[0], pair[1]))
                    bias.append(torch.cat([bi_f.detach() + bh_f.detach(), bi_r.detach() + bh_r.detach()]))
                    whh[e, 0].copy_(h_f.detach())
                    whh[e, 1].copy_(h_r.detach())
                layers.append({"wih": wih, "bias": bias, "whh": whh})
        self.key, self.layers = key, layers
        return layers


def _lstm_stack_forward(x1, x2, xs2, lens, packed, H, L, n_enc, save):
    """Runs all layers.  Early fusion: encoders=1, inputs (x1 | x2).  Late fusion: n_enc=2, encoder 0 reads x1,
    encoder 1 reads xs2.  Returns (y_last [B,T,n_enc*2H], saved list per layer)."""
    B, T = lens.B, lens.T
    dev = x1.device
    layers = packed.get()
    saved = []
    y_prev = y_corr = None
    bf16 = PRECISION == "bf16"
    if bf16 and (save or H != 256 or REC_IMPL != "tc" or GEMM_IMPL == "simt"):
        raise NotImplementedError("the bf16 path serves inference with H == 256 on the tensor-core kernels; train in fp32")
    for layer in range(L):
        gx = torch.empty((n_enc, B * T, 8 * H), device=dev, dtype=torch.float32)
        for e in range(n_enc):
            if bf16:
                if layer == 0:
                    a_lo = pack_rows_packed(x1, x2, B, T) if n_enc == 1 else pack_rows_packed(x1 if e == 0 else xs2, None, B, T)
                elif y_corr is not None:
                    a_lo = y_corr
                else:
                    src = y_prev.view(B * T, n_enc * 2 * H)[:, e * 2 * H:(e + 1) * 2 * H]
                    a_lo = split_tf32(src, cols=2 * H, ld=n_enc * 2 * H, rows=B * T)[1]
                _call("mts_gemm_bf16p", _ptr(a_lo), _ptr(packed.wih_packed_a(layer, e)), _ptr(layers[layer]["bias"][e]), _ptr(gx[e]),
                      B * T, 8 * H, a_lo.shape[1], 8 * H, 1, 0, _stream())
                continue
            if layer == 0 and GEMM_IMPL != "simt":
                w_hi, w_lo = layers[layer]["wih"][e]
                wp = lambda e=e: packed.wih_pieces(0, e)
                if n_enc == 1:
                    input_projection(x1, x2, B, T, w_hi, w_lo, layers[layer]["bias"][e], gx[e], 8 * H, w_pieces=wp)
                else:
                    input_projection(x1 if e == 0 else xs2, None, B, T, w_hi, w_lo, layers[layer]["bias"][e], gx[e], 8 * H,
                                     w_pieces=wp)
                continue
            if layer == 0:
                if n_enc == 1:
                    a_hi, a_lo = pack_rows_split(x1, x2, B, T)
                else:
                    a_hi, a_lo = pack_rows_split(x1 if e == 0 else xs2, None, B, T)
            elif y_corr is not None:  # the recurrence wrote the correction operand of y; y itself is the fp32 operand
                a_hi, a_lo = y_prev.view(B * T, 2 * H), y_corr
            else:
                src = y_prev.view(B * T, n_enc * 2 * H)[:, e * 2 * H:(e + 1) * 2 * H]
                a_hi, a_lo = split_tf32(src, cols=2 * H, ld=n_enc * 2 * H, rows=B * T)
            w_hi, w_lo = layers[layer]["wih"][e]
            if GEMM_IMPL == "simt":
                a, w = a_hi, w_hi  # the hi arrays are the fp32 values themselves
                gemm_f32(_ptr(a), a.shape[1], _ptr(w), w.shape[1], layers[layer]["bias"][e], _ptr(gx[e]), 8 * H, B * T,
                         8 * H, a.shape[1], layout=0, epilogue=1)
            else:
                gemm_tf32x3(a_hi, a_lo, w_hi, w_lo, layers[layer]["bias"][e], gx[e], B * T, 8 * H, epilogue=1,
                            ldc=8 * H)
        y = torch.empty((B, T, n_enc * 2 * H), device=dev, dtype=torch.float32)
        gates = torch.empty((n_enc, 2, B, T, 5, H), device=dev, dtype=torch.float32) if save else None
        if H == 256 and REC_IMPL == "tc":
            # early fusion, more layers above: the kernel also writes the GEMM operand of the next layer's input
            y_corr = (torch.empty((B * T, 2 * H), device=dev, dtype=torch.float32)
                      if (n_enc == 1 and layer + 1 < L and GEMM_IMPL != "simt") else None)
            _call("mts_lstm_rec_fwd_tc_bf16" if bf16 else "mts_lstm_rec_fwd_tc", _ptr(gx), _ptr(layers[layer]["whh"]),
                  _ptr(lens.dev), _ptr(lens.order), n_enc, B, T, H, _ptr(y), _ptr(gates), _ptr(y_corr), _stream())
        else:
            y_corr = None
            _call("mts_lstm_rec_fwd", _ptr(gx), _ptr(layers[layer]["whh"]), _ptr(lens.dev), _ptr(lens.order), n_enc, B, T,
                  H, _ptr(y), _ptr(gates), _stream())
        saved.append((y_prev, y, gates))
        y_prev = y
    return y_prev, saved


def bilstm_stack(x1, x2, xs2, lens, packed, n_enc):
    """The bi-LSTM stack as the modules call it.  Inference (grad mode off, or nothing to differentiate) skips autograd
    and, with it, the per-step gate record the backward pass needs (5 H floats per sentence and direction)."""
    # dense rows for the forward packing kernel AND the backward weight-gradient transposes (both index by strides)
    x1, x2, xs2 = (_rows_ok(x1, "input", lens.B, lens.T), _rows_ok(x2, "second input", lens.B, lens.T),
                   _rows_ok(xs2, "second encoder input", lens.B, lens.T))
    flat = packed.flat_params()
    if not (torch.is_grad_enabled() and (any(p.requires_grad for p in flat) or x1.requires_grad)):
        rnn0 = packed.rnns[0]
        return _lstm_stack_forward(x1, x2, xs2, lens, packed, rnn0.hidden_size, rnn0.num_layers, n_enc, save=False)[0]
    return BiLstmStackFn.apply(x1, x2, xs2, lens, packed, n_enc, *flat)


class BiLstmStackFn(torch.autograd.Function):
    """Differentiable (w.r.t. the LSTM parameters) bi-LSTM stack.  Embedding inputs are data, so layer-0 dX is skipped
    (SURVEY.md section 8a') -- unless the single input of an early-fusion stack itself requires a gradient (the stacked
    blocks of RecurrentLongformer feed one block's attention output into the next block's LSTM)."""

    @staticmethod
    def forward(ctx, x1, x2, xs2, lens, packed, n_enc, *flat):
        rnn0 = packed.rnns[0]
        H, L = rnn0.hidden_size, rnn0.num_layers
        need = any(ctx.needs_input_grad)  # true even under no_grad: callers go through bilstm_stack()
        y, saved = _lstm_stack_forward(x1, x2, xs2, lens, packed, H, L, n_enc, save=need)
        if need:
            ctx.x1, ctx.x2, ctx.xs2, ctx.lens, ctx.packed, ctx.n_enc = x1, x2, xs2, lens, packed, n_enc
            ctx.saved = saved
            ctx.HL = (H, L)
        return y

    @staticmethod
    def backward(ctx, dy):
        H, L = ctx.HL
        lens, packed, n_enc = ctx.lens, ctx.packed, ctx.n_enc
        B, T = lens.B, lens.T
        N = B * T
        layers = packed.get()
        dev = dy.device
        dy = dy.contiguous()
        grads = [[None] * (8 * L) for _ in range(n_enc)]
        dx_in = None
        splits = max(1, min(16, N // 2048))
        tensor_core = GEMM_IMPL != "simt"
        ycols = n_enc * 2 * H
        for layer in range(L - 1, -1, -1):
            y_in, y_out, gates = ctx.saved[layer]
            dgx = torch.empty((n_enc, N, 8 * H), device=dev, dtype=torch.float32)
            if H == 256 and REC_IMPL == "tc":
                _call("mts_lstm_rec_bwd_tc", _ptr(dy), _ptr(gates), _ptr(layers[layer]["whh"]), _ptr(lens.dev),
                      _ptr(lens.order), n_enc, B, T, H, _ptr(dgx), _stream())
            else:
                if "whh_t" not in layers[layer]:  # transposed copy, made once per weight version, only when training
                    layers[layer]["whh_t"] = layers[layer]["whh"].transpose(2, 3).contiguous()
                _call("mts_lstm_rec_bwd", _ptr(dy), _ptr(gates), _ptr(layers[layer]["whh"]), _ptr(layers[layer]["whh_t"]),
                      _ptr(lens.dev), _ptr(lens.order), n_enc, B, T, H, _ptr(dgx), _stream())
            dy_next = torch.empty((B, T, n_enc * 2 * H), device=dev, dtype=torch.float32) if layer > 0 else None
            for e in range(n_enc):
                rnn = packed.rnns[e]
                w_f, h_f, bi_f, bh_f, w_r, h_r, bi_r, bh_r = packed._params(rnn, layer)
                D = w_f.shape[1]
                dg = dgx[e]
                # biases: column sums of dgx (b_ih and b_hh receive identical gradients)
                db = torch.empty(8 * H, device=dev, dtype=torch.float32)
                colsum(_ptr(dg), 8 * H, N, 8 * H, db)
                dwih = torch.empty((8 * H, D), device=dev, dtype=torch.float32)
                dwhh = torch.empty((2, 4 * H, H), device=dev, dtype=torch.float32)
                yo = y_out.view(N, ycols)
                if layer == 0:
                    if n_enc == 1:  # early fusion: the two modality blocks of W_ih get their own GEMM (no concat copy)
                        srcs = [(ctx.x1, 0)] + ([(ctx.x2, ctx.x1.shape[2])] if ctx.x2 is not None else [])
                    else:
                        srcs = [(ctx.x1 if e == 0 else ctx.xs2, 0)]
                if tensor_core:
                    # weight gradients contract over tokens: both operands transposed to K-major (hi, lo) halves, then
                    # the tcgen05 3xTF32 GEMM.  dgx^T is shared by dW_ih and both dW_hh.
                    dgT = transpose_split(_ptr(dg), 0, 8 * H, N, 8 * H, N, dev)
                    if layer == 0:
                        for x, off in srcs:
                            weight_grad(dgT, _ptr(x), x.stride(0), x.stride(1), N, x.shape[2], T, dwih[:, off:], D, dev)
                    else:
                        weight_grad(dgT, y_in.data_ptr() + 4 * e * 2 * H, 0, ycols, N, 2 * H, N, dwih, D, dev)
                        # gradient to the lower layer's output: dgx W_ih, straight into its column block of dy_next
                        if "wih_t" not in layers[layer]:
                            layers[layer]["wih_t"] = {}
                        if e not in layers[layer]["wih_t"]:
                            layers[layer]["wih_t"][e] = split_tf32(torch.cat([w_f.detach(), w_r.detach()], dim=0).t().contiguous(),
                                                                   side=B_SIDE)
                        wt = layers[layer]["wih_t"][e]
                        dg_hl = split_tf32(dg)
                        gemm_tf32x3(dg_hl[0], dg_hl[1], wt[0], wt[1], None, dy_next.view(N, ycols)[:, e * 2 * H:], N, D,
                                    ldc=ycols)
                    for d, shift in ((0, -1), (1, 1)):
                        weight_grad((dgT[0][d * 4 * H:(d + 1) * 4 * H], dgT[1][d * 4 * H:(d + 1) * 4 * H]),
                                    yo.data_ptr() + 4 * (e * 2 * H + d * H), T * ycols, ycols, N, H, T, dwhh[d], H, dev,
                                    shift=shift, lengths=lens.dev)
                else:  # exact-fp32 CUDA-core GEMMs (MTS_GEMM_IMPL=simt): the second opinion for the tensor-core path
                    if layer == 0:
                        for x, off in srcs:
                            xc = x if (x.shape[1] == T and x.is_contiguous()) else x[:, :T].contiguous()
                            Dx = xc.shape[2]
                            gemm_f32(_ptr(dg), 8 * H, _ptr(xc), Dx, None, dwih.data_ptr() + 4 * off, D, 8 * H, Dx, N,
                                     layout=3, splits=splits)
                    else:
                        xin = y_in.view(N, ycols)
                        gemm_f32(_ptr(dg), 8 * H, xin.data_ptr() + 4 * e * 2 * H, ycols, None, _ptr(dwih), D,
                                 8 * H, D, N, layout=3, splits=splits)
                        wcat = torch.cat([w_f.detach(), w_r.detach()], dim=0)
                        gemm_f32(_ptr(dg), 8 * H, _ptr(wcat), D, None, dy_next.data_ptr() + 4 * e * 2 * H, ycols,
                                 N, D, 8 * H, layout=2)
                    for d, shift in ((0, -1), (1, 1)):
                        gemm_f32(dg.data_ptr() + 4 * d * 4 * H, 8 * H, yo.data_ptr() + 4 * (e * 2 * H + d * H),
                                 ycols, None, _ptr(dwhh[d]), H, 4 * H, H, N, layout=3, splits=splits, shift=shift,
                                 T=T, lengths=lens.dev)
                if layer == 0 and ctx.needs_input_grad[0] and n_enc == 1 and ctx.x2 is None:
                    # gradient to the stack's own input: dgx W_ih (same product as between layers)
                    wcat = torch.cat([w_f.detach(), w_r.detach()], dim=0)
                    dxt = torch.empty((N, D), device=dev, dtype=torch.float32)
                    if tensor_core:
                        wt = split_tf32(wcat.t().contiguous(), side=B_SIDE)
                        dg_hl = split_tf32(dg)
                        gemm_tf32x3(dg_hl[0], dg_hl[1], wt[0], wt[1], None, dxt, N, D)
                    else:
                        gemm_f32(_ptr(dg), 8 * H, _ptr(wcat), D, None, _ptr(dxt), D, N, D, 8 * H, layout=2)
                    dx_in = dxt.view(B, T, D)
                    if ctx.x1.shape[1] != T:
                        dx_in = torch.nn.functional.pad(dx_in, (0, 0, 0, ctx.x1.shape[1] - T))
                base = 8 * layer
                g = grads[e]
                g[base + 0], g[base + 1] = dwih[:4 * H], dwhh[0]
                # b_ih and b_hh receive the same gradient but must not share storage: AccumulateGrad may adopt the
                # tensors as .grad, and an in-place op on one (clip_grad_norm_, a second backward) would hit both
                g[base + 2], g[base + 3] = db[:4 * H], db[:4 * H].clone()
                g[base + 4], g[base + 5] = dwih[4 * H:], dwhh[1]
                g[base + 6], g[base + 7] = db[4 * H:], db[4 * H:].clone()
            dy = dy_next
        flat = [g for e in range(n_enc) for g in grads[e]]
        ctx.saved = None
        return (dx_in, None, None, None, None, None, *flat)


# --------------------------------------------------------------------------------------------------------
# head, decode, losses
# --------------------------------------------------------------------------------------------------------
class HeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, w, b):
        _check(feats, "features")
        feats = feats.contiguous()
        B, T, F = feats.shape
        n_out = w.shape[0]
        scores = torch.empty((B, T, n_out), device=feats.device, dtype=torch.float32)
        wc, bc = w.contiguous(), b.contiguous()
        _call("mts_head_fwd", _ptr(feats), _ptr(wc), _ptr(bc), 0, B, T, F, n_out, 0.0, _ptr(scores), 0, _stream())
        ctx.save_for_backward(feats, wc)
        return scores

    @staticmethod
    def backward(ctx, ds):
        feats, w = ctx.saved_tensors
        B, T, F = feats.shape
        n_out = w.shape[0]
        ds = ds.contiguous()
        dx = torch.empty_like(feats) if ctx.needs_input_grad[0] else None
        dw = torch.empty_like(w)
        db = torch.empty(n_out, device=w.device, dtype=torch.float32)
        ws = torch.empty(_lib.load().mts_head_bwd_ws_bytes(B, T, F, n_out) // 4, device=w.device, dtype=torch.float32)
        _call("mts_head_bwd", _ptr(ds), _ptr(feats), _ptr(w), B, T, F, n_out, _ptr(dx), _ptr(dw), _ptr(db), _ptr(ws),
              _stream())
        return dx, dw, db


def head_decode(feats, w, b, lens, th):
    """scores [B,T,n_out] and uint8 tags [B,T] (0xFF beyond len_b) in one kernel."""
    feats = _check(feats, "features").contiguous()
    B, T, F = feats.shape
    n_out = w.shape[0]
    scores = torch.empty((B, T, n_out), device=feats.device, dtype=torch.float32)
    tags = torch.empty((B, T), device=feats.device, dtype=torch.uint8)
    _call("mts_head_fwd", _ptr(feats), _ptr(w.contiguous()), _ptr(b.contiguous()), _ptr(lens.dev), B, T, F, n_out,
          float(th), _ptr(scores), _ptr(tags), _stream())
    return scores, tags


def seg_metrics(tags_u8, target, lens, zero_last=False):
    """Per-episode evaluation counts on the device: int32 [B, 8] = {Pk mismatches, WindowDiff mismatches, windows,
    k, tp, fp, fn, reference segments} (see mts_seg_metrics)."""
    tags_u8 = _check(tags_u8, "tags", torch.uint8)
    target = _check(target, "target")
    if target.stride(-1) != 1:
        target = target.contiguous()
    if tags_u8.stride(-1) != 1:
        tags_u8 = tags_u8.contiguous()
    B, T = tags_u8.shape
    out = torch.empty((B, 8), device=tags_u8.device, dtype=torch.int32)
    _call("mts_seg_metrics", _ptr(tags_u8), tags_u8.stride(0), _ptr(target), target.stride(0), _ptr(lens.dev), B, T,
          int(bool(zero_last)), _ptr(out), _stream())
    return out


LOSS_KINDS = {"FocalLoss": 0, "BinaryCrossEntropy": 1, "CrossEntropy": 2}


class SegLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scores, target, lens, kind, alpha, gamma, inv_count):
        scores = _check(scores, "scores").contiguous()
        target = _check(target, "target")
        if target.stride(-1) != 1:
            target = target.contiguous()
        B, T = scores.shape[0], scores.shape[1]
        out = torch.empty(2, device=scores.device, dtype=torch.float32)
        partial = torch.empty(2048, device=scores.device, dtype=torch.float32)
        _call("mts_seg_loss_fwd", _ptr(scores), _ptr(target), target.stride(0), _ptr(lens.dev), B, T, kind, alpha, gamma,
              inv_count, _ptr(out), _ptr(partial), _stream())
        ctx.save_for_backward(scores, target, out)
        ctx.args = (lens, kind, alpha, gamma, inv_count)
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        scores, target, out = ctx.saved_tensors
        lens, kind, alpha, gamma, inv_count = ctx.args
        B, T = scores.shape[0], scores.shape[1]
        ds = torch.empty_like(scores)
        go = grad_out.contiguous().reshape(1)
        _call("mts_seg_loss_bwd", _ptr(scores), _ptr(target), target.stride(0), _ptr(lens.dev), B, T, kind, alpha, gamma,
              inv_count, out.data_ptr() + 4, _ptr(go), _ptr(ds), _stream())
        return ds, None, None, None, None, None, None


# --------------------------------------------------------------------------------------------------------
# CRF
# --------------------------------------------------------------------------------------------------------
def crf_viterbi(emis, lens, trans):
    emis = _check(emis, "emissions").contiguous()
    B, L, C = emis.shape
    best = torch.empty(B, device=emis.device, dtype=torch.float32)
    paths = torch.empty((B, L), device=emis.device, dtype=torch.int32)
    bp = torch.empty((B, L), device=emis.device, dtype=torch.int32)
    _call("mts_crf_viterbi", _ptr(emis), _ptr(lens.dev), _ptr(trans.detach().contiguous()), B, L, C, _ptr(best),
          _ptr(paths), _ptr(bp), _stream())
    return best, paths


class CrfNllFn(torch.autograd.Function):
    """mean_b (log Z_b - gold_b)  (models/CRF.py:130-146 after `fc`)."""

    @staticmethod
    def forward(ctx, emis, trans, tags, lens):
        emis = _check(emis, "emissions").contiguous()
        trans_c = trans.contiguous()
        B, L, C = emis.shape
        tags = tags if tags.stride(-1) == 1 else tags.contiguous()
        stats = torch.empty((2, B), device=emis.device, dtype=torch.float32)
        alphas = torch.empty((B, L, C), device=emis.device, dtype=torch.float32)
        _call("mts_crf_nll_fwd", _ptr(emis), _ptr(tags), tags.stride(0), _ptr(lens.dev), _ptr(trans_c), B, L, C,
              _ptr(stats[0]), _ptr(stats[1]), _ptr(alphas), _stream())
        ctx.save_for_backward(emis, trans_c, tags, alphas, stats)
        ctx.lens = lens
        return stats  # [2, B]: log Z and gold score; the caller takes (stats[0] - stats[1]).mean()

    @staticmethod
    def backward(ctx, dstats):
        emis, trans, tags, alphas, stats = ctx.saved_tensors
        B, L, C = emis.shape
        # d loss / d logZ_b = dstats[0, b] stays on the device (the loss only ever uses logZ - gold, so
        # dstats[1] = -dstats[0]); for the reference's mean this is grad_out / B.
        scale = dstats[0].contiguous()
        de = torch.empty_like(emis)
        dt = torch.empty_like(trans)
        _call("mts_crf_nll_bwd", _ptr(emis), _ptr(tags), tags.stride(0), _ptr(ctx.lens.dev), _ptr(trans), _ptr(alphas),
              B, L, C, _ptr(scale), _ptr(de), _ptr(dt), _stream())
        return de, dt, None, None
