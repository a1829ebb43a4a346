"""Host-side mirror of the reference's segmenter objects -- same class names, constructor signatures,
method signatures, return conventions and state-dict keys as models/CRF.py and
models/NeuralArchitectures.py of Ighina/MultimodalTopicSegmentation -- with every arithmetic step
running in libmts_b200.so (sm_100a kernels).  Nothing here computes on the CPU.

    RNN                  <- models/NeuralArchitectures.py:23-145
    CRF                  <- models/CRF.py:98-240
    BiRnnCrf             <- models/CRF.py:243-272 (with the intended wiring; the reference's unpacking bug,
                            SURVEY.md fact 6, is not reproduced)
    BiLSTM               <- models/CRF.py:274-369
    BiLSTMLateFusion     <- models/CRF.py:371-479
    Transformer_segmenter<- models/CRF.py:508-610 (see transformer.py)

Additive API (SURVEY.md section 8f row 1): `xs` may be a pair (text, audio) of [B,T,D_i] tensors; the early-fusion
concat then happens inside the operand-packing kernel instead of on the host.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

IMPOSSIBLE = -1e4  # models/CRF.py:95


def _lens(lengths, x):
    """Lengths of a batch whose embeddings x are a [B, T, D] tensor or an early-fusion pair of them (time axis of the first)."""
    if isinstance(lengths, ops.Lengths):
        return lengths
    if isinstance(x, (tuple, list)):
        x = x[0]
    return ops.Lengths(lengths, x.device, x.shape[1])


def _host_tags_to_lists(host, lens, as_bool):
    """uint8 tag matrix on the host (numpy) -> the reference's per-episode cropped lists (CRF.py:369)."""
    full = (host.astype(bool) if as_bool else host.astype(int)).tolist()  # one conversion for the whole matrix
    return [row if n == len(row) else row[:n] for row, n in zip(full, lens.host)]


def _tags_to_lists(tags_dev, lens, as_bool):
    """One device->host copy of the uint8 tag matrix, then the per-episode crop."""
    return _host_tags_to_lists(tags_dev.cpu().numpy(), lens, as_bool)


class RNN(nn.Module):
    """Bi-LSTM encoder over variable-length episodes.  `self.rnn` is a plain nn.LSTM used as the parameter
    container (so checkpoints are interchangeable with the reference); its forward is never called."""

    def __init__(self, embed_size, hidden_size, num_layers=1, labels=1, bidirectional=False, dropout_in=0.0,
                 dropout_out=0.0, padding_idx=0, batch_first=True, LSTM=True):
        super().__init__()
        if not LSTM:
            raise NotImplementedError("the B200 path implements the LSTM cell only (GRU is outside BASELINE configs)")
        if not bidirectional or not batch_first:
            raise NotImplementedError("the B200 path implements the bidirectional, batch-first encoder only")
        self.embed_size, self.hidden_size = embed_size, hidden_size
        self.labels, self.num_layers, self.bidirectional = labels, num_layers, bidirectional
        self.rnn = nn.LSTM(input_size=embed_size, hidden_size=hidden_size, batch_first=True, num_layers=num_layers,
                           bidirectional=True)
        self.dropout_in, self.dropout_out = dropout_in, dropout_out
        self._reinitialize()
        self._packed = None

    def _reinitialize(self):
        # same order and the same initialisers as NeuralArchitectures.py:58-79 => identical weights under a seed
        for name, p in self.named_parameters():
            if "weight_ih" in name:
                nn.init.xavier_uniform_(p.data)
            elif "weight_hh" in name:
                nn.init.orthogonal_(p.data)
            elif "bias_ih" in name:
                p.data.fill_(0)
                n = p.size(0)
                p.data[(n // 4):(n // 2)].fill_(1)
            elif "bias_hh" in name:
                p.data.fill_(0)

    def packed(self):
        if self._packed is None:
            self._packed = ops.PackedLstm([self.rnn])
        return self._packed

    def forward(self, line, line_len=None, apply_softmax=False, return_final=False, classifier=False):
        if return_final:
            raise NotImplementedError("return_final is not used on the segmentation path")
        x1, x2 = (line if isinstance(line, (tuple, list)) else (line, None))
        if line_len is None:
            line_len = [x1.shape[1]] * x1.shape[0]
        lens = _lens(line_len, x1)
        if self.dropout_in:
            x1 = F.dropout(x1, p=self.dropout_in)  # active in eval too, as in the reference (SURVEY fact 9)
            x2 = F.dropout(x2, p=self.dropout_in) if x2 is not None else None
        packed = self.packed()
        out = ops.bilstm_stack(ops._check(x1, "input", x1.dtype if x1.dtype == torch.bfloat16 else torch.float32), x2, None, lens,
                               packed, 1)
        if self.dropout_out:
            out = F.dropout(out, p=self.dropout_out)
        return out


def _build_head(mod, in_features, tagset_size, loss_fn, threshold, alpha, gamma):
    if loss_fn not in ops.LOSS_KINDS:
        raise ValueError("Choose one of CrossEntropy or BinaryCrossEntropy as loss function")
    mod.loss_name = loss_fn
    mod.bce = loss_fn != "CrossEntropy"
    mod.fl = loss_fn == "FocalLoss"
    mod.classification = nn.Linear(in_features, 1 if mod.bce else tagset_size)
    mod.alpha, mod.gamma = float(alpha), float(gamma)
    mod.th = threshold


def _head_loss(mod, feats, lens, tags, global_count=None):
    """classification -> un-pad -> loss (CRF.py:340-356) as two kernels.  `global_count`: number of valid
    sentences over ALL data-parallel ranks (defaults to this batch's), so the mean matches the un-sharded loss."""
    if (not mod.bce) and mod.classification.out_features != 2:
        raise NotImplementedError("the CrossEntropy head is implemented for tagset_size == 2")
    scores = ops.HeadFn.apply(feats, mod.classification.weight, mod.classification.bias)
    kind = ops.LOSS_KINDS[mod.loss_name]
    tags = ops._check(tags.to(feats.device), "tags")
    if global_count is not None:
        # data parallel: normalise by the count over ALL ranks (for CrossEntropy that is the number of non-ignored
        # targets = the number of valid sentences, since the collater pads the tags with -1 exactly beyond len_b)
        inv = 1.0 / float(global_count)
    elif kind == 2:
        inv = -1.0  # CrossEntropyLoss(ignore_index=-1): the kernel counts the non-ignored targets itself
    else:
        inv = 1.0 / float(lens.N)
    return ops.SegLossFn.apply(scores, tags, lens, kind, mod.alpha, mod.gamma, inv)


def _head_decode_device(mod, feats, lens, threshold):
    """scores [B,T,n_out] and uint8 tags [B,T] (0xFF beyond len_b), both left on the device."""
    if mod.th is not None:
        threshold = mod.th
    return ops.head_decode(feats, mod.classification.weight.detach(), mod.classification.bias.detach(), lens, threshold)


def _head_decode(mod, feats, lens, threshold):
    scores, tags = _head_decode_device(mod, feats, lens, threshold)
    return scores, _tags_to_lists(tags, lens, as_bool=True)


class BiLSTM(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=1, bidirectional=True, dropout_in=0.0,
                 dropout_out=0.0, batch_first=True, LSTM=True, loss_fn="CrossEntropy", threshold=None, device=None,
                 alpha=0.9, gamma=2):
        super().__init__()
        self.embedding_dim, self.hidden_dim, self.tagset_size = embedding_dim, hidden_dim, tagset_size
        self.device = device if device is not None else "cuda"
        self.model = RNN(embedding_dim, hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                         batch_first=batch_first, LSTM=LSTM)
        _build_head(self, hidden_dim * 2, tagset_size, loss_fn, threshold, alpha, gamma)

    def loss(self, xs, lengths, tags, segments=None, global_count=None):
        if segments is not None:
            raise NotImplementedError("the auxiliary cosine loss (segments=...) is outside the B200 hot path")
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lengths, x0)
        return _head_loss(self, self.model(xs, lens), lens, tags, global_count)

    def forward(self, xs, lenghts, threshold=0.4):
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lenghts, x0)
        with torch.no_grad():
            return _head_decode(self, self.model(xs, lens), lens, threshold)

    def decode_device(self, xs, lenghts, threshold=0.4):
        """forward() without the device->host hop: (scores, uint8 tags [B,T] on the device, Lengths)."""
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lenghts, x0)
        with torch.no_grad():
            return (*_head_decode_device(self, self.model(xs, lens), lens, threshold), lens)


class BiLSTMLateFusion(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=1, bidirectional=True, dropout_in=0.0,
                 dropout_out=0.0, batch_first=True, LSTM=True, loss_fn="CrossEntropy", threshold=None, device=None,
                 alpha=0.9, gamma=2):
        super().__init__()
        self.embedding_dim, self.hidden_dim, self.tagset_size = embedding_dim, hidden_dim, tagset_size
        self.device = device if device is not None else "cuda"
        self.model1 = RNN(embedding_dim[0], hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                          batch_first=batch_first, LSTM=LSTM)
        self.model2 = RNN(embedding_dim[1], hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                          batch_first=batch_first, LSTM=LSTM)
        _build_head(self, hidden_dim * 4, tagset_size, loss_fn, threshold, alpha, gamma)
        self._packed = None

    def _features(self, x1, x2, lens):
        """Both encoders advance in ONE recurrence launch per layer (n_enc = 2): their clusters run side by side
        and the output already has the reference's torch.cat((x1, x2), axis=2) layout (CRF.py:425)."""
        if self._packed is None:
            self._packed = ops.PackedLstm([self.model1.rnn, self.model2.rnn])
        p_in = self.model1.dropout_in
        if p_in:
            x1, x2 = F.dropout(x1, p=p_in), F.dropout(x2, p=p_in)
        dt = x1.dtype if x1.dtype == torch.bfloat16 else torch.float32   # bf16 embeddings: the bf16 path (ops.set_precision)
        out = ops.bilstm_stack(ops._check(x1, "x1", dt), None, ops._check(x2, "x2", dt), lens, self._packed, 2)
        if self.model1.dropout_out:
            out = F.dropout(out, p=self.model1.dropout_out)
        return out

    def loss(self, x1, x2, lengths, tags, segments=None, global_count=None):
        if segments is not None:
            raise NotImplementedError("the auxiliary cosine loss (segments=...) is outside the B200 hot path")
        lens = _lens(lengths, x1)
        return _head_loss(self, self._features(x1, x2, lens), lens, tags, global_count)

    def forward(self, x1, x2, lenghts, threshold=0.4):
        lens = _lens(lenghts, x1)
        with torch.no_grad():
            return _head_decode(self, self._features(x1, x2, lens), lens, threshold)

    def decode_device(self, x1, x2, lenghts, threshold=0.4):
        lens = _lens(lenghts, x1)
        with torch.no_grad():
            return (*_head_decode_device(self, self._features(x1, x2, lens), lens, threshold), lens)


class BiLSTMLateFusionCrf(nn.Module):
    """Late-fusion dual encoder with a CRF output layer: text and audio bi-LSTM stacks -> cat [B,T,4H] -> CRF(4H, tags).
    BASELINE configs[3] names this combination; the reference has both halves (BiLSTMLateFusion, models/CRF.py:371-479,
    and CRF, :98-240) but no class wiring them, so this is the composition SURVEY.md fact 6 describes for BiRnnCrf,
    applied to the late-fusion encoder.  Parameter names: model1.rnn.*, model2.rnn.*, crf.fc.*, crf.transitions."""

    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=1, bidirectional=True, dropout_in=0.0,
                 dropout_out=0.0, batch_first=True, LSTM=True):
        super().__init__()
        self.embedding_dim, self.hidden_dim, self.tagset_size = embedding_dim, hidden_dim, tagset_size
        self.device = "cuda"
        self.model1 = RNN(embedding_dim[0], hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                          batch_first=batch_first, LSTM=LSTM)
        self.model2 = RNN(embedding_dim[1], hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                          batch_first=batch_first, LSTM=LSTM)
        self.crf = CRF(hidden_dim * 4, tagset_size)
        self.th = None
        self._packed = None

    _features = BiLSTMLateFusion._features

    def loss(self, x1, x2, lengths, tags, segments=None, global_count=None):
        lens = _lens(lengths, x1)
        return self.crf.loss(self._features(x1, x2, lens), tags[:, : lens.T], lens, global_count=global_count)

    def forward(self, x1, x2, lenghts, threshold=None):
        lens = _lens(lenghts, x1)
        with torch.no_grad():
            return self.crf(self._features(x1, x2, lens), lens)

    def decode_device(self, x1, x2, lenghts, threshold=None):
        lens = _lens(lenghts, x1)
        with torch.no_grad():
            best, paths = ops.crf_viterbi(self.crf.emissions(self._features(x1, x2, lens)), lens, self.crf.transitions)
        return best, paths.to(torch.uint8), lens


class CRF(nn.Module):
    """General CRF module: inner Linear to tag space, transitions[i, j] = j -> i, START/STOP appended."""

    def __init__(self, in_features, num_tags):
        super().__init__()
        self.num_tags = num_tags + 2
        self.start_idx, self.stop_idx = self.num_tags - 2, self.num_tags - 1
        self.fc = nn.Linear(in_features, self.num_tags)
        self.transitions = nn.Parameter(torch.randn(self.num_tags, self.num_tags), requires_grad=True)
        self.transitions.data[self.start_idx, :] = IMPOSSIBLE
        self.transitions.data[:, self.stop_idx] = IMPOSSIBLE

    @staticmethod
    def _lens_from_masks(masks, features):
        if isinstance(masks, ops.Lengths):
            return masks
        return ops.Lengths(masks[:, : features.size(1)].sum(1), features.device, features.size(1))

    def emissions(self, features):
        return ops.LinearFn.apply(features, self.fc.weight, self.fc.bias)

    def forward(self, features, masks):
        """-> (best_score [B], best_paths list[B] of list[len_b] of int)   (CRF.py:119-128, 172-216)"""
        lens = self._lens_from_masks(masks, features)
        with torch.no_grad():
            best, paths = ops.crf_viterbi(self.emissions(features), lens, self.transitions)
        return best, _tags_to_lists(paths, lens, as_bool=False)

    def loss(self, features, ys, masks, global_count=None):
        """negative log likelihood, mean over the batch (CRF.py:130-146).  `global_count`: number of episodes over
        all data-parallel ranks (defaults to this batch's)."""
        lens = self._lens_from_masks(masks, features)
        emis = self.emissions(features)
        ys = ops._check(ys.to(features.device).float(), "tags")
        stats = ops.CrfNllFn.apply(emis, self.transitions, ys, lens)
        nll = stats[0] - stats[1]
        return nll.mean() if global_count is None else nll.sum() / float(global_count)


class BiRnnCrf(nn.Module):
    def __init__(self, tagset_size, embedding_dim, hidden_dim, num_layers=1, bidirectional=True, dropout_in=0.0,
                 dropout_out=0.0, batch_first=True, LSTM=True, architecture="rnn"):
        super().__init__()
        self.embedding_dim, self.hidden_dim, self.tagset_size = embedding_dim, hidden_dim, tagset_size
        self.device = "cuda"
        if architecture != "rnn":
            raise ValueError("only the 'rnn' encoder is implemented for BiRnnCrf")
        self.model = RNN(embedding_dim, hidden_dim, num_layers, tagset_size, bidirectional, dropout_in, dropout_out,
                         batch_first=batch_first, LSTM=LSTM)
        self.crf = CRF(hidden_dim * 2, self.tagset_size)
        self.th = None  # test_step assigns it on every model (lightning_model.py:587); unused by Viterbi

    def loss(self, xs, lengths, tags, segments=None, global_count=None):
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lengths, x0)
        return self.crf.loss(self.model(xs, lens), tags[:, : lens.T], lens, global_count=global_count)

    def forward(self, xs, lenghts, threshold=None):
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lenghts, x0)
        with torch.no_grad():
            return self.crf(self.model(xs, lens), lens)

    def decode_device(self, xs, lenghts, threshold=None):
        """(best_score [B], uint8 Viterbi tags [B,T] on the device (0xFF beyond len_b), Lengths)."""
        x0 = xs[0] if isinstance(xs, (tuple, list)) else xs
        lens = _lens(lenghts, x0)
        with torch.no_grad():
            best, paths = ops.crf_viterbi(self.crf.emissions(self.model(xs, lens)), lens, self.crf.transitions)
        return best, paths.to(torch.uint8), lens  # -1 (padding) wraps to 0xFF
