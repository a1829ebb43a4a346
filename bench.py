#!/usr/bin/env python
"""Benchmark of the segmentation hot path on B200 (contract: one JSON line on stdout from rank 0).

    python bench.py --gpus 1 --steps 20 --warmup 5            # our arm (CUDA kernels through the C ABI)
    python bench.py --impl reference --steps 5 --warmup 1     # reference arm: the reference's CPU path on host cores
    python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...   # one rank per GPU, weak scaling

Headline workload (BASELINE.json configs[0] shape, the configuration the sentences/sec metric is quoted on):
early-fusion BiLSTM segmenter, 64 episodes x 300 sentences, 384-d text + 512-d audio embeddings, hidden 256,
2 layers, sigmoid head thresholded at 0.5.  A step = one inference pass over one batch: operand packing
(fused concat), two input-projection GEMMs (tcgen05, TF32 + bf16 error compensation), two bidirectional recurrence
launches, head+decode.

  value  : sentences/s with the inputs resident in HBM (CUDA events over exactly K steps, max over ranks).
  e2e    : the same through TextSegmenter.predict_batches with HOST (pinned) inputs, H2D copies and the D2H of the
           tags inside the timed region.
  roofline: the LSTM recurrence kernel (dominant), algorithmic HBM bytes per launch / its CUDA-event time, at the
           configuration's batch and (`saturating`) at the batch where the fraction stops growing.
  cpu_baseline: the reference's CPU path on the box's host cores, same batch shape.
  legs   : every other BASELINE configuration, one short key each (full records under their own keys):
           configs[1] focal + CRF training step and BiLSTM+CRF decode, configs[2] windowed-attention segmenter,
           configs[3] late-fusion (+CRF) data-parallel training, configs[4] 8192-sentence episodes, CRF kernels.
Synthetic data, random-init weights (reference initialisers, seed 0).  L2: rotating input sets larger than the 126 MB L2.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(B=64, T=300, D1=384, D2=512, H=256, L=2)
WORKLOAD = "cfg1-shaped early-fusion BiLSTM inference: 64 episodes x 300 sentences, 384-d text + 512-d audio, H256 x 2 layers"
ALGO_BYTES_PER_SENTENCE_REC = 10240  # SURVEY.md section 8(d): read gx 8 H x 4 B + write h 2 H x 4 B, both directions
# DRAM traffic of ONE lstm_fwd_tc_kernel launch at the cfg1 shape (64 x 300, inference) from the ncu --set full capture in
# profiles/r01_ncu_summary.md: 159.46 MB read + 25.64 MB written (algorithmic: 157.3 MB gx in + 39.3 MB h out; part of
# the output is still in L2 when the kernel ends)
NCU_REC_DRAM_BYTES = 159459840 + 25640448
# the same for lstm_fwd_h3_kernel (profiles/r02_ncu_summary.md, capture r02b): 159.63 MB read + 25.96 MB written
NCU_REC_H3_DRAM_BYTES = 159627264 + 25957120


def synth(seed, B, T, D1, D2, ragged=False):
    g = torch.Generator().manual_seed(1234 + seed)
    x1 = torch.randn(B, T, D1, generator=g)
    x2 = torch.randn(B, T, D2, generator=g)
    if ragged:
        lengths = torch.randint(84, T + 1, (B,), generator=g)
        lengths[0] = T
    else:
        lengths = torch.full((B,), T, dtype=torch.long)
    return x1, x2, lengths


def dump_outputs(out_dir, scores, tags):
    """What the last timed headline step returned, as <out_dir>/<name>.npy in float32: the head's scores [B, T, n_out]
    and the thresholded boundary tags [B, T] (255 beyond an episode's length), the batches of all ranks in rank order.
    The inputs and weights are seeded, so the files of two builds can be compared array for array."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("scores", scores), ("tags", tags)):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        """Median SM clock over the samples taken UNDER LOAD (power draw >= 60 % of the highest seen: the legs contain
        host-side set-up during which the GPU idles), throttle reasons over all samples."""
        rows, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                rows.append((float(r[0]), float(r[1]), float(r[2])))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(reasons), "samples": 0}
        pmax = max(p for _, _, p in rows)
        loaded = [r for r in rows if r[2] >= 0.6 * pmax]
        return {"sm_mhz": statistics.median(r[0] for r in loaded), "sm_max_mhz": max(r[1] for r in rows),
                "reasons": sorted(reasons), "samples": len(rows), "samples_under_load": len(loaded),
                "power_w_max": pmax}


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


_AFFINITY0 = None


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank (and the e2e leg may have bound this rank to its GPU's NUMA node);
    the CPU legs run on rank 0 alone and may use the whole host."""
    if _AFFINITY0 is not None:
        try:
            os.sched_setaffinity(0, _AFFINITY0)
        except OSError:
            pass
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    if torch.get_num_threads() < n:
        torch.set_num_threads(n)
    return torch.get_num_threads()


# ----------------------------------------------------------------------------------------------------------------
# the reference arm: the reference's own modules from baseline/_ref (copied there by __graft_entry__.build() when
# /root/reference is present; git-ignored, travels to the GPU box), else the oracle port of the same torch calls
# ----------------------------------------------------------------------------------------------------------------
def reference_modules():
    """-> (kind, BiLSTM class of the reference or None).  kind "reference" = the unmodified models/CRF.py."""
    base = os.path.join(ROOT, "baseline", "_ref")
    if os.path.exists(os.path.join(base, "models", "CRF.py")):
        try:
            import types

            import torch.nn as nn

            if base not in sys.path:
                sys.path.insert(0, base)
            stub = types.ModuleType("models.longformer_noffn")   # missing upstream (SURVEY fact 7), never used on this path

            class LongformerLayer(nn.Module):
                def __init__(self, *a, **k):
                    super().__init__()

            stub.LongformerLayer = LongformerLayer
            sys.modules.setdefault("models.longformer_noffn", stub)
            import models.CRF as ref_crf

            return "reference", ref_crf
        except Exception as exc:  # e.g. an HF version the reference's imports do not survive
            print(f"[bench] baseline/_ref present but not importable ({type(exc).__name__}: {exc}); using the port", file=sys.stderr)
    return "port", None


def cpu_reference(steps, warmup):
    """The reference's CPU implementation of the headline path, all host threads."""
    use_all_host_threads()
    torch.manual_seed(0)
    c = CFG
    kind, ref_crf = reference_modules()
    if ref_crf is not None:
        model = ref_crf.BiLSTM(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], bidirectional=True, dropout_in=0.0,
                               dropout_out=0.0, batch_first=True, LSTM=True, loss_fn="FocalLoss", threshold=0.5)
        what = "baseline/_ref/models/CRF.py::BiLSTM (the unmodified reference module)"
    else:
        from oracle import ref_torch as rt

        model = rt.Segmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], loss_fn="FocalLoss", threshold=0.5)
        what = "oracle/ref_torch.py (the reference's torch calls: nn.LSTM + Linear + sigmoid threshold)"
    x1, x2, lengths = synth(0, c["B"], c["T"], c["D1"], c["D2"])
    x = torch.cat([x1, x2], dim=-1)  # the reference concatenates at load time (not timed)
    cores = torch.get_num_threads()
    with torch.no_grad():
        for _ in range(warmup):
            model(x, lengths)
        t0 = time.perf_counter()
        for _ in range(steps):
            model(x, lengths)
        dt = time.perf_counter() - t0
    n_sent = int(lengths.sum()) * steps
    return n_sent / dt, dt / steps * 1e3, cores, kind, what


def run_reference(args, rank, world):
    if rank != 0:
        return
    value, ms, cores, kind, what = cpu_reference(args.steps, max(args.warmup, 1))
    line = {"impl": "reference", "metric": "segmented sentences/sec", "value": value, "unit": "sentences/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": value, "unit": "sentences/s", "cores": cores, "kind": kind,
                             "sample": f"{args.steps} full batches of 64x300 sentences through {what} on host cores, all torch threads"},
            "e2e": {"value": value, "unit": "sentences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# helpers for the GPU legs
# ----------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, m, dev, rank, world, local_rank):
        self.m, self.dev, self.rank, self.world, self.local_rank = m, dev, rank, world, local_rank

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        import torch.distributed as dist

        t = torch.tensor([float(v)], device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, step, steps, warm=2):
        """ms per step: CUDA events around exactly `steps` calls, barrier + synchronize on both sides, max over ranks."""
        from multimodaltopicsegmentation_b200 import ops

        for i in range(warm):
            step(i)
        self.barrier()
        ops.reset_launch_count()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for i in range(steps):
            step(i)
        end.record()
        self.barrier()
        launches = ops.launch_count()
        return self.max_over_ranks(start.elapsed_time(end)) / steps, launches / steps

    def profile(self, step, n=1):
        """per ABI entry point: list of CUDA-event durations (ms) over n eager calls of step"""
        from multimodaltopicsegmentation_b200 import ops

        ops.PROFILE = {}
        for i in range(n):
            step(i)
        torch.cuda.synchronize()
        prof = {k: [s.elapsed_time(e) for s, e in v] for k, v in ops.PROFILE.items()}
        ops.PROFILE = None
        return prof


def rec_roofline(prof, n_sent, note=None):
    """HBM roofline record of the recurrence kernel from a profile pass: algorithmic bytes per launch / mean launch time"""
    name = "mts_lstm_rec_fwd_tc" if "mts_lstm_rec_fwd_tc" in prof else "mts_lstm_rec_fwd"
    if name not in prof:
        return None
    hbm_peak, peak_src = peaks()
    ms = sum(prof[name]) / len(prof[name])
    nbytes = n_sent * ALGO_BYTES_PER_SENTENCE_REC
    achieved = nbytes / (ms / 1e3) / 1e9
    tc_kernel = "lstm_fwd_tc_kernel" if os.environ.get("MTS_REC_TC", "").startswith("t") else "lstm_fwd_h3_kernel"
    out = {"kernel": (tc_kernel if name.endswith("_tc") else "lstm_fwd_cluster_kernel") + " (one launch per layer, both directions)",
           "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
           "peak_source": peak_src, "algorithmic_bytes_per_launch": nbytes, "avg_launch_ms": ms}
    if note:
        out["note"] = note
    return out


# ----------------------------------------------------------------------------------------------------------------
# training legs (configs[1] focal / CRF, configs[3] late fusion focal / CRF)
# ----------------------------------------------------------------------------------------------------------------
TRAIN_LEGS = {
    # key: (architecture, per-GPU batch, (Tmin, Tmax), dims, workload text)
    "train": ("BiLSTM", 10, (84, 2437), (896,),
              "configs[1]: early-fusion BiLSTM focal-loss training step (fwd + BPTT + Adam), NonNews-shaped batch of 10 "
              "episodes, 84..2437 sentences, 896-d inputs, H256 x 2 layers"),
    "train_crf": ("biLSTMCRF", 10, (84, 2437), (896,),
                  "configs[1]: early-fusion BiLSTM -> CRF training step (NLL by the forward algorithm, fwd + bwd + Adam), same batch"),
    "latefusion_train": ("BiLSTMLateFusion", 10, (84, 300), (384, 512),
                         "configs[3]: late-fusion dual-encoder BiLSTM focal-loss training step, 10 episodes per GPU, 84..300 "
                         "sentences, 384-d text + 512-d audio, H256 x 2 layers per encoder (24.2 MB gradient bucket)"),
    "latefusion_train_b64": ("BiLSTMLateFusion", 64, (84, 300), (384, 512),
                             "configs[3] at 64 episodes per GPU (the upper end SURVEY.md section 8d names)"),
    "latefusion_crf_train": ("BiLSTMLateFusionCRF", 10, (84, 300), (384, 512),
                             "configs[3] with the CRF output layer: dual encoders -> CRF(4H, 2) NLL training step, 10 episodes per GPU"),
}


def train_batch(key, rank, variant):
    """The SAME multiset of episode lengths on every rank (weak scaling keeps the per-GPU work fixed: the recurrence's
    step count is the longest episode of the rank), different embeddings / labels per rank and variant."""
    arch, B, (tmin, tmax), dims, _ = TRAIN_LEGS[key]
    g = torch.Generator().manual_seed(4321 + variant)
    lengths = torch.randint(tmin, tmax + 1, (B,), generator=g)
    lengths[0] = tmax
    gr = torch.Generator().manual_seed(99 + 1000 * rank + variant)
    lengths = lengths[torch.randperm(B, generator=gr)]
    T = int(lengths.max())
    xs = [torch.randn(B, T, d, generator=gr) for d in dims]
    y = (torch.rand(B, T, generator=gr) < 0.07).float()
    crf = arch.lower().endswith("crf")
    for b, n in enumerate(lengths.tolist()):
        for x in xs:
            x[b, n:] = 0
        y[b, n - 1] = 0
        y[b, n:] = 0 if crf else -1
    return {"src_tokens": xs[0], "src_tokens2": xs[1] if len(xs) > 1 else None, "src_lengths": lengths, "tgt_tokens": y,
            "id": torch.arange(B), "domain": None}


def train_leg(ctx, key, steps):
    from multimodaltopicsegmentation_b200 import dist as mdist

    m, dev = ctx.m, ctx.dev
    arch, B, _, dims, workload = TRAIN_LEGS[key]
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, list(dims) if len(dims) > 1 else dims[0], CFG["H"], num_layers=CFG["L"], architecture=arch,
                          loss_fn="FocalLoss", optimizer="Adam", lr=1e-3).to(dev)
    opt = seg.configure_optimizers()["optimizer"]
    bucket = mdist.GradBucket(seg.parameters())
    batches = [m.to_device(train_batch(key, ctx.rank, i), dev) for i in range(2)]
    n_sent = sum(int(b["src_lengths"].sum()) for b in batches) / len(batches)
    last = {}

    def step(i):
        last["loss"] = mdist.train_step(seg, batches[i % 2], opt, bucket)

    ms, launches = ctx.timed(step, steps)
    return {"metric": "training episodes/sec", "value": B * ctx.world / (ms / 1e3), "unit": "episodes/s",
            "ms_per_step": ms, "steps": steps, "workload": workload, "per_gpu_batch": B,
            "sentences_per_step_per_gpu": n_sent, "gpu_launches_per_step": launches, "grad_bucket_bytes": bucket.nbytes,
            "collective": "one NCCL all_reduce(SUM) over the flat gradient bucket + its count slot per step, no host sync"
                          if ctx.world > 1 else "none (single GPU)",
            "last_loss": float(last["loss"].detach())}


def cpu_train_reference(key):
    from oracle import ref_torch as rt

    use_all_host_threads()
    arch, B, _, dims, _ = TRAIN_LEGS[key]
    torch.manual_seed(0)
    H, L = CFG["H"], CFG["L"]
    if arch == "BiLSTM":
        model = rt.Segmenter(2, dims[0], H, num_layers=L, loss_fn="FocalLoss")
        loss_of = lambda b: model.loss(b["src_tokens"], b["src_lengths"], b["tgt_tokens"])  # noqa: E731
    elif arch == "biLSTMCRF":
        model = rt.EncoderCRF(2, dims[0], H, num_layers=L)
        loss_of = lambda b: model.loss(b["src_tokens"], b["src_lengths"], b["tgt_tokens"])  # noqa: E731
    elif arch == "BiLSTMLateFusion":
        model = rt.LateFusion(2, list(dims), H, num_layers=L, loss_fn="FocalLoss")
        loss_of = lambda b: model.loss(b["src_tokens"], b["src_tokens2"], b["src_lengths"], b["tgt_tokens"])  # noqa: E731
    else:
        enc = rt.LateFusion(2, list(dims), H, num_layers=L, loss_fn="FocalLoss")
        crf = rt.ChainCRF(4 * H, 2)
        model = torch.nn.ModuleList([enc.model1, enc.model2, crf])
        loss_of = lambda b: crf.loss(enc._features(b["src_tokens"], b["src_tokens2"], b["src_lengths"]), b["tgt_tokens"],  # noqa: E731
                                     rt.length_mask(b["src_tokens"].shape[1], b["src_lengths"]))
    opt = torch.optim.Adam(model.parameters(), eps=1e-7, lr=1e-3)
    batch = train_batch(key, 0, 0)
    times = []
    n_steps = 2 if batch["src_tokens"].shape[1] > 1000 else 3   # a configs[1] step takes tens of seconds on the host
    for i in range(n_steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = loss_of(batch)
        loss.backward()
        opt.step()
        times.append(time.perf_counter() - t0)
    best = min(times[1:])
    return {"value": B / best, "unit": "episodes/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"best of {n_steps - 1} step(s) (after 1 warm-up) on one batch of {B} episodes, oracle/ref_torch.py on host cores"}


# ----------------------------------------------------------------------------------------------------------------
# configs[2]: windowed-attention segmenter
# ----------------------------------------------------------------------------------------------------------------
XF_CFG = dict(B=256, S=960, D=896, F=256, L=6, heads=8, window=16)
XF_WORKLOAD = ("configs[2]: RestrictedTransformer (pyramidal windowed attention, 6 layers, window 16 -> reaches 48..8, 8 heads, "
               "d 896, FFN 256) inference, 256 episodes x 960 sentences (960 not 1000: HF needs S % lcm(windows) == 0), "
               "lengths 100..960")
XF_ATTN_BYTES_PER_TOKEN = 16 * 896   # SURVEY.md section 8(d): read q,k,v + write o, fp32
XF_GEMM_FLOPS_PER_TOKEN = 2 * 896 * (3 * 896 + 896 + 256 + 256)  # qkv + out-proj + FFN1 + FFN2 per layer


def xf_batch(seed, B):
    c = XF_CFG
    g = torch.Generator().manual_seed(777 + seed)
    lengths = torch.randint(100, c["S"] + 1, (B,), generator=g)
    lengths[0] = c["S"]
    return lengths


def transformer_leg(ctx, steps):
    """cfg3: windowed-attention segmenter inference.  Device-resident value, e2e from pinned host memory, per-kernel
    CUDA-event times, roofline fractions of the banded-attention kernel (HBM) and the dense layers (tensor)."""
    from multimodaltopicsegmentation_b200 import ops

    m, dev = ctx.m, ctx.dev
    c = XF_CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D"], c["F"], num_layers=c["L"], architecture="Transformer", loss_fn="FocalLoss",
                          nheads=c["heads"], attention_window=c["window"], threshold=0.5).to(dev).eval()
    seg.model.th = 0.5
    model = seg.model
    lengths = xf_batch(0, c["B"])   # the same length multiset on every rank (weak scaling), different embeddings
    n_sent = int(lengths.sum())
    g = torch.Generator(device=dev).manual_seed(5 + ctx.rank)
    xs = [torch.randn(c["B"], c["S"], c["D"], device=dev, generator=g) for _ in range(2)]  # 2 x 881 MB >> L2
    lens = ops.Lengths(lengths, dev, c["S"])

    def step(i):
        with torch.no_grad():
            return model.decode_device(xs[i % 2], lens)

    ms, launches = ctx.timed(step, steps)
    prof = ctx.profile(step)
    # e2e: host (pinned) embeddings in, host tag lists out
    host = xs[0].cpu().pin_memory()
    prefetcher = m.DevicePrefetcher(None, dev)   # one set of staging buffers for all passes, as over epochs

    def e2e(n):
        batches = ({"src_tokens": host, "src_lengths": lengths} for _ in range(n))
        for _ in seg.predict_batches(prefetcher.iterate(batches)):
            pass

    e2e(2)
    ctx.barrier()
    t0 = time.perf_counter()
    n_e2e = max(4, 2 * steps)   # the first copy of a pass cannot overlap anything: enough steps to amortise it
    e2e(n_e2e)
    ctx.barrier()
    e2e_s = ctx.max_over_ranks((time.perf_counter() - t0) / n_e2e)
    hbm_peak, _ = peaks()
    tokens = c["B"] * c["S"]
    attn = prof.get("mts_band_attn_fwd", [])
    gemm = prof.get("mts_gemm_tf32x3", []) + prof.get("mts_gemm_tf32x3_gelu_pair", []) + prof.get("mts_gemm_f16x3", [])
    out = {"metric": "segmented sentences/sec", "value": n_sent * ctx.world / (ms / 1e3), "unit": "sentences/s",
           "ms_per_step": ms, "steps": steps, "workload": XF_WORKLOAD, "valid_sentences_per_step_per_gpu": n_sent,
           "tokens_per_step_per_gpu": tokens, "gpu_launches_per_step": launches,
           "e2e": {"value": n_sent * ctx.world / e2e_s, "unit": "sentences/s", "h2d_bytes_per_step": host.numel() * 4,
                   "d2h_bytes_per_step": tokens,
                   "api": "DevicePrefetcher -> TextSegmenter.predict_batches, pinned host tensors in, host tag lists out"},
           "kernel_ms_per_step": {k: sum(v) for k, v in prof.items()},
           "kernel_calls_per_step": {k: len(v) for k, v in prof.items()}}
    if attn:
        per_layer = [n_sent * XF_ATTN_BYTES_PER_TOKEN / (x / 1e3) / 1e9 for x in attn]
        out["roofline_attention"] = {"kernel": "banded attention forward, per layer (reach 48,40,32,24,16,8)", "bound": "hbm",
                                     "achieved_gbs_per_layer": per_layer, "peak": hbm_peak,
                                     "frac_per_layer": [a / hbm_peak for a in per_layer],
                                     "algorithmic_bytes_per_launch": n_sent * XF_ATTN_BYTES_PER_TOKEN,
                                     "ms_per_layer": attn}
    if gemm:
        from multimodaltopicsegmentation_b200 import transformer as xf

        rows = n_sent if xf.LAYOUT == "ragged" else tokens   # the dense layers only see the valid sentences
        tf = rows * XF_GEMM_FLOPS_PER_TOKEN * c["L"] / (sum(gemm) / 1e3) / 1e12
        out["roofline_dense"] = {"kernel": "gemm_tf32x3_2sm_kernel (out-proj, output dense: TF32 + bf16 correction) and the same kernel "
                                           "in its fp16-split mode (q/k/v, intermediate dense: three kind::f16 products)", "bound": "tensor",
                                 "rows_per_launch": rows, "token_layout": xf.LAYOUT, "launches": len(gemm),
                                 "achieved_tflops_fp32_equiv": tf,
                                 "ms_by_entry": {k: sum(prof[k]) for k in ("mts_gemm_f16x3", "mts_gemm_tf32x3", "mts_gemm_tf32x3_gelu_pair")
                                                 if k in prof},
                                 "note": "fp32-grade products on the tensor cores: TF32 + one bf16 correction product (2 MMA streams "
                                         "per product, K = 8 / 16) or three fp16 products over split operands (K = 16 each)"}
    return out


def cpu_transformer_reference():
    from oracle import ref_torch as rt

    use_all_host_threads()
    c = XF_CFG
    torch.manual_seed(0)
    model = rt.WindowedSegmenter(2, c["D"], c["F"], num_layers=c["L"], nheads=c["heads"], loss_fn="FocalLoss",
                                 threshold=0.5, window_size=c["window"]).eval()
    B = 4
    lengths = xf_batch(0, B)
    x = torch.randn(B, c["S"], c["D"])
    with torch.no_grad():
        model(x, lengths)
        t0 = time.perf_counter()
        model(x, lengths)
        dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    mask = rt.reference_mask_loop(c["S"], lengths)   # the reference's host-side mask construction, timed on its own
    dt_mask = time.perf_counter() - t0
    assert torch.equal(mask.bool(), rt.length_mask(c["S"], lengths))
    n = int(lengths.sum())
    return {"value": n / dt, "value_incl_mask_loop": n / (dt + dt_mask), "mask_loop_ms_per_episode": dt_mask / B * 1e3,
            "unit": "sentences/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "1 batch of 4 episodes x 960 sentences (after 1 warm-up) through oracle/ref_torch.py (HF "
                      "LongformerModel on host cores); `value` excludes, `value_incl_mask_loop` includes the reference's "
                      "Python mask loop (RestrictedTransformerLayer.py:101-116)"}


# ----------------------------------------------------------------------------------------------------------------
# configs[4]: 8192-sentence episodes
# ----------------------------------------------------------------------------------------------------------------
LONG_CFG = dict(B=8, T=8192, D=1024)
LONG_WORKLOAD = ("configs[4]: long-episode BiLSTM inference, 8 episodes x 8192 sentences per GPU, 1024-d fused embeddings, "
                 "H256 x 2 layers, episodes sharded over the GPUs (no data-path collective)")


def long_leg(ctx, steps):
    from multimodaltopicsegmentation_b200 import ops

    m, dev = ctx.m, ctx.dev
    c = LONG_CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D"], CFG["H"], num_layers=CFG["L"], architecture="BiLSTM", loss_fn="FocalLoss",
                          threshold=0.5).to(dev).eval()
    seg.model.th = 0.5
    model = seg.model
    g = torch.Generator(device=dev).manual_seed(50 + ctx.rank)
    xs = [torch.randn(c["B"], c["T"], c["D"], device=dev, generator=g) for _ in range(2)]   # 2 x 268 MB > L2
    lengths = torch.full((c["B"],), c["T"], dtype=torch.long)
    lens = ops.Lengths(lengths, dev, c["T"])
    n_sent = c["B"] * c["T"]

    def step(i):
        return model.decode_device(xs[i % 2], lens)

    ms, launches = ctx.timed(step, steps)
    prof = ctx.profile(step)
    host = xs[0].cpu().pin_memory()
    prefetcher = m.DevicePrefetcher(None, dev)

    def e2e(n):
        batches = ({"src_tokens": host, "src_lengths": lengths} for _ in range(n))
        for _ in seg.predict_batches(prefetcher.iterate(batches)):
            pass

    e2e(2)
    ctx.barrier()
    t0 = time.perf_counter()
    n_e2e = max(4, steps)
    e2e(n_e2e)
    ctx.barrier()
    e2e_s = ctx.max_over_ranks((time.perf_counter() - t0) / n_e2e)
    return {"metric": "segmented sentences/sec", "value": n_sent * ctx.world / (ms / 1e3), "unit": "sentences/s",
            "ms_per_step": ms, "steps": steps, "workload": LONG_WORKLOAD, "gpu_launches_per_step": launches,
            "e2e": {"value": n_sent * ctx.world / e2e_s, "unit": "sentences/s", "h2d_bytes_per_step": host.numel() * 4,
                    "d2h_bytes_per_step": n_sent},
            "roofline": rec_roofline(prof, n_sent, "8 episodes x 2 directions = 16 sequences in flight, 8192 serial steps: "
                                                   "the step latency, not the bytes, bounds this shape"),
            "kernel_ms_per_step": {k: sum(v) for k, v in prof.items()}}


def cpu_long_reference():
    from oracle import ref_torch as rt

    use_all_host_threads()
    c = LONG_CFG
    torch.manual_seed(0)
    model = rt.Segmenter(2, c["D"], CFG["H"], num_layers=CFG["L"], loss_fn="FocalLoss", threshold=0.5)
    B = 2
    x = torch.randn(B, c["T"], c["D"])
    lengths = torch.full((B,), c["T"], dtype=torch.long)
    with torch.no_grad():
        model(x[:, :512], torch.full((B,), 512, dtype=torch.long))
        t0 = time.perf_counter()
        model(x, lengths)
        dt = time.perf_counter() - t0
    return {"value": B * c["T"] / dt, "unit": "sentences/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "1 batch of 2 episodes x 8192 sentences x 1024-d through oracle/ref_torch.py on host cores"}


# ----------------------------------------------------------------------------------------------------------------
# BiLSTM + CRF decode at the headline shape, and the CRF kernels on their own
# ----------------------------------------------------------------------------------------------------------------
CRF_BYTES = {"mts_crf_viterbi": 16 + 4,        # emissions in (C = 4 fp32), int32 path out
             "mts_crf_nll_fwd": 16 + 4 + 16,   # emissions + float tag in, saved alphas out (training)
             "mts_crf_nll_bwd": 16 + 4 + 16 + 16}   # emissions, tag, alphas in; d emissions out


def crf_leg(ctx, steps):
    """(1) the north_star model "early-fusion BiLSTM + CRF" decoding the headline batch (Viterbi instead of the threshold);
    (2) the CRF kernels alone at 64 x 300 and 8 x 8192: time per launch and algorithmic HBM fraction."""
    from multimodaltopicsegmentation_b200 import ops

    m, dev = ctx.m, ctx.dev
    c = CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], architecture="biLSTMCRF").to(dev).eval()
    sets = []
    for i in range(4):
        a, b, l = synth(300 + 100 * ctx.rank + i, c["B"], c["T"], c["D1"], c["D2"])
        sets.append((a.to(dev), b.to(dev), ops.Lengths(l, dev, c["T"])))
    n_sent = c["B"] * c["T"]

    def step(i):
        a, b, lens = sets[i % 4]
        return seg.model.decode_device((a, b), lens)

    ms, launches = ctx.timed(step, steps, warm=3)
    out = {"bilstm_crf_decode": {"metric": "segmented sentences/sec", "value": n_sent * ctx.world / (ms / 1e3), "unit": "sentences/s",
                                 "ms_per_step": ms, "gpu_launches_per_step": launches,
                                 "workload": "early-fusion BiLSTM -> CRF Viterbi decode, 64 episodes x 300 sentences (the headline "
                                             "batch with the CRF output layer), eager launches"}}
    hbm_peak, _ = peaks()
    kern = {}
    crf = seg.model.crf
    for (B, T) in ((64, 300), (8, 8192), (4096, 300)):
        g = torch.Generator(device=dev).manual_seed(B + T)
        emis = torch.randn(B, T, 4, device=dev, generator=g, requires_grad=True)
        tags = (torch.rand(B, T, device=dev, generator=g) < 0.07).float()
        lens = ops.Lengths([T] * B, dev, T)

        def kstep(i):
            ops.crf_viterbi(emis.detach(), lens, crf.transitions)
            stats = ops.CrfNllFn.apply(emis, crf.transitions, tags, lens)
            (stats[0] - stats[1]).mean().backward()

        kstep(0)
        prof = ctx.profile(kstep, n=3)
        rec = {}
        for name, per in CRF_BYTES.items():
            t = statistics.median(prof[name])
            gbs = B * T * per / (t / 1e3) / 1e9
            rec[name] = {"ms": t, "algorithmic_bytes": B * T * per, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak}
        kern[f"{B}x{T}"] = rec
    out["kernels"] = kern
    out["note"] = ("warp-per-episode scans: T serial steps per episode, B episodes in flight -- 64 or 8 warps cannot load the "
                   "memory system (SURVEY.md section 8d: ~9.5 k episodes fill the machine); the 4096 x 300 row shows the same kernels with the machine filled")
    return out


def cpu_crf_reference():
    from oracle import ref_torch as rt

    use_all_host_threads()
    torch.manual_seed(0)
    crf = rt.ChainCRF(512, 2)
    out = {}
    for (B, T) in ((64, 300), (8, 8192)):
        feats = torch.randn(B, T, 512)
        tags = (torch.rand(B, T) < 0.07).long()
        mask = torch.ones(B, T)
        with torch.no_grad():
            t0 = time.perf_counter()
            crf(feats, mask)
            dt_v = time.perf_counter() - t0
        t0 = time.perf_counter()
        crf.loss(feats, tags, mask).backward()
        dt_n = time.perf_counter() - t0
        out[f"{B}x{T}"] = {"viterbi_ms": dt_v * 1e3, "nll_fwd_bwd_ms": dt_n * 1e3}
    return {"value": out, "unit": "ms", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "one call each of ChainCRF.forward (fc + Viterbi + host back-trace) and ChainCRF.loss + backward, oracle/ref_torch.py"}


# ----------------------------------------------------------------------------------------------------------------
# where the recurrence's HBM fraction saturates (SURVEY.md section 8d asks for the sweep), N = 1 only
# ----------------------------------------------------------------------------------------------------------------
def saturating_leg(ctx):
    from multimodaltopicsegmentation_b200 import ops

    dev = ctx.dev
    H, T = CFG["H"], CFG["T"]
    hbm_peak, _ = peaks()
    whh = torch.randn((1, 2, 4 * H, H), device=dev) * 0.06
    rows = []
    for B in (64, 256, 1024, 4096):
        gx = torch.randn((1, B * T, 8 * H), device=dev)
        lens = ops.Lengths([T] * B, dev, T)
        y = torch.empty((B, T, 2 * H), device=dev)

        def step(i):
            ops._call("mts_lstm_rec_fwd_tc", gx.data_ptr(), whh.data_ptr(), lens.dev.data_ptr(), lens.order.data_ptr(), 1, B, T, H,
                      y.data_ptr(), 0, 0, ops._stream())

        step(0)
        prof = ctx.profile(step, n=3)
        ms = statistics.median(prof["mts_lstm_rec_fwd_tc"])
        gbs = B * T * ALGO_BYTES_PER_SENTENCE_REC / (ms / 1e3) / 1e9
        rows.append({"B": B, "ms": ms, "achieved_gbs": gbs, "frac": gbs / hbm_peak})
        del gx, y
    best = max(rows, key=lambda r: r["frac"])
    return {"B": best["B"], "frac": best["frac"], "achieved": best["achieved_gbs"], "sweep": rows,
            "shape": f"B episodes x {T} sentences, one layer, both directions, inference",
            "kernel": "lstm_fwd_h3_kernel while every tile has a cluster of its own (B <= 112 here), lstm_fwd_h3p_kernel (CTA pairs share "
                      "the h tile: half the DSMEM bytes per CTA) beyond"}


def bf16_leg(ctx, steps):
    """The headline batch through the explicit bf16 switch (ops.set_precision("bf16")): bf16 x bf16 products in the input
    projections and the recurrence (fp32 state, gates, accumulation, outputs), embeddings stored and shipped as bf16.  Reported
    BESIDE the f32 headline, never instead of it; tolerances in DESIGN.md, measured by tests/test_gpu_config_shapes.py."""
    from multimodaltopicsegmentation_b200 import ops

    m, dev = ctx.m, ctx.dev
    c = CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], architecture="BiLSTM", loss_fn="FocalLoss",
                          threshold=0.5).to(dev)
    seg.model.th = 0.5
    model = seg.model
    n_sets = 4
    host = [synth(500 + 100 * ctx.rank + i, c["B"], c["T"], c["D1"], c["D2"]) for i in range(n_sets)]
    pinned = [(a.to(torch.bfloat16).pin_memory(), b.to(torch.bfloat16).pin_memory(), l) for a, b, l in host]
    dev_sets = [(a.to(dev), b.to(dev), ops.Lengths(l, dev, c["T"])) for a, b, l in pinned]
    n_sent = c["B"] * c["T"]
    ops.set_precision("bf16")
    try:
        def step(i):
            x1, x2, lens = dev_sets[i % n_sets]
            return model.decode_device((x1, x2), lens)

        ms, launches = ctx.timed(step, steps, warm=3)
        prof = ctx.profile(step, n=4)
        prefetcher = m.DevicePrefetcher(None, dev)

        def batches(n):
            for i in range(n):
                a, b, l = pinned[i % n_sets]
                yield {"src_tokens": (a, b), "src_lengths": l}

        def e2e(n):
            for _ in seg.predict_batches(prefetcher.iterate(batches(n))):
                pass

        e2e(4)
        ctx.barrier()
        t0 = time.perf_counter()
        e2e(steps)
        ctx.barrier()
        e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    finally:
        ops.set_precision("f32")
    h2d = c["B"] * c["T"] * (c["D1"] + c["D2"]) * 2 + c["B"] * 8
    rec = "mts_lstm_rec_fwd_tc_bf16"
    return {"metric": "segmented sentences/sec", "dtype": "bf16", "value": n_sent * ctx.world / (ms / 1e3), "unit": "sentences/s",
            "ms_per_step": ms, "gpu_launches_per_step": launches, "workload": WORKLOAD + " -- bf16 path, bf16 embeddings, eager launches",
            "e2e": {"value": n_sent * steps * ctx.world / e2e_s, "unit": "sentences/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": c["B"] * c["T"]},
            "kernel_ms_per_call": {k: sum(v) / len(v) for k, v in prof.items()},
            "roofline": {"kernel": "lstm_fwd_tc_kernel, bf16 mode (32 MMAs per step)", "bound": "hbm",
                         "achieved": n_sent * ALGO_BYTES_PER_SENTENCE_REC / (sum(prof[rec]) / len(prof[rec]) / 1e3) / 1e9 if rec in prof else None,
                         "peak": peaks()[0], "unit": "GB/s",
                         "note": "gx and h stay fp32 in HBM: same algorithmic bytes as the f32 path, shorter step"},
            "tolerance": "logits within 2e-2 of the logit scale of the fp32 oracle (measured 5e-3), boundary flips <= 0.5 % (measured 0.1 %) (tests/test_gpu_config_shapes.py::"
                         "test_bf16_path_tolerance_and_flips prints the measured values)"}


def library_gpu_info(ctx):
    """Information only (VERDICT r01 item 14): what torch's own GPU libraries (cuDNN RNN, cuBLAS; TF32 off) need for the
    headline batch and for the configs[1] training step on this same GPU.  Not a contract arm."""
    from oracle import ref_torch as rt

    dev = ctx.dev
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    c = CFG
    out = {}
    try:
        torch.manual_seed(0)
        model = rt.Segmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], loss_fn="FocalLoss", threshold=0.5).to(dev)
        x1, x2, lengths = synth(0, c["B"], c["T"], c["D1"], c["D2"])
        x = torch.cat([x1, x2], -1).to(dev)
        with torch.no_grad():
            for _ in range(3):
                model.classification(model.model(x, lengths))
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(10):
                model.classification(model.model(x, lengths))
            e.record()
            torch.cuda.synchronize()
        out["cfg1_inference_ms"] = s.elapsed_time(e) / 10
        batch = train_batch("train", 0, 0)
        xb, yb, lb = batch["src_tokens"].to(dev), batch["tgt_tokens"].to(dev), batch["src_lengths"]
        opt = torch.optim.Adam(model.parameters(), eps=1e-7, lr=1e-3)

        def tstep():
            opt.zero_grad()
            model.loss(xb, lb, yb).backward()
            opt.step()

        for _ in range(2):
            tstep()
        torch.cuda.synchronize()
        s.record()
        for _ in range(5):
            tstep()
        e.record()
        torch.cuda.synchronize()
        out["cfg2_train_step_ms"] = s.elapsed_time(e) / 5
        out["what"] = ("oracle/ref_torch.py Segmenter on cuda:0 = torch nn.LSTM (cuDNN, packed sequences) + cuBLAS, TF32 "
                       "disabled, logits only (no host decode); information, not a contract arm")
    except Exception as exc:
        out["error"] = f"{type(exc).__name__}: {exc}"
    return out


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist

    import multimodaltopicsegmentation_b200 as m
    from multimodaltopicsegmentation_b200 import dist as mdist
    from multimodaltopicsegmentation_b200 import ops

    global _AFFINITY0
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    ops.device_ok()
    ctx = Ctx(m, dev, rank, world, local_rank)
    legs = set(args.legs.split(",")) if args.legs != "all" else {"train", "train_crf", "latefusion", "long", "crf", "transformer",
                                                                 "saturating", "library", "bf16"}
    if args.skip_transformer:
        legs.discard("transformer")
    try:
        _AFFINITY0 = os.sched_getaffinity(0)
    except AttributeError:
        _AFFINITY0 = None
    # host buffers of a rank should live on the NUMA node its GPU hangs off (8 ranks reading pinned memory of ONE node
    # capped the round-1 e2e scaling); restored before the CPU legs
    numa = mdist.bind_to_gpu_numa_node(local_rank) if world > 1 else None
    c = CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], architecture="BiLSTM", loss_fn="FocalLoss",
                          threshold=0.5).to(dev)
    seg.model.th = 0.5
    model = seg.model
    # 4 rotating input sets so that consecutive steps do not find their inputs in L2 (4 x 68.8 MB > 126 MB)
    n_sets = 4
    host_sets = [synth(100 * rank + i, c["B"], c["T"], c["D1"], c["D2"]) for i in range(n_sets)]
    pinned = [(a.pin_memory(), b.pin_memory(), l) for a, b, l in host_sets]
    dev_sets = [(a.to(dev), b.to(dev), ops.Lengths(l, dev, c["T"])) for a, b, l in host_sets]
    n_sent_step = int(host_sets[0][2].sum())
    barrier = ctx.barrier

    def device_step(i):
        x1, x2, lens = dev_sets[i % n_sets]
        with torch.no_grad():
            feats = model.model((x1, x2), lens)
            return ops.head_decode(feats, model.classification.weight, model.classification.bias, lens, 0.5)

    def host_batches(n):  # what a DataLoader(pin_memory=True) over the collater yields
        for i in range(n):
            a, b, l = pinned[i % n_sets]
            yield {"src_tokens": (a, b), "src_lengths": l}

    prefetcher = m.DevicePrefetcher(None, dev)

    def e2e_run(n, batches=host_batches):
        # public API: DevicePrefetcher (H2D of batch i+1 on a side stream) + TextSegmenter.predict_batches, which yields
        # predict_step's host lists for every batch -- so every step includes its H2D copies and the D2H of its tags
        out = None
        for out in seg.predict_batches(prefetcher.iterate(batches(n))):
            pass
        return out

    # ---- device-resident timing ------------------------------------------------------------------------
    for i in range(args.warmup):
        device_step(i)
    barrier()
    # The launches of a step are captured into one CUDA graph per rotating input set, so that the step is not paced by
    # the host's launch path.  The step holds no collective (episodes are sharded; the only exchange is ONE gather of the
    # boundary predictions after the last step), so the same graphs serve every world size.
    ops.reset_launch_count()
    device_step(0)
    launches_per_step = ops.launch_count()   # counted on an eager step: graph replays launch exactly these kernels
    graphs = None
    eager = device_step
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            graphs, outs = [], []
            with torch.cuda.stream(side):
                for i in range(n_sets):
                    gph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gph, stream=side):
                        outs.append(eager(i))
                    graphs.append(gph)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()

            def device_step(i, _g=graphs, _o=outs):  # noqa: E306,F811
                _g[i % n_sets].replay()
                return _o[i % n_sets]
            for i in range(n_sets):
                device_step(i)
            torch.cuda.synchronize()
        except Exception as exc:  # capture not possible: keep the eager launches and say so
            print(f"[bench] CUDA-graph capture unavailable ({type(exc).__name__}: {exc}); timing eager launches", file=sys.stderr)
            graphs = None
            device_step = eager
    barrier()
    ops.reset_launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(local_rank)   # re-entered around every GPU-busy timed leg; the samples accumulate
    clk.__enter__()
    start.record()
    scores = tags = None
    for i in range(args.steps):
        scores, tags = device_step(i)
    if world > 1:  # inference needs only a final gather of the boundary predictions: once, after the last step
        gathered = mdist.gather_tags(tags)
    end.record()
    barrier()
    launches = ops.launch_count() if graphs is None else launches_per_step * args.steps
    ms = ctx.max_over_ranks(start.elapsed_time(end))
    if args.dump_outputs:
        if world > 1:   # every rank takes part in the gather, outside the timed region
            scores, tags = torch.cat(mdist.gather_tags(scores)), torch.cat(gathered)
        if rank == 0:
            dump_outputs(args.dump_outputs, scores, tags)

    # ---- per-kernel CUDA-event pass (roofline of the dominant kernel) ------------------------------------
    prof_lists = ctx.profile(eager, n=args.steps)
    prof = {k: sum(v) / len(v) for k, v in prof_lists.items()}
    calls = {k: len(v) // args.steps for k, v in prof_lists.items()}

    # ---- end to end through the reference-facing API, host buffers ---------------------------------------
    e2e_run(max(3, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    # the same loop with the split RESIDENT on the device (ResidentDataset: the embeddings were uploaded once, the
    # collater is a gather kernel): what a user gets who keeps the data set on the GPU -- no per-step H2D
    g = torch.Generator().manual_seed(4000 + rank)
    episodes = []
    for i in range(n_sets):
        a, b, l = host_sets[i]
        for e in range(c["B"]):
            episodes.append(((a[e], b[e]), torch.zeros(c["T"]), f"ep{i}_{e}"))
    resident = m.ResidentDataset(episodes, dev)
    del episodes

    def resident_batches(n):
        for i in range(n):
            s0 = (i % n_sets) * c["B"]
            yield resident.batch(range(s0, s0 + c["B"]))

    def e2e_resident(n):
        out = None
        for out in seg.predict_batches(resident_batches(n)):
            pass
        return out

    e2e_resident(3)
    barrier()
    t0 = time.perf_counter()
    e2e_resident(args.steps)
    barrier()
    e2e_res_s = ctx.max_over_ranks(time.perf_counter() - t0)
    clk.__exit__(None, None, None)
    del resident, dev_sets, pinned
    torch.cuda.empty_cache()

    total_sent = n_sent_step * args.steps * world
    results = {}
    heavy = max(3, args.steps // 2)
    with clk:
        if "train" in legs:
            results["train"] = train_leg(ctx, "train", heavy)
        if "train_crf" in legs:
            results["train_crf"] = train_leg(ctx, "train_crf", heavy)
        if "latefusion" in legs:
            for key in ("latefusion_train", "latefusion_train_b64", "latefusion_crf_train"):
                results[key] = train_leg(ctx, key, heavy)
        if "bf16" in legs:
            results["bf16"] = bf16_leg(ctx, args.steps)
        if "crf" in legs:
            results["crf"] = crf_leg(ctx, heavy)
        if "long" in legs:
            results["long_episode"] = long_leg(ctx, max(3, args.steps // 4))
        torch.cuda.empty_cache()
        if "transformer" in legs:
            results["transformer"] = transformer_leg(ctx, max(3, args.steps // 4))
        torch.cuda.empty_cache()
        if "saturating" in legs and world == 1:
            results["saturating"] = saturating_leg(ctx)

    if rank != 0:
        return
    cpu_val = cpu_ms = cores = None
    kind = "port"
    library = None
    if world == 1:
        if "library" in legs:
            library = library_gpu_info(ctx)
        for key in ("train", "train_crf", "latefusion_train", "latefusion_crf_train"):
            if key in results:
                results[key]["cpu_baseline"] = cpu_train_reference(key)
        if "transformer" in results:
            results["transformer"]["cpu_baseline"] = cpu_transformer_reference()
        if "long_episode" in results:
            results["long_episode"]["cpu_baseline"] = cpu_long_reference()
        if "crf" in results:
            results["crf"]["cpu_baseline"] = cpu_crf_reference()
        cpu_val, cpu_ms, cores, kind, what = cpu_reference(5, 1)
    value = total_sent / (ms / 1e3)
    roof = rec_roofline(prof_lists, n_sent_step,
                        "latency-bound at 64 episodes per GPU (T serial steps; per step: tcgen05 MMAs, DSMEM all-gather of h, "
                        "gate epilogue): see DESIGN.md section 4; `saturating` = the batch at which the fraction stops growing")
    roof["traffic"] = (NCU_REC_DRAM_BYTES if roof["kernel"].startswith("lstm_fwd_tc")
                       else NCU_REC_H3_DRAM_BYTES if roof["kernel"].startswith("lstm_fwd_h3") else None)
    roof["traffic_source"] = ("dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel at this shape, ncu --set full "
                              "(profiles/r01_ncu_summary.md for lstm_fwd_tc_kernel, profiles/r02_ncu_summary.md for lstm_fwd_h3_kernel)")
    if "saturating" in results:
        sat = results.pop("saturating")
        roof["saturating"] = sat
    h2d = c["B"] * c["T"] * (c["D1"] + c["D2"]) * 4 + c["B"] * 8
    d2h = c["B"] * c["T"]
    legs_short = {"e2e_resident_sps": total_sent / e2e_res_s}
    for key, short in (("train", "train_eps"), ("train_crf", "train_crf_eps"), ("latefusion_train", "latefusion_train_eps"),
                       ("latefusion_train_b64", "latefusion_train_b64_eps"), ("latefusion_crf_train", "latefusion_crf_train_eps"),
                       ("long_episode", "long_episode_sps"), ("transformer", "transformer_sps")):
        if key in results:
            legs_short[short] = results[key]["value"]
            if "e2e" in results[key]:
                legs_short[short.replace("_sps", "_e2e_sps")] = results[key]["e2e"]["value"]
    if "crf" in results:
        legs_short["bilstm_crf_decode_sps"] = results["crf"]["bilstm_crf_decode"]["value"]
    if "bf16" in results:
        legs_short["bf16_sps"] = results["bf16"]["value"]
        legs_short["bf16_e2e_sps"] = results["bf16"]["e2e"]["value"]
        if results["bf16"]["roofline"]["achieved"]:
            results["bf16"]["roofline"]["frac"] = results["bf16"]["roofline"]["achieved"] / results["bf16"]["roofline"]["peak"]
    line = {
        "metric": "segmented sentences/sec", "value": value, "unit": "sentences/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "per_gpu_batch": c["B"], "global_batch": c["B"] * world,
                   "l2": "4 rotating input sets (275 MB) exceed the 126 MB L2", "gemm": "tcgen05: layer-0 projection over fp16-split operands (3 kind::f16 products), layer 1 TF32 + bf16 correction",
                   "launch": f"one CUDA graph per input set ({launches_per_step} kernels)" if graphs is not None else "eager launches",
                   "recurrence": ("tcgen05 fp16-split operands (3 kind::f16 products), W_hh resident in TMEM" if roof["kernel"].startswith("lstm_fwd_h3")
                                  else "tcgen05 TF32 + bf16 correction, W_hh resident in TMEM" if roof["kernel"].startswith("lstm_fwd_tc") else "packed-fp32 FMA"),
                   "parallelism": (f"dp{world} (episodes sharded, no collective inside the step, ONE all_gather of the tags after "
                                   "the last step, inside the timed region)") if world > 1 else "single GPU",
                   "numa_node_of_rank0": numa},
        "e2e": {"value": total_sent / e2e_s, "unit": "sentences/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "h2d_gbs_aggregate": h2d * args.steps * world / e2e_s / 1e9,
                "api": "DevicePrefetcher (side-stream H2D of the next batch) -> TextSegmenter.predict_batches (the "
                       "trainer.predict loop over predict_step, device work of batch i+1 enqueued before the tags of batch i "
                       "are awaited), pinned host tensors in, host tag lists out",
                "resident": {"value": total_sent / e2e_res_s, "unit": "sentences/s", "h2d_bytes_per_step": c["B"] * 4,
                             "d2h_bytes_per_step": d2h,
                             "api": "ResidentDataset.batch (device-side collater over a split uploaded once) -> "
                                    "TextSegmenter.predict_batches, host tag lists out"}},
        "gpu_launches": launches,
        "roofline": roof,
        "legs": legs_short,
        "kernel_ms_per_call": prof, "kernel_calls_per_step": calls,
        "cpu_baseline": {"value": cpu_val, "unit": "sentences/s", "cores": cores, "kind": kind,
                         "sample": "5 full batches of 64x300 sentences on host cores, all torch threads" if cpu_val else
                                   "measured at N = 1 only"},
        "clocks": clk.summary(),
    }
    if library is not None:
        line["library_gpu_info"] = library
    line.update(results)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--legs", default="all", help="comma list of train,train_crf,latefusion,long,crf,transformer,saturating,library,bf16 "
                                                   "(the headline leg always runs); 'none' = headline only")
    ap.add_argument("--skip-transformer", action="store_true", help="skip the configs[2] windowed-attention leg")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the scores and tags of the last timed headline step to "
                                                           "DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
