"""The windowed-attention segmenter fed an early-fusion pair (384-d text, 512-d audio) at the configs[2] geometry (256 episodes x
960 sentences, d 896, 6 layers, window 16, FFN 256): the pair read in place by the embeddings LayerNorm against a device torch.cat
followed by the single-source path, in fp32 and under the bf16 precision switch (bf16 embeddings), all four legs in one call.

  python tests/xf_pair_bench.py --steps 10 --warmup 3 --out profiles/<name>.json

* device-resident step time (CUDA events), the legs alternating step by step over two input sets (2 x 0.88 GB of fp32
  embeddings, 2 x 0.44 GB of bf16 ones: larger than the 126 MB L2); the cat leg's time includes its torch.cat;
* the embedding stage alone -- the embeddings-LayerNorm kernel, and for the cat leg the torch.cat before it -- over repeated
  launches, legs and input sets alternating (CUDA events; the inputs are larger than L2, so each launch reads HBM);
* per-kernel times of one step (CUDA events per ABI call, separate untimed pass);
* end to end: batches from two pinned host buffers (text, audio) through DevicePrefetcher into decode_device, host clock around
  the whole run ending in a device synchronise; the cat leg concatenates the staged pair on the device;
* pair and cat outputs compared bit for bit;
* the card's name and power limit (read-only query), written next to the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import XF_CFG, xf_batch  # noqa: E402

D1, D2 = 384, 512
LN_ENTRY = {("f32", "pair"): "mts_embed_ln_fwd_f16_pair", ("f32", "cat"): "mts_embed_ln_fwd_f16",
            ("bf16", "pair"): "mts_embed_ln_fwd_bf16in_pair", ("bf16", "cat"): "mts_embed_ln_fwd_bf16in"}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"unknown ({torch.cuda.get_device_name(0)})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-batches", type=int, default=8)
    ap.add_argument("--e2e-reps", type=int, default=5)
    ap.add_argument("--stage-reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "xf_pair_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is measured without one")
    import multimodaltopicsegmentation_b200 as m
    from multimodaltopicsegmentation_b200 import ops, transformer

    _p = ops._ptr
    dev = torch.device("cuda:0")
    c = XF_CFG
    assert c["D"] == D1 + D2
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D"], c["F"], num_layers=c["L"], architecture="Transformer", loss_fn="FocalLoss", nheads=c["heads"],
                          attention_window=c["window"], threshold=0.5).to(dev).eval()
    model = seg.model
    lengths = xf_batch(0, c["B"])
    n_sent = int(lengths.sum())
    lens = ops.Lengths(lengths, dev, c["S"])
    g = torch.Generator(device=dev).manual_seed(5)
    pairs = {"f32": [(torch.randn(c["B"], c["S"], D1, device=dev, generator=g), torch.randn(c["B"], c["S"], D2, device=dev, generator=g))
                     for _ in range(2)]}
    pairs["bf16"] = [tuple(t.to(torch.bfloat16) for t in p) for p in pairs["f32"]]

    def src(form, p):
        return p if form == "pair" else torch.cat(p, dim=-1)

    def run(prec, form, p, lengths_=lens):
        ops.set_precision(prec)
        try:
            assert transformer._bf16_eligible(c["D"], c["heads"]) == (prec == "bf16")
            with torch.no_grad():
                return model.decode_device(src(form, p), lengths_)
        finally:
            ops.set_precision("f32")

    legs = [(prec, form) for prec in ("f32", "bf16") for form in ("pair", "cat")]
    identical = {}
    for prec in ("f32", "bf16"):
        sp, tp, _ = run(prec, "pair", pairs[prec][0])
        sc, tc, _ = run(prec, "cat", pairs[prec][0])
        identical[prec] = bool(torch.equal(sp, sc) and torch.equal(tp, tc))
    for i in range(a.warmup):
        for leg in legs:
            run(*leg, pairs[leg[0]][i % 2])
    torch.cuda.synchronize()
    times = {leg: [] for leg in legs}
    for i in range(a.steps):
        for leg in (legs if i % 2 == 0 else legs[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(*leg, pairs[leg[0]][i % 2])
            e1.record()
            e1.synchronize()
            times[leg].append(e0.elapsed_time(e1))

    def kernels(prec, form):
        ops.PROFILE = {}
        try:
            run(prec, form, pairs[prec][0])
            torch.cuda.synchronize()
            return {k: sum(s.elapsed_time(e) for s, e in v) for k, v in ops.PROFILE.items()}
        finally:
            ops.PROFILE = None

    emb = model.model.model.embeddings
    pos, typ = emb.position_embeddings.weight.detach(), emb.token_type_embeddings.weight.detach()[0]
    gamma, beta = emb.LayerNorm.weight.detach(), emb.LayerNorm.bias.detach()

    def stage(prec, form, p):
        """The embeddings LayerNorm the step runs (ragged rows), preceded by the concatenation in the cat leg: (cat ms, LN ms)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        x1, x2 = (p[0], p[1]) if form == "pair" else (torch.cat(p, dim=-1), None)
        ev[1].record()
        B, S, d = c["B"], c["S"], c["D"]
        if prec == "f32":
            transformer._ln_f16(0, x1, pos, typ, gamma, beta, B, S, d, lens, a2=x2)
        else:
            y = torch.empty((lens.N, d), device=dev)
            y_lo = torch.empty((lens.N, d), device=dev)
            tail = (_p(pos), _p(typ), _p(gamma), _p(beta), B, S)
            outs = (transformer.LN_EPS, _p(y), _p(y_lo), d, _p(lens.dev), _p(lens.offs), ops._stream())
            if x2 is not None:
                ops._call("mts_embed_ln_fwd_bf16in_pair", _p(x1), x1.stride(0), D1, _p(x2), x2.stride(0), D2, *tail, *outs)
            else:
                ops._call("mts_embed_ln_fwd_bf16in", _p(x1), x1.stride(0), *tail, d, *outs)
        ev[2].record()
        ev[2].synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])

    for leg in legs:
        stage(*leg, pairs[leg[0]][0])
    stage_ms = {leg: [] for leg in legs}
    for i in range(a.stage_reps):
        for leg in (legs if i % 2 == 0 else legs[::-1]):
            stage_ms[leg].append(stage(*leg, pairs[leg[0]][i % 2]))

    # end to end from pinned host memory: two host input sets, alternating, through the side-stream prefetcher
    host = {prec: [{"src_tokens": tuple(t.cpu().pin_memory() for t in p), "src_lengths": lengths} for p in pairs[prec]]
            for prec in ("f32", "bf16")}

    def e2e(prec, form):
        batches = [host[prec][i % 2] for i in range(a.e2e_batches)]
        pf = m.DevicePrefetcher(batches, dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in pf:
            run(prec, form, b["src_tokens"], b["src_lengths"])
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    for leg in legs:
        e2e(*leg)   # warm-up: staging buffers, pinned-copy paths
    e2e_s = {leg: [] for leg in legs}
    for rep in range(a.e2e_reps):
        for leg in (legs if rep % 2 == 0 else legs[::-1]):
            e2e_s[leg].append(e2e(*leg))

    res = {"card": card(),
           "workload": f"configs[2] geometry {c} with the embeddings as a ({D1}, {D2}) pair, {n_sent} valid sentences per step",
           "steps": a.steps, "warmup": a.warmup,
           "timing": "CUDA events around each device-resident step, the four legs alternating; end to end: host clock around "
                     f"{a.e2e_batches} batches from pinned host memory through DevicePrefetcher, ending in a synchronise",
           "pair_equals_cat_bitwise": identical}
    for prec, form in legs:
        ms = statistics.median(times[(prec, form)])
        tot = kernels(prec, form)
        ln = LN_ENTRY[(prec, form)]
        e2e_med = statistics.median(e2e_s[(prec, form)])
        cat_t = [t[0] for t in stage_ms[(prec, form)]]
        ln_t = [t[1] for t in stage_ms[(prec, form)]]
        res[f"{prec}_{form}"] = {"ms_per_step_median": ms, "ms_per_step_all": times[(prec, form)],
                                 "sentences_per_s_device_resident": n_sent / (ms / 1e3),
                                 "embeddings_ln_entry": ln, "kernel_ms_per_step": tot,
                                 "stage_embeddings_ln_ms_median": statistics.median(ln_t),
                                 "stage_device_cat_ms_median": statistics.median(cat_t) if form == "cat" else 0.0,
                                 "stage_total_ms_median": statistics.median([x + y for x, y in stage_ms[(prec, form)]]),
                                 "stage_ms_all": stage_ms[(prec, form)],
                                 "e2e_s_all": e2e_s[(prec, form)],
                                 "e2e_sentences_per_s_median": a.e2e_batches * n_sent / e2e_med}
    for prec in ("f32", "bf16"):
        p, q = res[f"{prec}_pair"], res[f"{prec}_cat"]
        res[f"{prec}_cat_over_pair"] = {"step": q["ms_per_step_median"] / p["ms_per_step_median"],
                                        "embedding_stage": q["stage_total_ms_median"] / p["stage_total_ms_median"],
                                        "e2e": p["e2e_sentences_per_s_median"] / q["e2e_sentences_per_s_median"]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    short = {k: res[k] for k in ("card", "pair_equals_cat_bitwise", "f32_cat_over_pair", "bf16_cat_over_pair")}
    for prec, form in legs:
        r = res[f"{prec}_{form}"]
        short[f"{prec}_{form}"] = {k: r[k] for k in ("ms_per_step_median", "stage_embeddings_ln_ms_median", "stage_device_cat_ms_median",
                                                     "e2e_sentences_per_s_median")}
    print(json.dumps(short, indent=1))


if __name__ == "__main__":
    main()
