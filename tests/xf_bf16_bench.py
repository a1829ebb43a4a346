"""configs[2] (windowed-attention segmenter, bench.py's XF_CFG) in fp32 and under the bf16 precision switch, same card, same call.

  python tests/xf_bf16_bench.py --steps 10 --warmup 3 --out profiles/<name>.json

* device-resident step time and sentences/s, the two precisions alternating step by step over two input sets (2 x 881 MB of fp32
  embeddings, 2 x 440 MB of bf16 ones: larger than the 126 MB L2); the bf16 leg reads bf16 embeddings;
* per-kernel CUDA-event times of one step of each (separate, untimed pass): attention, GEMMs by entry, LayerNorm;
* the attention kernel's algorithmic bandwidth: q, k, v read and o written once per valid token (fp32: 16 d bytes, bf16: 8 d bytes
  in and the fp32-sized packed operand out -- counted as 8 d as the algorithm needs no more) over HBM peak (7.7 TB/s, data sheet);
* end to end from pinned host embeddings (fp32 / bf16) through DevicePrefetcher and TextSegmenter.predict_batches;
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

HBM_PEAK_GBS = 7700.0


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"unknown ({torch.cuda.get_device_name(0)})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "xf_bf16_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is measured without one")
    import multimodaltopicsegmentation_b200 as m
    from multimodaltopicsegmentation_b200 import ops

    dev = torch.device("cuda:0")
    c = XF_CFG
    torch.manual_seed(0)
    seg = m.TextSegmenter(2, c["D"], c["F"], num_layers=c["L"], architecture="Transformer", loss_fn="FocalLoss", nheads=c["heads"],
                          attention_window=c["window"], threshold=0.5).to(dev).eval()
    seg.model.th = 0.5
    model = seg.model
    lengths = xf_batch(0, c["B"])
    n_sent = int(lengths.sum())
    g = torch.Generator(device=dev).manual_seed(5)
    xs = {"f32": [torch.randn(c["B"], c["S"], c["D"], device=dev, generator=g) for _ in range(2)]}
    xs["bf16"] = [x.to(torch.bfloat16) for x in xs["f32"]]
    lens = ops.Lengths(lengths, dev, c["S"])

    def step(prec, i):
        ops.set_precision(prec)
        try:
            with torch.no_grad():
                return model.decode_device(xs[prec][i % 2], lens)
        finally:
            ops.set_precision("f32")

    for i in range(a.warmup):
        for prec in ("f32", "bf16"):
            step(prec, i)
    torch.cuda.synchronize()
    times = {"f32": [], "bf16": []}
    for i in range(a.steps):
        for prec in (("f32", "bf16") if i % 2 == 0 else ("bf16", "f32")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(prec, i)
            e1.record()
            e1.synchronize()
            times[prec].append(e0.elapsed_time(e1))

    def kernels(prec):
        ops.PROFILE = {}
        try:
            step(prec, 0)
            torch.cuda.synchronize()
            return {k: sum(s.elapsed_time(e) for s, e in v) for k, v in ops.PROFILE.items()}, \
                   {k: [s.elapsed_time(e) for s, e in v] for k, v in ops.PROFILE.items()}
        finally:
            ops.PROFILE = None

    res = {"card": card(), "workload": f"configs[2] XF_CFG {XF_CFG}, {n_sent} valid sentences per step",
           "steps": a.steps, "warmup": a.warmup, "timing": "CUDA events around each device-resident step, f32 and bf16 alternating"}
    attn_entry = {"f32": "mts_band_attn_fwd", "bf16": "mts_band_attn_fwd_bf16"}
    attn_bytes = {"f32": 16 * c["D"], "bf16": 8 * c["D"]}
    for prec in ("f32", "bf16"):
        ms = statistics.median(times[prec])
        tot, per_call = kernels(prec)
        attn = per_call.get(attn_entry[prec], [])
        res[prec] = {"ms_per_step_median": ms, "ms_per_step_all": times[prec], "sentences_per_s": n_sent / (ms / 1e3),
                     "kernel_ms_per_step": tot,
                     "kernel_groups_ms": {"attention": sum(attn),
                                          "gemm": sum(v for k, v in tot.items() if k.startswith("mts_gemm")),
                                          "layernorm": sum(v for k, v in tot.items() if "_ln_" in k)},
                     "attention_ms_per_layer": attn,
                     "attention_algorithmic_gbs_per_layer": [n_sent * attn_bytes[prec] / (t / 1e3) / 1e9 for t in attn],
                     "attention_frac_of_hbm_peak_per_layer": [n_sent * attn_bytes[prec] / (t / 1e3) / 1e9 / HBM_PEAK_GBS for t in attn]}
    # end to end: pinned host embeddings in, host tag lists out
    for prec in ("f32", "bf16"):
        host = xs[prec][0].cpu().pin_memory()
        prefetcher = m.DevicePrefetcher(None, dev)

        def e2e(n):
            batches = ({"src_tokens": host, "src_lengths": lengths} for _ in range(n))
            for _ in seg.predict_batches(prefetcher.iterate(batches)):
                pass

        ops.set_precision(prec)
        try:
            e2e(2)
            torch.cuda.synchronize()
            n = max(4, 2 * a.steps)
            t0 = time.perf_counter()
            e2e(n)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / n
        finally:
            ops.set_precision("f32")
        res[prec]["e2e"] = {"s_per_batch": dt, "sentences_per_s": n_sent / dt, "h2d_bytes_per_batch": host.numel() * host.element_size()}
        del host, prefetcher
    res["bf16_speedup_device_resident"] = res["f32"]["ms_per_step_median"] / res["bf16"]["ms_per_step_median"]
    res["bf16_speedup_e2e"] = res["bf16"]["e2e"]["sentences_per_s"] / res["f32"]["e2e"]["sentences_per_s"]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    short = {k: res[k] for k in ("card", "bf16_speedup_device_resident", "bf16_speedup_e2e")}
    for prec in ("f32", "bf16"):
        short[prec] = {k: res[prec][k] for k in ("ms_per_step_median", "sentences_per_s", "kernel_groups_ms")}
        short[prec]["e2e_sentences_per_s"] = res[prec]["e2e"]["sentences_per_s"]
        short[prec]["attention_frac_of_hbm_peak_per_layer"] = res[prec]["attention_frac_of_hbm_peak_per_layer"]
    print(json.dumps(short, indent=1))


if __name__ == "__main__":
    main()
