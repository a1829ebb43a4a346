"""The windowed-attention segmenter at an early-fusion width: d = 1280 (768-d text + 512-d x-vectors), 8 heads of hd 160, at the
configs[2] geometry otherwise (256 episodes x 960 sentences, 6 layers, window 16, FFN 256); fp32 and the bf16 precision switch in
the same call.

  python tests/xf_wide_bench.py --steps 10 --warmup 3 --out profiles/<name>.json

* device-resident step time and sentences/s, the two precisions alternating step by step over two input sets (2 x 1.26 GB of fp32
  embeddings, 2 x 629 MB of bf16 ones: larger than the 126 MB L2); the bf16 leg reads bf16 embeddings;
* attention time per layer from CUDA events (separate, untimed pass) and its algorithmic bandwidth: q, k, v read and o written
  once per valid token (fp32: 16 d bytes; bf16: 6 d bytes in and 2 d bytes of packed operand out, 8 d) over the HBM data-sheet
  figure of 7.7 TB/s;
* the card's name and power limit (read-only query), written next to the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import XF_CFG, xf_batch  # noqa: E402

HBM_PEAK_GBS = 7700.0
CFG = dict(XF_CFG, D=1280)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"unknown ({torch.cuda.get_device_name(0)})"


def attn_bytes_per_token(prec, d):
    return {"f32": 16 * d, "bf16": 8 * d}[prec]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "xf_wide_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing is measured without one")
    import multimodaltopicsegmentation_b200 as m
    from multimodaltopicsegmentation_b200 import ops, transformer

    dev = torch.device("cuda:0")
    c = CFG
    assert transformer._bf16_eligible(c["D"], c["heads"]) is False   # the switch is off here
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
            assert transformer._bf16_eligible(c["D"], c["heads"]) == (prec == "bf16")
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

    res = {"card": card(), "workload": f"d 1280 (hd 160) at the configs[2] geometry {CFG}, {n_sent} valid sentences per step",
           "steps": a.steps, "warmup": a.warmup, "timing": "CUDA events around each device-resident step, f32 and bf16 alternating",
           "hbm_peak_gbs_datasheet": HBM_PEAK_GBS}
    attn_entry = {"f32": "mts_band_attn_fwd", "bf16": "mts_band_attn_fwd_bf16"}
    for prec in ("f32", "bf16"):
        ms = statistics.median(times[prec])
        tot, per_call = kernels(prec)
        attn = per_call.get(attn_entry[prec], [])
        nb = attn_bytes_per_token(prec, c["D"])
        res[prec] = {"ms_per_step_median": ms, "ms_per_step_all": times[prec], "sentences_per_s": n_sent / (ms / 1e3),
                     "kernel_ms_per_step": tot,
                     "kernel_groups_ms": {"attention": sum(attn),
                                          "gemm": sum(v for k, v in tot.items() if k.startswith("mts_gemm")),
                                          "layernorm": sum(v for k, v in tot.items() if "_ln_" in k)},
                     "attention_bytes_per_token": nb,
                     "attention_ms_per_layer": attn,
                     "attention_algorithmic_gbs_per_layer": [n_sent * nb / (t / 1e3) / 1e9 for t in attn],
                     "attention_frac_of_hbm_peak_per_layer": [n_sent * nb / (t / 1e3) / 1e9 / HBM_PEAK_GBS for t in attn]}
    res["bf16_speedup_device_resident"] = res["f32"]["ms_per_step_median"] / res["bf16"]["ms_per_step_median"]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    short = {k: res[k] for k in ("card", "bf16_speedup_device_resident")}
    for prec in ("f32", "bf16"):
        short[prec] = {k: res[prec][k] for k in ("ms_per_step_median", "sentences_per_s", "kernel_groups_ms", "attention_ms_per_layer",
                                                 "attention_frac_of_hbm_peak_per_layer")}
    print(json.dumps(short, indent=1))


if __name__ == "__main__":
    main()
