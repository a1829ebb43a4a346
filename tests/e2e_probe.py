import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multimodaltopicsegmentation_b200 as m
import bench
dev = torch.device('cuda:0')
c = bench.CFG
torch.manual_seed(0)
seg = m.TextSegmenter(2, c["D1"] + c["D2"], c["H"], num_layers=c["L"], architecture="BiLSTM", loss_fn="FocalLoss", threshold=0.5).to(dev)
seg.model.th = 0.5
host = [bench.synth(i, c["B"], c["T"], c["D1"], c["D2"]) for i in range(4)]
pinned = [(a.pin_memory(), b.pin_memory(), l) for a, b, l in host]
def batches(n):
    for i in range(n):
        a, b, l = pinned[i % 4]
        yield {"src_tokens": (a, b), "src_lengths": l}
def run_pref(n):
    for i, batch in enumerate(m.DevicePrefetcher(batches(n), dev)):
        seg.predict_step(batch, i)
def run_plain(n):
    for i, batch in enumerate(batches(n)):
        a, b = batch["src_tokens"]
        seg.predict_step({"src_tokens": (a.to(dev, non_blocking=True), b.to(dev, non_blocking=True)), "src_lengths": batch["src_lengths"]}, i)
for name, fn in (("plain", run_plain), ("prefetch", run_pref), ("plain", run_plain), ("prefetch", run_pref)):
    fn(4); torch.cuda.synchronize()
    t0 = time.perf_counter(); fn(20); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    print(f"{name}: {dt/20*1e3:.3f} ms/step  {19200*20/dt/1e6:.2f} M sentences/s")
# H2D alone
t0 = time.perf_counter()
for i in range(20):
    a, b, l = pinned[i % 4]; a.to(dev, non_blocking=True); b.to(dev, non_blocking=True)
torch.cuda.synchronize(); dt = time.perf_counter() - t0
print(f"H2D alone: {dt/20*1e3:.3f} ms/step ({68.8e6*20/dt/1e9:.1f} GB/s)")

# host-side cost of one predict_step with device-resident inputs (no H2D): where the CPU time goes
from multimodaltopicsegmentation_b200 import ops
a, b, l = host[0]
ad, bd = a.to(dev), b.to(dev)
batch = {"src_tokens": (ad, bd), "src_lengths": l}
for _ in range(5):
    seg.predict_step(batch, 0)
torch.cuda.synchronize()
N = 30
t0 = time.perf_counter()
for _ in range(N):
    ops.Lengths(l, dev, 300)
t_len = (time.perf_counter() - t0) / N
torch.cuda.synchronize()
lens = ops.Lengths(l, dev, 300)
model = seg.model
t0 = time.perf_counter()
for _ in range(N):
    with torch.no_grad():
        feats = model.model((ad, bd), lens)
        scores, tags = ops.head_decode(feats, model.classification.weight, model.classification.bias, lens, 0.5)
t_issue = (time.perf_counter() - t0) / N
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(N):
    out = seg.predict_step(batch, 0)
t_full = (time.perf_counter() - t0) / N
torch.cuda.synchronize()
from multimodaltopicsegmentation_b200 import modules
t0 = time.perf_counter()
for _ in range(N):
    modules._tags_to_lists(tags, lens, True)
t_lists = (time.perf_counter() - t0) / N
t_d2h = 0.0
print(f"Lengths() {t_len*1e3:.3f} ms | issue of the 6 launches (no sync) {t_issue*1e3:.3f} ms | tags D2H {t_d2h*1e3:.3f} ms | "
      f"lists {t_lists*1e3:.3f} ms | predict_step (sync) {t_full*1e3:.3f} ms")
