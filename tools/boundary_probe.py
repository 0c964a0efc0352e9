"""Marginal cost of one more dependent tensor-core launch: time CUDA graphs holding 1, 2, 4, 8, 16 copies of the same
layer (chained: copy i reads the output of copy i-1 when shapes allow, else the same input), each a separate launch
chained by programmatic dependent launch.  Slope = steady-state time per layer, intercept = graph launch overhead."""
import os

os.environ.setdefault("RTEN_B200_F32_MODE", "tf32")  # these tools measure the single-pass TF32 kernels unless told otherwise
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import rten_b200 as rt  # noqa: E402

torch.cuda.set_device(0)
stream = torch.cuda.Stream()
torch.cuda.set_stream(stream)
B = 32


def build(ctx, ci, co, k, hw):
    x = rt.from_torch(ctx, torch.randn(B, hw, hw, ci, device="cuda")).permute(0, 3, 1, 2)
    wt = ctx.to_device((np.random.randn(co, ci, k, k) / np.sqrt(ci * k * k)).astype(np.float32))
    bias = ctx.to_device(np.zeros(co, np.float32))
    op = rt.Conv(1, (1, 1), (k // 2,) * 4, (1, 1), activation=rt.ACT_RELU)
    pk = op.prepack(ctx, 1, wt)
    y0 = op.run(ctx, x, wt, bias, packed_w=pk)
    y1 = op.run(ctx, x, wt, bias, packed_w=pk)
    chain = ci == co

    def run(n):
        src = x
        for i in range(n):
            dst = y0 if i % 2 == 0 else y1
            op.run(ctx, src if chain else x, wt, bias, packed_w=pk, out=dst)
            src = dst
    return run


def time_graph(ctx, run, n, reps=30):
    run(n)
    ctx.sync()
    ctx.graph_begin()
    run(n)
    g = ctx.graph_end()
    for _ in range(3):
        g.launch()
    ctx.sync()
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        g.launch()
        e.record(stream)
        e.synchronize()
        ts.append(s.elapsed_time(e) * 1e3)
    return float(np.median(ts))


cases = [(64, 64, 3, 56), (128, 128, 3, 28), (256, 256, 3, 14), (512, 512, 3, 7), (64, 64, 1, 56), (256, 256, 1, 14)]
os.environ["RTEN_B200_NO_CTA2"] = "1"
ctx = rt.Context(0, stream=stream.cuda_stream)
ctx.set_autotune(True)
for (ci, co, k, hw) in cases:
    run = build(ctx, ci, co, k, hw)
    ns = [1, 2, 4, 8, 16]
    t = [time_graph(ctx, run, n) for n in ns]
    slope = (t[-1] - t[2]) / (ns[-1] - ns[2])
    print(f"single conv {k}x{k} {ci}->{co} @{hw}: " + " ".join(f"n={n}:{v:.1f}us" for n, v in zip(ns, t)) + f"  | marginal {slope:.2f} us/layer", flush=True)
