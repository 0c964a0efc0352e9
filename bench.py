#!/usr/bin/env python
"""bench.py -- one "step" = one pass of the hot path over one batch of synthetic input.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--model resnet50|bert|resnet50_int8|gpt2] [--dump-outputs DIR]

Default workload = BASELINE.json configs[1]: the post-fusion ResNet-50 fp32 op list, batch 32 per GPU.  Prints ONE
JSON line (rank 0).

  value     whole-job throughput, inputs resident in HBM, the step replayed from a CUDA graph, CUDA events on the
            launching stream, 256 MiB L2 flush between steps (outside the events), max over ranks.
  e2e       the same metric through the public operator API with HOST (pinned) input and output buffers, host<->device
            copies inside the timed region.
  modes     fp32 models are measured in BOTH arithmetic modes of the library: "tf32" (single tcgen05 kind::tf32 pass,
            an explicit opt-in) and "tf32x3" (the library default: error-compensated, meets the reference's own f32
            tolerance).  The top-level value / e2e / roofline are the tf32 block (north_star names the TF32 roofline);
            `modes.tf32x3` carries the same keys for the fp32-grade path.  Algorithmic flops are counted 1x in both.
  roofline  dominant kernel: algorithmic flops (or bytes) per step / that kernel's time inside the GRAPH replay (CUPTI
            kernel records through torch.profiler; `lower_bound` = the same work / the whole step time), against the
            tensor peak measured in this run (cuBLASLt 8192^3 through torch: burst = best of 10, sustained = 3 s).
  cpu_baseline / --impl reference: the CPU restatement of the reference path (oracle/; the Rust reference cannot be
            built here: no cargo) on the host cores, bounded sample.

--dump-outputs DIR writes, after the timed steps of each measured mode, what the last timed step returned (the logits, or
BERT's last hidden state; the all-gathered whole-job output at N > 1) as DIR/<output>_<mode>.npy in float32.  Inputs and
weights come from fixed seeds, so two builds run with the same arguments can be compared output for output (to the
rounding of the arithmetic mode: autotuned launch plans may differ from run to run).  The files stay within 64 MiB in
all: an output larger than its share is stored as a fixed, seeded sample of its flattened elements.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

MODELS = {
    "resnet50": dict(batch=32, unit="img/s", metric="resnet50_fp32_inferences_per_sec", modes=["tf32", "tf32x3"]),
    "bert": dict(batch=16, unit="seq/s", metric="bert_base_fp32_seq128_inferences_per_sec", modes=["tf32", "tf32x3"]),
    "resnet50_int8": dict(batch=64, unit="img/s", metric="resnet50_int8_inferences_per_sec", modes=["int8"]),
    "gpt2": dict(batch=8, unit="tokens/s", metric="gpt2_int8_decode_tokens_per_sec", modes=["int8"]),
}
GPT2_PREFILL, GPT2_CACHE = 512, 576
OUTPUT_NAME = {"resnet50": "logits", "resnet50_int8": "logits", "bert": "last_hidden_state", "gpt2": "logits"}
DUMP_BYTES = 64 << 20


def dump_output(dirname, name, a, budget):
    """DIR/<name>.npy in float32; above `budget` bytes, a fixed seeded sample of the flattened elements (ascending order)."""
    a = np.ascontiguousarray(a, np.float32)
    if a.nbytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(a.size, budget // a.itemsize, replace=False))
        a = a.reshape(-1)[idx]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"], "src": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and throttle reasons sampled every ~4 ms DURING a timed region through NVML."""

    def __init__(self, index: int):
        self.index, self.rows, self.stop_flag, self.thread = index, [], False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, mx, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        self.rows = []
        if self.nv is None:
            return
        self.stop_flag = False
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "NVML binding unavailable: clocks not sampled"}
        self.stop_flag = True
        self.thread.join(timeout=1)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        reasons = set()
        for _, _, rs in self.rows:
            for n, bit in names.items():
                if rs & bit:
                    reasons.add(n)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# workload definitions shared by both arms
# ------------------------------------------------------------------------------------------
def make_inputs(oracle, model, batch):
    rng = oracle.XorShiftRng(1234)
    if model in ("resnet50", "resnet50_int8"):
        return {"x": rng.uniform((batch, 3, 224, 224))}
    if model == "bert":
        ids = (rng.u64(batch * 128) % 30522).astype(np.int32).reshape(batch, 128)
        return {"ids": ids, "tt": np.zeros((batch, 128), np.int32), "mask": np.zeros((batch, 1, 1, 128), np.float32)}
    ids = (oracle.XorShiftRng(1).u64(batch * GPT2_CACHE) % 50257).astype(np.int32).reshape(batch, GPT2_CACHE)
    return {"ids": ids}


def make_spec(oracle, model):
    from rten_b200 import graphs
    rng = oracle.XorShiftRng(5678)
    if model == "resnet50":
        return graphs.make_resnet50(lambda s: rng.uniform(s))
    if model == "resnet50_int8":
        return graphs.quantize_resnet50(graphs.make_resnet50(lambda s: rng.uniform(s)))
    if model == "bert":
        return graphs.make_bert(lambda s: rng.uniform(s))
    return graphs.make_gpt2_int8(lambda s: rng.uniform(s))


def metric_name(model):
    return MODELS[model]["metric"]


def config_of(model, batch, n):
    common = {"global_batch": batch * n, "per_gpu_batch": batch, "l2": "256 MiB memset between timed steps",
              "f32_modes": "top level = tf32 (explicit opt-in, single kind::tf32 pass); modes.tf32x3 = library default (fp32-grade)"}
    if model == "resnet50":
        return {"workload": "ResNet-50 fp32 (post-fusion op list, BN folded), batch 32 per GPU, 224x224, synthetic weights XorShift(5678)",
                "parallelism": f"dp{n} (batch shard, all-gather of logits)", **common}
    if model == "bert":
        return {"workload": "BERT-base fp32 (post-fusion op list), batch 16 x seq 128 per GPU, synthetic weights XorShift(5678)",
                "seq_len": 128, "parallelism": f"dp{n} (batch shard, all-gather of hidden states)", **common}
    if model == "resnet50_int8":
        return {"workload": "ResNet-50 dynamically quantised (DynamicQuantizeLinear -> ConvIntegerToFloat), batch 64 per GPU, 224x224",
                "parallelism": f"dp{n} (batch shard; quantisation ranges all-reduced over the ranks, all-gather of logits)", **common}
    return {"workload": f"GPT-2 small int8 (dynamic quantisation), batch 8 per GPU: decode steps against a KV cache holding a {GPT2_PREFILL}-token prefill",
            "seq_len": GPT2_PREFILL, "parallelism": f"dp{n} (independent replicas per GPU, all-gather of logits)", **common}


def run_reference_arm(args, model, batch):
    """CPU restatement of the reference path on all host threads.  One step processes what ONE step of the GPU arm
    processes at this N (batch x N inputs), in chunks of one per-GPU batch, so the two arms are like for like."""
    from oracle import oracle
    import model_ref
    ncores = oracle.use_all_cores()
    spec = make_spec(oracle, model)
    n = max(1, args.gpus)
    unit = MODELS[model]["unit"]
    if model == "gpt2":
        # bounded sample: a 128-token prefill (untimed), then decode steps of 8 tokens; each step = N per-GPU batches
        inp = make_inputs(oracle, model, batch)["ids"]
        state = {"past": None}

        def prefill():
            return model_ref.gpt2_int8_decoder(oracle, spec, inp[:, :128])

        dec = prefill()
        pos = [128]

        def run():
            for _ in range(n):
                dec.step(inp[:, pos[0]:pos[0] + 1])
            pos[0] += 1

        per_step = batch * n
        sample = f"decode steps of {batch} tokens x {n} after a 128-token prefill (the GPU arm decodes after {GPT2_PREFILL}); oracle port"
    else:
        chunk = batch if ncores >= 16 else max(1, batch // 4)
        inp = make_inputs(oracle, model, chunk)
        arena = oracle.Arena()  # = the reference's BufferPool: operator outputs are recycled from pass to pass
        if model == "resnet50":
            one = lambda: model_ref.resnet50_oracle(oracle, spec, inp["x"], arena)
        elif model == "resnet50_int8":
            one = lambda: model_ref.resnet50_int8_oracle(oracle, spec, inp["x"])
        else:
            one = lambda: model_ref.bert_oracle(oracle, spec, inp["ids"], inp["tt"], inp["mask"])
        reps = n * (batch // chunk)

        def run():
            for _ in range(reps):
                one()

        per_step = chunk * reps
        sample = f"{per_step} inputs per step in chunks of {chunk} (= batch {batch} x {n} GPU(s)); CPU restatement of the rten path (oracle/), the Rust reference cannot be built here"
    for _ in range(max(1, min(args.warmup, 1))):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = time.perf_counter() - t0
    val = per_step * args.steps / dt
    cores = oracle.num_threads()
    return {
        "impl": "reference", "metric": metric_name(model), "value": val, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if model in ("resnet50", "bert") else "u8 x i8 -> i32 (f32 between layers)", "data": "synthetic",
        "config": config_of(model, batch, args.gpus),
        "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


# ------------------------------------------------------------------------------------------
# measurement helpers (GPU arm)
# ------------------------------------------------------------------------------------------
def measure_matmul_peaks(torch, n=8192, sustained_s=3.0):
    """cuBLASLt through torch on this box, in this run: burst (best of 10) and sustained (back to back for 3 s)."""
    out = {}
    torch.backends.cuda.matmul.allow_tf32 = True
    cases = {"tf32": (torch.float32, torch.matmul), "int8": (torch.int8, torch._int_mm), "bf16": (torch.bfloat16, torch.matmul)}
    for name, (dt, fn) in cases.items():
        try:
            if dt == torch.int8:
                a = torch.randint(-128, 127, (n, n), device="cuda", dtype=dt)
                b = torch.randint(-128, 127, (n, n), device="cuda", dtype=dt)
            else:
                a = torch.randn(n, n, device="cuda", dtype=dt)
                b = torch.randn(n, n, device="cuda", dtype=dt)
            for _ in range(3):
                fn(a, b)
            torch.cuda.synchronize()
            best = 1e9
            for _ in range(10):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                fn(a, b)
                e.record()
                torch.cuda.synchronize()
                best = min(best, s.elapsed_time(e))
            t0 = time.time()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            cnt = 0
            while time.time() - t0 < sustained_s:
                for _ in range(20):
                    fn(a, b)
                cnt += 20
                torch.cuda.synchronize()
            e.record()
            torch.cuda.synchronize()
            out[name] = {"burst": 2.0 * n ** 3 / best / 1e9, "sustained": 2.0 * n ** 3 * cnt / s.elapsed_time(e) / 1e9}
            del a, b
        except Exception as ex:  # noqa: BLE001
            out[name] = {"error": str(ex)[:200]}
    torch.backends.cuda.matmul.allow_tf32 = False
    return out


def graph_kernel_times(torch, launch, reps=3):
    """Per-kernel device time of `reps` graph replays from CUPTI kernel records (torch.profiler) -> {name: (count, us)}
    per replay, or None when the profiler is unavailable."""
    try:
        from torch.profiler import ProfilerActivity, profile
        launch()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                launch()
            torch.cuda.synchronize()
        rows = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0.0)
            if t and ev.count:
                rows[ev.key] = (ev.count / reps, float(t) / reps)
        return rows or None
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="resnet50", choices=sorted(MODELS))
    ap.add_argument("--no-graph", action="store_true", help="issue ops one by one instead of replaying a CUDA graph (profiling aid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-autotune", action="store_true", help="use the cost model's launch plans instead of timing candidates during warm-up")
    ap.add_argument("--plans", default=None, help="file of measured launch plans: loaded if it exists, (re)written after the warm-up pass")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary numbers (other configs, 8192^3 GEMM TFLOP/s)")
    ap.add_argument("--no-peaks", action="store_true", help="skip the on-box cuBLAS peak measurement (uses MEASURED_PEAKS.json ratios)")
    ap.add_argument("--modes", default=None, help="comma list restricting the f32 modes measured (tf32,tf32x3)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<output>_<mode>.npy (float32, 64 MiB at most in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    model = args.model
    batch = int(os.environ.get("RTEN_BENCH_BATCH", MODELS[model]["batch"]))  # (the override is a tuning aid: not a BASELINE config)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(run_reference_arm(args, model, batch)), flush=True)
        return

    import torch
    import torch.distributed as dist
    import rten_b200 as rt
    from rten_b200 import graphs, shard
    from oracle import oracle  # inputs / weights RNG + the cpu_baseline leg only

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: rten_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    comm_stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    spec = make_spec(oracle, model)
    inp = make_inputs(oracle, model, batch)
    unit = MODELS[model]["unit"]
    modes = MODELS[model]["modes"]
    if args.modes:
        modes = [m for m in modes if m in args.modes.split(",")] or modes

    def copy_desc(ctx, src, dst):
        ctx.check(ctx.lib.rten_b200_copy(ctx.handle, C.byref(src), C.byref(dst)))

    def host_desc(h):
        return rt.ops._desc(h.ctypes.data, h.dtype, h.shape, rt.ops._contig(h.shape), -1)

    def run_mode(mode, want_kernel_times):
        """One arithmetic mode: build the runner on a fresh context, warm up / autotune, capture, time value and e2e."""
        ctx = rt.Context(local_rank, stream=stream.cuda_stream)
        ctx.set_f32_mode(mode != "tf32")  # tf32 = explicit opt-in; everything else keeps the library default
        ctx.set_autotune(not args.no_autotune)
        if args.plans and os.path.exists(args.plans):
            ctx.load_plans(args.plans)
        comm = None
        if world > 1 and model == "resnet50_int8":
            ids = [rt.Comm.unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            comm = rt.Comm(ctx, ids[0], rank, world)
        res = {"mode": mode}
        if model == "gpt2":
            return run_gpt2(ctx, res)
        if model == "resnet50":
            runner = graphs.ResNet50Runner(ctx, spec, fuse=True)
            dev_inputs = [ctx.to_device(inp["x"], channels_last=True)]
            order = ["x"]
            flops = graphs.resnet50_flops(spec) * batch
        elif model == "resnet50_int8":
            runner = graphs.ResNet50Int8Runner(ctx, spec, fuse=True, comm=comm)
            dev_inputs = [ctx.to_device(inp["x"], channels_last=True)]
            order = ["x"]
            flops = None  # (the roofline block counts the integer ops of the same convolutions)
        else:
            runner = graphs.BertRunner(ctx, spec, fuse=True)
            dev_inputs = [ctx.to_device(inp["ids"]), ctx.to_device(inp["tt"]), ctx.to_device(inp["mask"])]
            order = ["ids", "tt", "mask"]
            flops = graphs.bert_flops(spec, batch, 128)
        step_fn = lambda: runner.run(*dev_inputs)
        out = step_fn()  # eager pass: plans measured, buffer pool warm
        ctx.sync()
        if args.plans and rank == 0:
            ctx.save_plans(args.plans)
        out_shape = tuple(out.shape)
        del out
        out_t = torch.empty(out_shape, dtype=torch.float32, device="cuda")
        out_dst = rt.from_torch(ctx, out_t)
        gather_bufs = [torch.empty(shard.gather_layout(world, out_shape), dtype=torch.float32, device="cuda") for _ in range(2)] if world > 1 else None
        graph, o_fixed = None, None
        # With a communicator the quantise kernels exchange their ranges over NVLink peer mailboxes inside the step: plain
        # kernels, capturable (the epoch lives in device memory, so replays stay in step across ranks as long as every rank
        # replays the same number of times).  Only the NCCL fallback (peer memory unavailable) keeps the step eager.
        use_graph = not args.no_graph and (comm is None or comm.uses_peer_memory)
        if use_graph:
            ctx.graph_begin()
            o_fixed = step_fn()
            if world == 1:
                copy_desc(ctx, o_fixed.desc(), out_dst.desc())
            graph = ctx.graph_end()
        ev_copied, ev_gathered = torch.cuda.Event(), [torch.cuda.Event(), torch.cuda.Event()]
        counter = {"i": 0}

        def device_step():
            """One step; at N > 1 the all-gather of step i runs on the comm stream, overlapped with step i + 1."""
            i = counter["i"]
            counter["i"] += 1
            if graph is not None:
                graph.launch()
                o = o_fixed
            else:
                o = step_fn()
            if world == 1:
                if graph is None:
                    copy_desc(ctx, o.desc(), out_dst.desc())
                return
            if i >= 1:
                stream.wait_event(ev_gathered[(i - 1) % 2])  # out_t is free again (long since)
            copy_desc(ctx, o.desc(), out_dst.desc())
            ev_copied.record(stream)
            comm_stream.wait_event(ev_copied)
            with torch.cuda.stream(comm_stream):
                shard.all_gather_outputs(dist, out_t, gather_bufs[i % 2])
                ev_gathered[i % 2].record(comm_stream)

        def timed(fn, steps, warmup, smp):
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            if smp:
                smp.start()
            evs = []
            l0 = ctx.launches
            for _ in range(steps):
                flush.zero_()  # L2 flush, outside the timed events
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(stream)
                fn()
                e.record(stream)
                evs.append((s, e))
            tail = torch.cuda.Event(enable_timing=True)
            tail.record(comm_stream if world > 1 else stream)  # after the last (overlapped) all-gather
            torch.cuda.synchronize()
            clocks = smp.stop() if smp else None
            if world > 1:
                dist.barrier()
            ms = sum(s.elapsed_time(e) for s, e in evs) + max(0.0, evs[-1][1].elapsed_time(tail))
            launches = ctx.launches - l0
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms, launches, clocks

        ms, launches, clocks = timed(device_step, args.steps, args.warmup, sampler)
        if args.dump_outputs and rank == 0:
            last = gather_bufs[(args.steps - 1) % 2] if world > 1 else out_t
            dump_output(args.dump_outputs, f"{OUTPUT_NAME[model]}_{mode}", last.cpu().numpy(), DUMP_BYTES // len(modes))
        res.update(value=batch * world * args.steps / (ms / 1e3), ms_per_step=ms / args.steps, gpu_launches=int(launches), clocks=clocks,
                   cuda_graph=graph is not None, flops_per_step=flops)
        if flops:
            res["model_tflops"] = flops * world * args.steps / (ms / 1e3) / 1e12
        if want_kernel_times and graph is not None and (rank == 0 or comm is not None):
            # (a step with cross-rank exchanges must be replayed by every rank the same number of times)
            kt = graph_kernel_times(torch, graph.launch)
            if rank == 0:
                res["kernel_times"] = kt

        # ---- e2e: pinned host inputs -> H2D -> step -> D2H of the result, every step, double-buffered on a copy stream
        pinned = []
        for name, d in zip(order, dev_inputs):
            h = ctx.pinned_empty(inp[name].shape, inp[name].dtype)
            h[...] = inp[name]
            pinned.append((h, d))
        h2d = sum(h.nbytes for h, _ in pinned)
        copy_stream = torch.cuda.Stream()
        cctx = rt.Context(local_rank, stream=copy_stream.cuda_stream)
        raw = [[cctx.empty(h.shape, h.dtype) for h, _ in pinned] for _ in range(2)]
        ev_in, ev_used, ev_done = ([torch.cuda.Event() for _ in range(2)] for _ in range(3))
        host_outs = [ctx.pinned_empty(out_shape, np.float32) for _ in range(2)]
        d2h = host_outs[0].nbytes
        out_bufs = [ctx.empty(out_shape, np.float32) for _ in range(2)]

        def issue_h2d(i):
            b = i % 2
            if i >= 2:
                copy_stream.wait_event(ev_used[b])
            for (h, _), r in zip(pinned, raw[b]):
                copy_desc(cctx, host_desc(h), r.desc())
            ev_in[b].record(copy_stream)

        def issue_d2h(i):
            b = i % 2
            copy_stream.wait_event(ev_done[b])
            copy_desc(cctx, out_bufs[b].desc(), host_desc(host_outs[b]))

        def e2e_run(steps):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(copy_stream)
            issue_h2d(0)
            for i in range(steps):
                b = i % 2
                stream.wait_event(ev_in[b])
                for (_, d), r in zip(pinned, raw[b]):
                    copy_desc(ctx, r.desc(), d.desc())  # layout change (channels-last), device to device
                ev_used[b].record(stream)
                flush.zero_()  # L2 flush between steps (inside the timed region here)
                device_step()
                copy_desc(ctx, out_dst.desc(), out_bufs[b].desc())
                ev_done[b].record(stream)
                if i + 1 < steps:
                    issue_h2d(i + 1)  # the host feeds the NEXT step and collects the PREVIOUS result while this one runs
                if i >= 1:
                    issue_d2h(i - 1)
            issue_d2h(steps - 1)
            t1.record(copy_stream)
            torch.cuda.synchronize()
            ms2 = t0.elapsed_time(t1)
            if world > 1:
                t = torch.tensor([ms2], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms2 = float(t.item())
            return ms2

        e2e_run(3)
        ms_e2e = e2e_run(args.steps)
        res["e2e"] = {"value": batch * world * args.steps / (ms_e2e / 1e3), "unit": unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                      "ms_per_step": ms_e2e / args.steps,
                      "how": "double-buffered: the copy stream moves step i+1's input H2D and step i-1's result D2H while step i computes; every step's H2D + D2H and the L2 flush are inside the timed region"}
        if comm is not None:
            res["comm"] = {"range_exchange": "NVLink peer mailboxes (one kernel prologue per DynamicQuantizeLinear)" if comm.uses_peer_memory else "ncclAllReduce x2",
                           "timeouts": comm.timeouts()}
            comm.close()
        return res

    def run_gpt2(ctx, res):
        """configs[4]: step = one decode step (8 tokens per GPU) replayed from one CUDA graph against a cache that holds a
        512-token prefill.  e2e = the same step driven the way rten-generate drives it: token ids H2D, graph, logits D2H."""
        run = graphs.GPT2Int8Runner(ctx, spec, batch, GPT2_CACHE)
        ids = inp["ids"]
        run.forward(ids[:, :GPT2_PREFILL])  # warm-up (autotune, pool)
        run.reset()
        ctx.set_autotune(False)
        run.build_prefill_graph(GPT2_PREFILL)  # the prefill's ~250 launches as ONE graph replay (eager issue is host-bound)
        run.prefill(ids[:, :GPT2_PREFILL])
        run.reset()
        torch.cuda.synchronize()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        run.prefill(ids[:, :GPT2_PREFILL])  # (token ids H2D + graph replay)
        e0.record(stream)
        ctx.set_autotune(not args.no_autotune)
        run.build_decode_graph()
        ctx.set_autotune(False)
        torch.cuda.synchronize()
        res["prefill_tokens_per_sec"] = batch * world * GPT2_PREFILL / (s0.elapsed_time(e0) / 1e3)
        vocab = run._g_logits.shape[1]
        host_logits = ctx.pinned_empty((batch, vocab), np.float32)
        gather_buf = torch.empty((world * batch, vocab), dtype=torch.float32, device="cuda") if world > 1 else None
        logits_t = torch.empty((batch, vocab), dtype=torch.float32, device="cuda")
        logits_dst = rt.from_torch(ctx, logits_t)
        nmax = GPT2_CACHE - GPT2_PREFILL - 1

        def replay_only():
            run._graph.launch()  # same cache position every time: the work of a step does not depend on it
            if world > 1:
                copy_desc(ctx, run._g_logits.desc(), logits_dst.desc())
                shard.all_gather_outputs(dist, logits_t, gather_buf)

        run._write_step_inputs(ids[:, GPT2_PREFILL:GPT2_PREFILL + 1])
        for _ in range(args.warmup):
            replay_only()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if sampler:
            sampler.start()
        evs, l0 = [], ctx.launches
        for _ in range(args.steps):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            replay_only()
            e.record(stream)
            evs.append((s, e))
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        if args.dump_outputs and rank == 0:
            last = gather_buf.cpu().numpy() if world > 1 else run._g_logits.numpy()
            dump_output(args.dump_outputs, f"{OUTPUT_NAME[model]}_{res['mode']}", last, DUMP_BYTES // len(modes))
        ms = sum(s.elapsed_time(e) for s, e in evs)
        launches = ctx.launches - l0
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        res.update(value=batch * world * args.steps / (ms / 1e3), ms_per_step=ms / args.steps, gpu_launches=int(launches), clocks=clocks, cuda_graph=True,
                   flops_per_step=None)
        if rank == 0:
            res["kernel_times"] = graph_kernel_times(torch, run._graph.launch)
        # e2e: ids H2D (+ position bookkeeping), replay, logits D2H to pinned host memory, synchronously per step
        steps = min(args.steps, nmax)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for i in range(steps):
            lg = run.decode_step(ids[:, GPT2_PREFILL + i:GPT2_PREFILL + i + 1])
            copy_desc(ctx, lg.desc(), host_desc(host_logits))
        t1.record(stream)
        torch.cuda.synchronize()
        ms2 = t0.elapsed_time(t1)
        res["e2e"] = {"value": batch * world * steps / (ms2 / 1e3), "unit": unit, "h2d_bytes_per_step": int(run._host_ints.nbytes + run._host_len.nbytes),
                      "d2h_bytes_per_step": int(host_logits.nbytes), "ms_per_step": ms2 / steps,
                      "how": "per step: token ids / position / cache length H2D, one graph replay, logits D2H to pinned host memory, host-synchronous (the next token depends on the logits)"}
        # algorithmic HBM bytes of a decode step: int8 weights once + the valid part of the f32 KV cache once
        wbytes = sum(l.wq.size for L in spec.layers for l in (L.attn, L.proj, L.fc, L.fc2)) + spec.lm_head.wq.size
        kv = 2 * len(spec.layers) * batch * spec.hidden * 4 * (GPT2_PREFILL + 1)
        res["algorithmic_bytes_per_step"] = float(wbytes + kv)
        return res

    # ---- the measured modes
    results = {}
    for k, mode in enumerate(modes):
        results[mode] = run_mode(mode, want_kernel_times=True)
    head = results[modes[0]]

    peaks_meas = None
    if rank == 0 and not args.no_peaks:
        peaks_meas = measure_matmul_peaks(torch)
    extras = None
    if rank == 0 and not args.no_extras and model == "resnet50":
        extras = secondary_numbers(rt, graphs, oracle, stream, torch, flush, sampler, local_rank)

    if rank == 0:
        peaks = load_peaks()

        def peak_of(kind):
            if peaks_meas and kind in peaks_meas and "burst" in peaks_meas[kind]:
                return peaks_meas[kind]["burst"], peaks_meas[kind]["sustained"], "measured in this run: cuBLASLt 8192^3 through torch (burst = best of 10, sustained = 3 s)"
            f = 0.5 if kind == "tf32" else 2.0
            return f * peaks["bf16_burst"], f * peaks["bf16_sustained"], f"{f} x bf16 of {peaks['src']} (no on-box measurement in this run)"

        def roofline_of(r):
            kt = r.get("kernel_times")
            step_ms = r["ms_per_step"]
            if model == "gpt2":
                ach_lb = r["algorithmic_bytes_per_step"] / (step_ms / 1e3) / 1e9
                kern_us = sum(t for name, (_, t) in kt.items() if "qlinear" in name or "attn_decode" in name) if kt else None
                if kern_us:
                    kern_us = min(kern_us, step_ms * 1e3)  # (durations overlap under programmatic dependent launch)
                ach = r["algorithmic_bytes_per_step"] / (kern_us / 1e6) / 1e9 if kern_us else ach_lb
                return {"bound": "hbm", "kernel": "rtb::qlinear_kernel + rtb::attn_decode_kernel (decode step: int8 weights + f32 KV cache streamed once)",
                        "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                        "lower_bound": {"achieved": ach_lb, "frac": ach_lb / peaks["hbm_gbs"], "how": "algorithmic bytes / whole step time"},
                        "kernel_time_us_per_step": kern_us, "source": "CUPTI kernel records of the graph replay" if kern_us else "whole step time",
                        "peak_source": peaks["src"]}
            kind = "int8" if model == "resnet50_int8" else "tf32"
            fl = r.get("flops_per_step")
            if model == "resnet50_int8":
                fl = graphs.resnet50_flops(make_spec(oracle, "resnet50")) * batch
            burst, sust, psrc = peak_of(kind)
            lb = fl / (step_ms / 1e3) / 1e12
            kern_us = sum(t for name, (_, t) in kt.items() if "umma_" in name) if kt else None
            n_kern = sum(c for name, (c, _) in kt.items() if "umma_" in name) if kt else None
            # With programmatic dependent launch the kernels of a step OVERLAP (kernel n + 1 is resident, waiting in
            # griddepcontrol.wait, while kernel n drains), so the sum of the CUPTI durations can exceed the step time: the
            # time the tensor-core kernels occupy the GPU is then bounded by the step itself.
            busy_us = min(kern_us, step_ms * 1e3) if kern_us else None
            ach = fl / (busy_us / 1e6) / 1e12 if busy_us else lb
            lw = layerwise_floor_us(model, spec, batch, burst, peaks["hbm_gbs"])
            if lw:
                lw["frac"] = lw["floor_us"] / (step_ms * 1e3)
                lw["how"] = ("sum over the conv layers of max(layer flops / tensor peak, layer HBM bytes / HBM peak) divided by the step time: "
                             "the fraction of the per-layer roofline this step reaches (flops counted 1x in both f32 modes)")
            return {"bound": "tensor", "layerwise": lw, "kernel": f"rtb::umma_gemm_kernel<{1 if kind == 'int8' else 0}> (tcgen05 kind::{'i8' if kind == 'int8' else 'tf32'} implicit-GEMM conv / GEMM)",
                    "achieved": ach, "peak": burst, "unit": "TFLOP/s" if kind == "tf32" else "TOP/s", "frac": ach / burst, "frac_of_sustained_peak": ach / sust,
                    "traffic": ncu_traffic(model),
                    "lower_bound": {"achieved": lb, "frac": lb / burst, "how": "algorithmic flops / whole step time (kernel time <= step time)"},
                    "kernel_time_us_per_step": busy_us, "sum_of_kernel_durations_us": kern_us, "launches_per_step": n_kern,
                    "share_of_step": (busy_us / 1e3 / step_ms) if busy_us else None,
                    "source": ("CUPTI kernel records of the GRAPH replay (torch.profiler); durations overlap under programmatic dependent launch, "
                               "so the busy time is min(sum of durations, step time)") if kern_us else "whole step time (profiler unavailable)",
                    "peak_source": psrc,
                    "hbm_view": {"achieved": hbm_bytes(model, spec, batch) / (step_ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": hbm_bytes(model, spec, batch) / (step_ms / 1e3) / 1e9 / peaks["hbm_gbs"],
                                 "bytes": "algorithmic: every operand / output / residual of every conv and GEMM once, over the whole step time"}}

        def public(r):
            keep = {k: r[k] for k in ("value", "ms_per_step", "gpu_launches", "clocks", "e2e", "cuda_graph", "comm") if k in r}
            if r.get("model_tflops"):
                keep["model_tflops"] = r["model_tflops"]
            if r.get("prefill_tokens_per_sec"):
                keep["prefill_tokens_per_sec"] = r["prefill_tokens_per_sec"]
            keep["roofline"] = roofline_of(r)
            if r.get("kernel_times"):
                top = sorted(r["kernel_times"].items(), key=lambda kv: -kv[1][1])[:6]
                keep["top_kernels_us_per_step"] = {k[:70]: round(v[1], 1) for k, v in top}
            return keep

        dtype = {"tf32": "f32(tf32 mma, explicit opt-in)", "tf32x3": "f32(3xtf32 mma, fp32-grade)", "int8": "u8 x i8 -> i32 (f32 between layers)"}[modes[0]]
        line = {"metric": metric_name(model), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config_of(model, batch, world)}
        line.update(public(head))
        line["f32_mode"] = modes[0] if modes[0] != "int8" else None
        if len(modes) > 1:
            line["modes"] = {m: public(results[m]) for m in modes[1:]}
            for m in modes[1:]:
                line["modes"][m]["dtype"] = "f32(3xtf32 mma, fp32-grade: library default)"
        if peaks_meas:
            line["peaks_measured"] = peaks_meas
        if extras:
            b_tf32, _, src = peak_of("tf32")
            b_i8, _, _ = peak_of("int8")
            extras["gemm_tf32_8192_frac_of_peak"] = extras["gemm_tf32_8192_tflops"] / b_tf32
            extras["gemm_int8_8192_frac_of_peak"] = extras["gemm_int8_8192_tops"] / b_i8
            extras["peaks"] = src
            line["also"] = extras
        if not args.no_cpu_baseline:
            a2 = argparse.Namespace(**vars(args))
            a2.steps, a2.warmup, a2.gpus = 1, 1, 1
            line["cpu_baseline"] = run_reference_arm(a2, model, batch)["cpu_baseline"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def hbm_bytes(model, spec, batch):
    """Algorithmic bytes of the tensor-core ops of one step: activations in / out (+ residual) and weights once (SURVEY.md 8d)."""
    if model == "bert":
        h, f, t = spec.hidden, spec.ffn, batch * 128
        per_layer = 4 * (4 * h * h + 2 * h * f) + 4 * t * (h * 8 + 2 * f) + 4 * 2 * batch * spec.heads * 128 * 128
        return float(per_layer * len(spec.layers))
    es_in = 1 if model == "resnet50_int8" else 4
    total, hw = 0.0, 224

    def conv(c, h_in):
        w = c.wq if hasattr(c, "wq") else c.w
        o, i, k, _ = w.shape
        ho = (h_in + 2 * c.pad - k) // c.stride + 1
        return batch * (i * h_in * h_in * es_in + o * ho * ho * 4) + w.size * es_in, ho

    b0, h = conv(spec.stem, hw)
    total += b0
    h = (h + 2 - 3) // 2 + 1
    for blk in spec.blocks:
        b1, h1 = conv(blk.c1, h)
        b2, h2 = conv(blk.c2, h1)
        b3, h3 = conv(blk.c3, h2)
        total += b1 + b2 + b3 + batch * blk.c3.b.size * h3 * h3 * 4  # + the residual read
        if blk.down is not None:
            total += conv(blk.down, h)[0]
        h = h3
    return total


def layerwise_floor_us(model, spec, batch, tensor_tflops, hbm_gbs):
    """Per-layer roofline of the ResNet-50 step: every conv layer takes at least max(flops / tensor peak, algorithmic HBM
    bytes / HBM peak); the sum is the step's floor.  (A whole-step `flops / peak` ignores that the 1x1 layers of the first
    stages are HBM-bound at this batch size: no kernel can run them at the tensor peak.)"""
    if model not in ("resnet50", "resnet50_int8"):
        return None
    es_in = 1 if model == "resnet50_int8" else 4
    rows = []

    def conv(c, h_in, residual=False):
        w = c.wq if hasattr(c, "wq") else c.w
        o, i, k, _ = w.shape
        ho = (h_in + 2 * c.pad - k) // c.stride + 1
        by = batch * (i * h_in * h_in * es_in + o * ho * ho * 4 * (2 if residual else 1)) + w.size * es_in
        fl = 2.0 * batch * o * ho * ho * i * k * k
        rows.append((fl, by))
        return ho

    h = conv(spec.stem, 224)
    h = (h + 2 - 3) // 2 + 1
    for blk in spec.blocks:
        h1 = conv(blk.c1, h)
        h2 = conv(blk.c2, h1)
        h3 = conv(blk.c3, h2, residual=True)
        if blk.down is not None:
            conv(blk.down, h)
        h = h3
    t_f = sum(fl / (tensor_tflops * 1e12) for fl, _ in rows) * 1e6
    t_b = sum(by / (hbm_gbs * 1e9) for _, by in rows) * 1e6
    t = sum(max(fl / (tensor_tflops * 1e12), by / (hbm_gbs * 1e9)) for fl, by in rows) * 1e6
    return {"floor_us": t, "tensor_only_us": t_f, "hbm_only_us": t_b, "layers": len(rows),
            "hbm_bound_layers": sum(1 for fl, by in rows if by / (hbm_gbs * 1e9) > fl / (tensor_tflops * 1e12))}


def ncu_traffic(model):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture of this same command (profiles/r02_ncu_<model>.json, falling back to round 1's); None if absent."""
    for name in (f"r02_ncu_{model}.json", "r01_ncu_resnet50.json" if model == "resnet50" else ""):
        p = os.path.join(ROOT, "profiles", name)
        try:
            return json.load(open(p))["umma_avg_dram_bytes_per_launch"]
        except Exception:
            continue
    return None


def secondary_numbers(rt, graphs, oracle, stream, torch, flush, sampler, device):
    """Secondary numbers the BASELINE metric names, same timing hygiene, few steps, each with its own clock sample."""
    out = {}
    ctx = rt.Context(device, stream=stream.cuda_stream)
    ctx.set_f32_mode(False)
    ctx.set_autotune(True)

    def timed(fn, iters=5, warm=2, tag=None):
        fn()
        ctx.graph_begin()
        fn()
        g = ctx.graph_end()
        for _ in range(warm):
            g.launch()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        ms = []
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            g.launch()
            e.record(stream)
            torch.cuda.synchronize()
            ms.append(s.elapsed_time(e))
        if sampler and tag:
            out.setdefault("clocks", {})[tag] = sampler.stop()
        del g
        return float(np.median(ms))

    n = 8192
    a = rt.from_torch(ctx, torch.randn(n, n, device="cuda"))
    b = rt.from_torch(ctx, torch.randn(n, n, device="cuda")).permute(1, 0)
    o = ctx.empty((n, n))
    out["gemm_tf32_8192_tflops"] = 2.0 * n ** 3 / timed(lambda: rt.MatMul().run(ctx, a, b, out=o), tag="gemm_tf32_8192") / 1e9
    ai = rt.from_torch(ctx, torch.randint(0, 255, (n, n), device="cuda", dtype=torch.uint8))
    bi = rt.from_torch(ctx, torch.randint(-128, 127, (n, n), device="cuda", dtype=torch.int8)).permute(1, 0)
    oi = ctx.empty((n, n), np.int32)
    out["gemm_int8_8192_tops"] = 2.0 * n ** 3 / timed(lambda: rt.MatMulInteger().run(ctx, ai, bi, out=oi), tag="gemm_int8_8192") / 1e9
    del a, b, o, ai, bi, oi
    spec = make_spec(oracle, "bert")
    inp = make_inputs(oracle, "bert", 16)
    for mode, x3 in (("tf32", False), ("tf32x3", True)):
        ctx.set_f32_mode(x3)
        runner = graphs.BertRunner(ctx, spec)
        ids, tt, mask = ctx.to_device(inp["ids"]), ctx.to_device(inp["tt"]), ctx.to_device(inp["mask"])
        ms = timed(lambda: runner.run(ids, tt, mask), tag=f"bert_{mode}")
        out[f"bert_base_fp32_b16_s128_seq_per_sec_{mode}"] = 16 / (ms / 1e3)
        out[f"bert_base_model_tflops_{mode}"] = graphs.bert_flops(spec, 16, 128) / ms / 1e9
        del runner
    ctx.set_f32_mode(False)
    # configs[3]: dynamically quantised ResNet-50, batch 64
    qrunner = graphs.ResNet50Int8Runner(ctx, make_spec(oracle, "resnet50_int8"), fuse=True)
    x64 = ctx.to_device(make_inputs(oracle, "resnet50", 64)["x"], channels_last=True)
    ms = timed(lambda: qrunner.run(x64), tag="resnet50_int8")
    out["resnet50_int8_b64_img_per_sec"] = 64 / (ms / 1e3)
    del qrunner, x64
    # configs[4]: GPT-2 small int8, batch 8: prefill of 512 tokens, then graph-replayed decode steps (fused decode path)
    ctx.set_f32_mode(True)  # the f32 attention products of the prefill at fp32 grade (library default)
    gspec = make_spec(oracle, "gpt2")
    grun = graphs.GPT2Int8Runner(ctx, gspec, 8, GPT2_CACHE)
    gids = make_inputs(oracle, "gpt2", 8)["ids"]
    grun.forward(gids[:, :GPT2_PREFILL])
    grun.reset()
    ctx.set_autotune(False)
    grun.build_prefill_graph(GPT2_PREFILL)
    grun.prefill(gids[:, :GPT2_PREFILL])
    grun.reset()
    torch.cuda.synchronize()
    s0, e0 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
    s0.record(stream)
    grun.prefill(gids[:, :GPT2_PREFILL])  # graph-replayed prefill (token ids H2D + one replay)
    e0.record(stream)
    ctx.set_autotune(True)
    grun.build_decode_graph()
    ctx.set_autotune(False)
    torch.cuda.synchronize()
    ndec = 32
    if sampler:
        sampler.start()
    e0b, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0b.record(stream)
    for i in range(ndec):
        grun.decode_step(gids[:, GPT2_PREFILL + i:GPT2_PREFILL + i + 1])  # per step: small H2D copies + one graph replay
    e1.record(stream)
    torch.cuda.synchronize()
    if sampler:
        out.setdefault("clocks", {})["gpt2"] = sampler.stop()
    out["gpt2_int8_b8_prefill512_tokens_per_sec"] = 8 * GPT2_PREFILL / (s0.elapsed_time(e0) / 1e3)
    out["gpt2_int8_b8_decode_tokens_per_sec"] = 8 * ndec / (e0b.elapsed_time(e1) / 1e3)
    return out


if __name__ == "__main__":
    main()
