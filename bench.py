#!/usr/bin/env python
"""bench.py -- headline measurement of the GPTQ-4bit hot path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model 7b] [--ctx 1920]
                    [--groupsize 128] [--act-order] [--seq 2048] [--dump-outputs DIR]

One "step" = one decode token of a Llama-shaped stack on random GPTQ tensors of the named architecture (no checkpoints
exist offline): every layer's rms_norm + q/k/v projections + rope + cache write, attention over ctx cached positions,
o_proj + residual, rms_norm + gate/up + silu*mul + down + residual, then final norm + fp16 lm_head.

  value    : decode tok/s with inputs resident in HBM.  N = 1, no act-order: the whole token is ONE persistent kernel
             (exl_decode_step, csrc/decode_step.cu), K launches timed with CUDA events.  Otherwise (tensor parallel,
             act-order): the per-op kernels (q4_attn, decode_attn, q4_attn_2, q4_mlp) replayed as a CUDA graph.
  e2e      : the same metric through the C ABI called from the host every step, with the step's input hidden state
             copied from pinned host memory and the logits copied back inside the timed region.
  roofline : the dominant kernel.  Fused step: decode_step_kernel, algorithmic bytes = every q4 tensor + lm_head + the
             KV rows attended over, divided by the measured launch duration.  Per-op path: the gate+up launch.
  kernels  : the per-op launches (what the unchanged model.py drives) timed per launch, with their own fractions.
  cpu_baseline : the oracle's CPU port of dequant + GEMV on the box's host cores (bounded sample, own process, explicit
             thread count).

--impl reference times that CPU restatement (the reference ships no CPU path for q4; BASELINE.md section 3) and loads
nothing of this repo's native code.

--dump-outputs DIR writes what the timed path returned in its last timed step (the logits, float32) to DIR/logits.npy.
Weights, KV cache and hidden state are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="7b")
    ap.add_argument("--groupsize", type=int, default=128)
    ap.add_argument("--act-order", action="store_true", help="act-order (g_idx) GPTQ tensors (BASELINE configs 3 and 4)")
    ap.add_argument("--ctx", type=int, default=None, help="KV-cache length the decode step attends over (default seq - 128)")
    ap.add_argument("--seq", type=int, default=2048)
    ap.add_argument("--no-prefill", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-fused-step", action="store_true", help="time the per-op path even where the persistent kernel applies")
    ap.add_argument("--no-per-op", action="store_true", help="skip the per-op comparison rows (large models: saves time)")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="CPU sample budget per repetition (reference arm / cpu_baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's logits to DIR/logits.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.ctx is None:
        a.ctx = a.seq - 128
    return a


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region, sampled by a separate `nvidia-smi -lms` process (B200_PROFILING.md):
    an in-process NVML thread was seen to take ~60 ms per sample when several ranks share a box and stalled the launch loop."""

    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def result(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill(); out = ""
        clocks, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6 or not f[0].isdigit():
                continue
            clocks.append(int(f[0])); mx = int(f[1]) if f[1].isdigit() else mx
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        if not clocks:
            return {"sm_mhz": None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": 0}
        c = sorted(clocks)
        return {"sm_mhz": c[len(c) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(c)}


def measured_peaks():
    """(hbm GB/s, bf16 TF/s burst, bf16 TF/s sustained, kind).  The fallback (B200_PROFILING.md) is used LOUDLY."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "hbm_gbs" in d and "bf16_tflops" in d:
            return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    print("bench.py: WARNING: MEASURED_PEAKS.json absent or incomplete -- roofline fractions are against the FALLBACK peaks "
          "(6650 GB/s, 1590 TF/s) of B200_PROFILING.md", file=sys.stderr, flush=True)
    return 6650.0, 1590.0, 1400.0, "fallback"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def workload_name(shape, gs, act, ctx, seq):
    return f"{shape.name}-gptq4-g{gs}-{'act' if act else 'noact'} decode token at ctx {ctx} of seq {seq}"


def metric_name(args, shape):
    if args.model == "7b" and args.groupsize == 128 and not args.act_order:
        return "decode tok/s Llama-7B 4b GPTQ g128 (q4 hot path)"
    return f"decode tok/s {shape.name} 4b GPTQ g{args.groupsize}{' act-order' if args.act_order else ''}"


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the CPU restatement, own process, explicit thread count, nothing of exllama_b200's native code
# ---------------------------------------------------------------------------------------------------------------------
def cgroup_cpu_limit():
    """CPUs the container may actually use (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return max(1, int(float(q) / float(p)))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, q // p)
    except Exception:
        pass
    return None


def cpu_sample(shape, gs, act, seconds_budget, threads):
    """Oracle CPU port timed on the host: one decoder layer's seven q4 matmuls at M = 1 (bounded sample).
    threads: an int, or a list of candidate counts -- the fastest is used (an OpenMP team larger than the CPUs the container
    may use spends its time in spin barriers: 128 threads measured 400x slower than 64 on the round-2 box)."""
    from oracle import oracle as O
    O.lib()                                         # built by build(): bench.py compiles nothing into the tree
    dims = [(shape.hidden, shape.hidden)] * 4 + [(shape.hidden, shape.inter)] * 2 + [(shape.inter, shape.hidden)]
    tensors = []
    for i, (K, N) in enumerate(dims):
        qw, qz, sc, g_idx = O.synth_q4(K, N, gs, act_order=act, seed=i)
        x_map = None
        if act:
            x_map = O.make_x_map(g_idx, K // gs)
            qw = O.make_sequential(qw, x_map)
        tensors.append((O.synth_x(1, K, seed=i), qw, qz, sc, x_map))

    def layer():
        for x, qw, qz, sc, x_map in tensors:
            O.q4_matmul_cpu_f32(x, qw, qz, sc, x_map)
    if isinstance(threads, (list, tuple)):
        best = None
        for c in threads:
            O.set_num_threads(c)
            layer()
            dt = 1e9
            for _ in range(3):                      # best of 3: one noisy run must not pick a small team
                t0 = time.perf_counter(); layer(); dt = min(dt, time.perf_counter() - t0)
                if dt > 1.5:
                    break
            if best is None or dt < best[0]:
                best = (dt, c)
        threads = best[1]
    O.set_num_threads(threads)
    layer()
    t0 = time.perf_counter(); n = 0
    while True:
        layer(); n += 1
        if time.perf_counter() - t0 > seconds_budget or n >= 40:
            break
    return (time.perf_counter() - t0) * 1e3 / n, O.num_threads(), n


def run_reference(args):
    from exllama_b200.shapes import SHAPES          # torch-free, loads no native code of this repo
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape = SHAPES[args.model]
    ncpu = host_threads()                             # NOT OMP_NUM_THREADS: torchrun exports 1 to its children
    lim = cgroup_cpu_limit()
    cands = sorted({c for c in (ncpu, lim or ncpu, ncpu // 2, ncpu // 4, 64, 32, 16, 8) if c and 1 <= c <= ncpu}, reverse=True)
    _, threads, _ = cpu_sample(shape, args.groupsize, args.act_order, min(args.cpu_seconds, 3.0), cands)      # warm-up + pick the fastest team size
    samples = []
    for _ in range(max(1, min(args.steps, 3))):
        ms_layer, used, n = cpu_sample(shape, args.groupsize, args.act_order, args.cpu_seconds, threads)
        samples.append(ms_layer)
    ms_layer = sorted(samples)[len(samples) // 2]
    ms_tok = ms_layer * shape.layers
    val = 1000.0 / ms_tok
    sample = (f"oracle port (dequant + fp32 GEMV, OpenMP, {used} threads = fastest of {cands}; {ncpu} CPUs visible, cgroup limit {lim}) of one {shape.name} decoder layer's 7 q4 matmuls at M=1, "
              f"x{shape.layers} layers; attention/lm_head not included; median of {len(samples)} samples of ~{args.cpu_seconds:.0f} s")
    line = {
        "impl": "reference", "metric": metric_name(args, shape), "value": round(val, 4), "unit": "tok/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_tok, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(shape, args.groupsize, args.act_order, args.ctx, args.seq)},
        "detail": "CPU restatement of the q4 matmuls of the step, bounded sample (the reference has no CPU path for q4)",
        "cpu_baseline": {"value": round(val, 4), "unit": "tok/s", "cores": used, "kind": "port", "sample": sample},
        "e2e": {"value": round(val, 4), "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "native_modules_loaded": sorted(m for m in sys.modules if m.startswith("exllama_b200") and m not in ("exllama_b200", "exllama_b200.shapes")),
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args):
    """cpu_baseline of the main arm: the reference arm in its own process (a clean OpenMP runtime, no CUDA context polling
    threads beside it -- the in-process sample of round 1 was 9x low)."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--model", args.model, "--groupsize", str(args.groupsize),
           "--steps", "1", "--warmup", "0", "--ctx", str(args.ctx), "--seq", str(args.seq), "--cpu-seconds", str(args.cpu_seconds)]
    if args.act_order:
        cmd.append("--act-order")
    try:
        out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=180).stdout
        line = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
        return line["cpu_baseline"]
    except Exception as ex:  # noqa: BLE001
        return {"value": None, "unit": "tok/s", "cores": host_threads(), "kind": "port", "sample": f"failed: {ex!r}"[:200]}


def dump_outputs(directory, arrays):
    """--dump-outputs: each tensor as DIR/<name>.npy in float32 (64 MB at most: the logits of any SHAPES model are far less)."""
    import numpy as np
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > 64 << 20:
        raise ValueError(f"--dump-outputs: {total} bytes exceed 64 MB")
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from exllama_b200 import capi, cuda_ext
    from exllama_b200.shapes import SHAPES, q4_bytes
    from exllama_b200.stack import DecodeStack

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    else:
        torch.cuda.set_device(0)
    dev = torch.device(f"cuda:{local_rank}")
    shape = SHAPES[args.model]
    gs = args.groupsize
    hbm_peak, tf_peak, tf_sustained, peak_kind = measured_peaks()
    ext = cuda_ext.exllama_ext

    stack = DecodeStack(shape, groupsize=gs, act_order=args.act_order, device=str(dev), max_seq=args.seq,
                        tp_rank=rank, tp_size=world, tp_group=None)
    fused_ar = False
    if world > 1 and os.environ.get("EXL_TP_FUSED", "1") == "1":
        from exllama_b200 import tp as tpmod
        tpmod.init_fused_allreduce(ext, dev.index)      # row-parallel projections: GEMV + peer-memory all-reduce in one kernel
        fused_ar = True
    use_step = not args.no_fused_step and not (args.act_order and world > 1)      # act-order under TP: per-op path (o_proj needs the all-gathered attention output)
    if use_step:
        stack.make_plan()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    torch.manual_seed(0)                                          # the same step inputs in every run (the weights are seeded too)
    hidden0 = (torch.randn((1, 1, shape.hidden), device=dev) * 0.5).half()
    hidden = hidden0.clone()
    past = args.ctx
    for kc, vc in zip(stack.key_cache, stack.value_cache):        # fill the cache so attention reads real data
        kc.normal_(0, 0.5); vc.normal_(0, 0.5)

    def per_op_step():
        hidden.copy_(hidden0)
        return stack.decode_step(hidden, past)

    def fused_step():
        return stack.decode_step_fused(hidden0, past)

    def capture(fn):
        fn(); torch.cuda.synchronize()
        side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            out = fn()
        return g, out

    def time_events(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    # ------------------------------------------------------------------ parity of the two decode paths (same inputs)
    launches0 = capi.launch_count()
    logits_per_op = per_op_step().clone()
    torch.cuda.synchronize()
    launches_per_op = capi.launch_count() - launches0
    assert torch.isfinite(logits_per_op).all(), "non-finite logits in the synthetic stack"
    step_parity = None
    if use_step:
        lf = fused_step().clone()
        torch.cuda.synchronize()
        r = float(logits_per_op.pow(2).mean().sqrt())
        step_parity = {"max_abs_diff_vs_per_op_path": float((lf - logits_per_op).abs().max()), "logit_rms": r}
        assert step_parity["max_abs_diff_vs_per_op_path"] <= 2e-2 * max(r, 1e-6) + 2e-2 * float(logits_per_op.abs().max()), step_parity

    # ------------------------------------------------------------------ value: device-resident decode
    if use_step:
        step_device = fused_step                   # ONE launch per token: no graph needed
        launches_per_step = 1
        mode = "one persistent kernel per token (exl_decode_step)" + (f", {world} ranks: partials reduced over NVLink peer memory inside the kernel" if world > 1 else "")
        graph = None
    else:
        # NCCL inside stream capture hung on this stack; the fused all-reduce kernels are plain launches and capture fine
        use_graph = not args.no_graph and (world == 1 or (fused_ar and not args.act_order) or os.environ.get("EXL_BENCH_TP_GRAPH", "0") == "1")
        # (act-order + tensor parallel falls back to NCCL for the MLP; NCCL inside stream capture hung on this stack in round 1)
        graph, graph_out = capture(per_op_step) if use_graph else (None, None)

        def replay():
            graph.replay()
            return graph_out
        step_device = replay if graph is not None else per_op_step
        launches_per_step = launches_per_op
        mode = "per-op kernels, " + ("CUDA graph" if graph is not None else "eager")

    sampler = ClockSampler(local_rank)
    if rank == 0:
        # one GPU's clocks (rank 0's); started before the warm-up steps (the same kernel under the same load) so that the ~100 ms
        # timed region is covered by more than a couple of 50 ms samples; stopped right after the timed region
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.cudart().cudaProfilerStart()          # no-op unless run under `ncu --profile-from-start off`
    e0.record()
    for _ in range(args.steps):
        out = step_device()
    e1.record()
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": out})
    ms = e0.elapsed_time(e1)
    clocks = sampler.result() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = 1000.0 / ms_per_step

    # ------------------------------------------------------------------ e2e: C ABI called per step + host copies
    host_in = torch.randn((1, 1, shape.hidden)).half().pin_memory()
    host_out = torch.empty((1, shape.vocab), dtype=torch.float32).pin_memory()
    dev_in = torch.empty((1, 1, shape.hidden), dtype=torch.float16, device=dev)

    def step_e2e():
        dev_in.copy_(host_in, non_blocking=True)
        if use_step:
            lg = stack.decode_step_fused(dev_in, past)
        else:
            lg = stack.decode_step(dev_in, past)
        host_out.copy_(lg, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    n_e2e = args.steps
    for _ in range(n_e2e):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
    te = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())

    # ------------------------------------------------------------------ roofline
    wbytes = stack.q4_weight_bytes_per_token()
    head_bytes = shape.vocab * shape.hidden * 2
    kv_bytes = 2 * len(stack.layers) * past * stack.local_heads * shape.head_dim * 2
    kern_rows = []
    il = stack.layers[0].gate.width
    none = stack.none
    nl = len(stack.layers)

    def traffic_of(name):
        p = os.path.join(ROOT, "profiles", "traffic_r2.json")
        if world == 1 and args.model == "7b" and gs == 128 and not args.act_order and os.path.exists(p):
            return json.load(open(p)).get(name)
        return None

    if not args.no_per_op:
        x1 = (torch.randn((1, shape.hidden), device=dev) * 0.5).half()
        xm = x1.clone()
        tmp_i = stack.temp_mlp[:1, :il]
        tmp_h = x1[:, :stack.layers[0].o.height].contiguous()

        def mlp_all():
            for L in stack.layers:
                ext.q4_mlp(xm, L.ln2, shape.eps, L.gate.q4, L.up.q4, L.down.q4, none, none, none, none, none, none, none)

        def down_all():
            for L in stack.layers:
                ext.q4_attn_2(xm, tmp_i, L.down.q4, none, none, none)

        def o_all():
            for L in stack.layers:
                ext.q4_attn_2(xm, tmp_h, L.o.q4, none, none, none)
        if world == 1:
            rows = [("q4_mlp = [norm, gate+up, silu*mul] + [down += residual] (2 launches)", mlp_all,
                     2 * (q4_bytes(shape.hidden, il, gs, act=args.act_order) - 2 * shape.hidden) + 2 * shape.hidden - 2 * il + q4_bytes(il, shape.hidden, gs, act=args.act_order, accumulate=True), 2),
                    ("down (+residual)", down_all, q4_bytes(il, shape.hidden, gs, act=args.act_order, accumulate=True), 1),
                    ("o_proj (+residual)", o_all, q4_bytes(stack.layers[0].o.height, shape.hidden, gs, act=args.act_order, accumulate=True), 1)]
            for name, fn, by, nlaunch in rows:
                g, _ = capture(fn)
                for _ in range(2): g.replay()
                us = time_events(g.replay, 8) * 1e3 / nl
                kern_rows.append({"kernel": name, "launches": nlaunch, "us": round(us, 3), "bytes": by, "GBps": round(by / us / 1e3, 1),
                                  "frac": round(by / us / 1e3 / hbm_peak, 4), "timing": "CUDA events over a graph of all layers' launches (distinct weights >> L2)"})
                del g

    if use_step:
        step_bytes = wbytes + head_bytes + kv_bytes + 2 * shape.hidden + 4 * shape.vocab
        us_launch = ms_per_step * 1e3
        roofline = {"bound": "hbm", "achieved": round(step_bytes / us_launch / 1e3, 1), "peak": hbm_peak, "unit": "GB/s",
                    "frac": round(step_bytes / us_launch / 1e3 / hbm_peak, 4), "traffic": traffic_of("decode_step_kernel"),
                    "kernel": "decode_step_kernel (whole token: 32 x [qkv, attention, o, gate+up, down] + norm + lm_head)",
                    "peak_kind": peak_kind, "algorithmic_bytes_per_launch": step_bytes, "us_per_launch": round(us_launch, 2),
                    "us_per_launch_how": "CUDA events around the K timed launches (the step is one launch)",
                    "bytes_breakdown": {"q4_weights": wbytes, "lm_head_fp16": head_bytes, "kv_cache_read": kv_bytes}}
    else:
        # per-op path: the fused gate+up launch, measured as (q4_mlp - down) is not a measurement -> time q4_mlp directly and
        # report it (two launches) as the dominant row
        dom = kern_rows[0] if kern_rows else {"GBps": None, "frac": None, "bytes": None, "us": None, "kernel": None}
        roofline = {"bound": "hbm", "achieved": dom["GBps"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["frac"], "traffic": None,
                    "kernel": dom["kernel"], "peak_kind": peak_kind, "algorithmic_bytes_per_launch": dom["bytes"], "us_per_launch": dom["us"]}

    # ------------------------------------------------------------------ comparison rows: per-op path as a graph, torch attention
    extra = {}
    if world == 1 and not args.no_per_op:
        g = graph if graph is not None else capture(per_op_step)[0]
        for _ in range(3): g.replay()
        per_op_ms = time_events(g.replay, 16)
        extra["decode_per_op_graph"] = {"value": round(1000.0 / per_op_ms, 2), "unit": "tok/s", "launches_per_step": int(launches_per_op),
                                        "note": "the per-op kernels model.py drives (q4_attn, decode_attn, q4_attn_2, q4_mlp) + cuBLAS lm_head, CUDA graph"}
        stack.fused_decode_attn = False
        g2, _ = capture(per_op_step)
        for _ in range(3): g2.replay()
        extra["decode_torch_attention"] = {"value": round(1000.0 / time_events(g2.replay, 16), 2), "unit": "tok/s",
                                           "note": "same, with the reference's torch attention ops instead of decode_attn"}
        stack.fused_decode_attn = True
        del g2
        keep = past
        past = 4
        if use_step:
            for _ in range(3): fused_step()
            extra["decode_best_ctx4"] = {"value": round(1000.0 / time_events(fused_step, 16), 2), "unit": "tok/s", "mode": mode}
        else:
            for _ in range(3): per_op_step()
            extra["decode_best_ctx4"] = {"value": round(1000.0 / time_events(per_op_step, 16), 2), "unit": "tok/s", "mode": "eager"}
        past = keep

    # ------------------------------------------------------------------ tensor parallel: parity + cost of the collective
    tp_info = None
    if world > 1 and not use_step:
        from exllama_b200 import tp as tpmod
        tp_info = {}
        if fused_ar:
            lf = per_op_step().clone()
            tpmod._fused_ready = False                       # the NCCL all-reduce variant of the same sharded step
            ln = per_op_step().clone()
            tpmod._fused_ready = True
            tp_info["tp_parity"] = {"max_abs_diff_fused_vs_nccl": float((lf - ln).abs().max()), "logit_rms": float(ln.pow(2).mean().sqrt()),
                                    "what": "logits of the sharded step: GEMV+all-reduce kernel vs q4_*_tp + NCCL all_reduce"}
            L0 = stack.layers
            xa = (torch.randn((1, shape.hidden), device=dev) * 0.5).half()
            ta = (torch.randn((1, L0[0].o.height), device=dev) * 0.5).half()

            def o_ar():
                for L in L0: ext.q4_attn_2_ar(xa, ta, L.o.q4)

            def o_plain():
                for L in L0: ext.q4_attn_2_tp(xa, ta, L.o.q4, True)
            ga, gp = capture(o_ar)[0], capture(o_plain)[0]
            for _ in range(2): ga.replay(); gp.replay()
            barrier(); ua = time_events(ga.replay, 8) * 1e3 / nl
            barrier(); up = time_events(gp.replay, 8) * 1e3 / nl
            tp_info["allreduce_us"] = {"o_proj_gemv_with_fused_allreduce": round(ua, 2), "o_proj_gemv_store_only": round(up, 2),
                                       "allreduce_epilogue": round(ua - up, 2), "bytes": 2 * shape.hidden,
                                       "how": "mean per launch over all layers, CUDA graph, this rank"}
            tt = torch.tensor([ext.tp_status(dev.index)], device=dev, dtype=torch.int64)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            tp_info["allreduce_timeouts"] = int(tt.item())          # must be 0

    # ------------------------------------------------------------------ prefill
    prefill = None
    if not args.no_prefill:
        T = args.seq - 128
        hp = (torch.randn((1, T, shape.hidden), device=dev) * 0.5).half()
        try:
            for _ in range(2):
                stack.prefill(hp)
            barrier()
            nrep = 3
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(nrep):
                stack.prefill(hp)
            b.record(); barrier()
            pms = a.elapsed_time(b) / nrep
            flops = 2.0 * T * sum((l.q.height * l.q.width * 3 + l.o.height * l.o.width + l.gate.height * l.gate.width * 2 + l.down.height * l.down.width)
                                  for l in stack.layers)
            prefill = {"value": round(T / pms * 1e3, 1), "unit": "tok/s", "tokens": T, "ms": round(pms, 3),
                       "q4_linear_tflops": round(flops / pms / 1e9, 1), "q4_path": capi.last_q4_path(),
                       "roofline_prefill": {"bound": "tensor", "achieved": round(flops / pms / 1e9, 1), "peak": tf_sustained, "unit": "TFLOP/s",
                                            "frac": round(flops / pms / 1e9 / tf_sustained, 4), "peak_kind": peak_kind + " (sustained bf16 cuBLAS)",
                                            "note": "q4 linear layers' 2MKN over the WHOLE forward time (attention, norms and the head included in the time)"}}
        except Exception as ex:  # noqa: BLE001
            prefill = {"error": repr(ex)[:200]}

    # ------------------------------------------------------------------ cpu baseline (rank 0, N == 1, own process)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess(args)

    dropin = None
    dp = os.path.join(ROOT, "profiles", "dropin_7b_r2.json")
    if os.path.exists(dp):
        d = json.load(open(dp))
        dropin = {"source": "profiles/dropin_7b_r2.json (unchanged test_benchmark_inference.py -p -ppl over both extensions, same box)",
                  "ref": d.get("ref"), "ours": d.get("ours"), "ppl_rel_diff": d.get("ppl_rel_diff")}

    if rank == 0:
        line = {
            "metric": metric_name(args, shape),
            "value": round(value, 2), "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": workload_name(shape, gs, args.act_order, args.ctx, args.seq)},      # identical in both arms
            "run": {"detail": f"{shape.layers} layers x (norm, q/k/v, rope, cache write, attention over {past} cached positions, o_proj, norm, gate/up, silu*mul, down) + final norm + fp16 lm_head",
                       "decode_mode": mode, "parallelism": f"tp{world}", "cuda_graph": graph is not None,
                       "allreduce": (("inside decode_step_kernel: peer-memory reductions + cross-GPU barrier" if use_step else
                                      ("fused GEMV epilogue over NVLink peer memory" if fused_ar else "nccl")) if world > 1 else None),
                       "l2": f"weights ({(wbytes + head_bytes) / 1e9:.2f} GB/token/rank) >> L2 (126 MB): every step streams them from HBM"},
            "e2e": {"value": round(1000.0 / e2e_ms, 2), "unit": "tok/s", "h2d_bytes_per_step": host_in.numel() * 2,
                    "d2h_bytes_per_step": host_out.numel() * 4, "ms_per_step": round(e2e_ms, 4),
                    "mode": "C ABI call per step (exl_decode_step)" if use_step else "plugin API calls per op, eager"},
            "gpu_launches": int(launches_per_step * args.steps),
            "launches_per_step": int(launches_per_step),
            "clocks": clocks,
            "roofline": roofline,
            "kernels": kern_rows,
            "cpu_baseline": cpu,
            "prefill": prefill,
            "step_parity": step_parity,
            "tp": tp_info,
            "dropin": dropin,
            "q4_weight_bytes_per_token": wbytes,
            "weights_only_bound_tok_s": round(hbm_peak * 1e9 / (wbytes + head_bytes), 1),
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush()
        try:
            dist.barrier()
        except Exception:
            pass
        os._exit(0)            # skip NCCL / IPC teardown: a hang there once cost a 15-minute timeout on 4 GPUs


if __name__ == "__main__":
    main()
