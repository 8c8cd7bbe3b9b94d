#!/usr/bin/env python
"""bench.py -- the reference's headline benchmark (BASELINE.json configs[1]): gemm_i4_o16, M=16, N=K=4096,
group 128, INT8 keeper 128, on synthetic random-quantised operands.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--m M] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Besides the headline line this also reports, in the same JSON object:
  "sweep": the reference's nvbench axis (bench_dense_layer_gemm_i4_o16.cu:64-69) at M = 16 / 256 / 1024 / 4096, each against
           min(HBM, tensor) roofline;
  "tp":    BASELINE config #5 -- one decode step of a Llama-65B-shaped W4A4 decoder layer, tensor-parallel over the N
           ranks of this run (N = 1: the whole layer on one GPU), one CUDA graph per step with the two all-reduces of the
           layer INSIDE the timed region -> tokens/s at 80 layers (strong scaling: the work is fixed, N grows).

One "step" = one pass of the hot path over one batch of synthetic input: `gemms_per_step` independent GEMM problems
(distinct operand sets, together larger than the 126 MB L2, so every launch streams its weights from HBM), launched
back to back from one CUDA graph.  `value` = whole-job TOP/s with operands resident in HBM (OP = 2*M*N*K, the
reference's convention, bench_dense_layer_gemm_i4_o16.cu:40-42); multi-GPU runs give every rank its own batch (weak
scaling, no data-path collective: GEMM problems are independent units).  `e2e` = the same metric through the public
operator (atom_b200.ops.dense_layer_gemm_i4_fp16) with HOST activations: per step one pinned H2D copy of the quantised
activation tuple, the GEMM, and a D2H read of the FP16 result.

--dump-outputs DIR writes, after the timed steps, what the last step returned to its caller as float32 .npy files (rank 0):
gemm_out.npy is the [M, N] result of the last GEMM of the last headline step (every GEMM of a step computes on a copy of the
same operands), e2e_out.npy the host result of the last e2e step.  The operands come from fixed seeds, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L2_BYTES = 126e6
DUMP_BYTES = 60 << 20          # --dump-outputs: under 64 MB in all, .npy headers included

# BASELINE.md section 1: the reference's published bench_gemm_i4_o16 numbers (RTX 4090, figures/bench_gemm.png), TOP/s by M
PUBLISHED_TOPS = {16: 20.079, 32: 38.334, 64: 78.997, 128: 151.281, 256: 312.242, 512: 546.035, 1024: 630.779,
                  2048: 713.778, 4096: 772.992}


def algorithmic_bytes(m, n, k):
    """SURVEY.md 8(d): packed operands + keepers + scales + FP16 output, per launch."""
    g1 = k // 128
    s_m = m // 16 * 64 + 64 - (1 - (m % 16) // 8) * (8 - (m % 8)) * 8
    return (m + n) * (k - 128) // 2 + (m + n) * 128 + 2 * g1 * s_m + 2 * g1 * n + 2 * m * n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = [n for i, n in ((4, "hw_slowdown"), (5, "hw_thermal_slowdown"), (6, "sw_thermal_slowdown"), (7, "sw_power_cap"))
                   if any(r[i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[3]) for r in rows if r[3] not in ("[N/A]", ""))}


def cpu_baseline(m, n, k, budget_s=12.0):
    """The reference's simulated-quantisation CPU path (model/quant.py + qLinearLayer, BASELINE config #1), restated in
    oracle/fakequant.py, timed on all host cores: quantise the weight once (untimed), then act fake-quant + F.linear."""
    from oracle import fakequant as FQ   # the one other place bench.py may execute oracle/
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    args = FQ.w4a4_args()
    torch.manual_seed(0)
    lin = torch.nn.Linear(k, n, bias=False)
    wq = FQ.fq_linear_weight(lin.weight.detach().float(), args)
    x = torch.randn(m, k)
    FQ.fq_linear_forward(x, wq, args)
    t0, it = time.perf_counter(), 0
    while True:
        FQ.fq_linear_forward(x, wq, args)
        it += 1
        el = time.perf_counter() - t0
        if el > budget_s or it >= 200:
            break
    tops = 2.0 * m * n * k * it / el * 1e-12
    return {"value": tops, "unit": "TOP/s", "cores": cores, "kind": "port",
            "sample": f"{it} forwards of the fake-quant W4A4 linear (fp32 torch, act quant + F.linear) at M={m}, N={n}, K={k} in {el:.1f} s"}


def dump_outputs(dirname, arrays):
    """Writes each array as DIRNAME/<name>.npy in float32.  Above DUMP_BYTES in all, every array keeps the same share of
    its elements, drawn with a fixed seed (flattened, in index order), so that runs stay comparable element for element."""
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    for name, a in arrays.items():
        a = a.detach().float()
        if total > DUMP_BYTES:
            keep = a.numel() * DUMP_BYTES // total
            idx = np.unique(np.random.default_rng(0).integers(0, a.numel(), keep))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(dirname, name + ".npy"), a.cpu().numpy())


def ncu_traffic(m):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        return json.load(open(p)).get(f"gemm_m{m}", {}).get("dram_bytes_per_launch")
    except (OSError, ValueError):
        return None


def graph_time_us(fn, nsets, launches, reps, dev):
    """Median device time per launch: `launches` calls of fn(i) captured in one CUDA graph, replayed `reps` times."""
    st = torch.cuda.Stream(dev)
    with torch.cuda.stream(st):
        for i in range(min(nsets, launches)):
            fn(i)
        st.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for i in range(launches):
                fn(i)
        for _ in range(3):
            g.replay()
        st.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); g.replay(); e1.record(st); e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / launches)
    ts.sort()
    return ts[len(ts) // 2]


def gemm_sweep(dev, peaks, ms=(16, 256, 1024, 4096), n=4096, k=4096):
    """bench_gemm_i4_o16 axis: device time per GEMM (graph replay over operand sets larger than L2) and the roofline
    fraction against min(HBM, tensor) with the measured denominators."""
    from atom_b200 import ops, synth
    hbm = peaks.get("hbm_gbs", 6650.0)
    tc = 2.0 * peaks.get("bf16_tflops", 1590.0)
    out = []
    for m in ms:
        one = synth.gemm_operands(m, n, k, dev, seed=99 + m)
        per_set = sum(t.numel() * t.element_size() for t in one) + m * n * 2
        nsets = max(3, int(2.4 * L2_BYTES // per_set) + 1)
        sets = [one] + [tuple(t.clone() for t in one) for _ in range(nsets - 1)]
        us = graph_time_us(lambda i: ops.dense_layer_gemm_i4_fp16(*sets[i % nsets]), nsets, launches=nsets if m <= 256 else 8,
                           reps=15, dev=dev)
        op, alg = 2.0 * m * n * k, algorithmic_bytes(m, n, k)
        t_hbm, t_tc = alg / (hbm * 1e9), op / (tc * 1e12)
        rec = {"M": m, "us": round(us, 2), "TOPS": round(op / us * 1e-6, 1), "bound": "hbm" if t_hbm >= t_tc else "tensor",
               "frac": round(max(t_hbm, t_tc) * 1e6 / us, 3),
               "vs_published_rtx4090": round(op / us * 1e-6 / PUBLISHED_TOPS[m], 2) if m in PUBLISHED_TOPS else None}
        out.append(rec)
        del sets
        torch.cuda.empty_cache()
    return {"shape": f"N={n} K={k}", "peaks": {"hbm_gbs": hbm, "int8_tensor_tops": tc, "int8_peak_is": "2 x measured bf16 cuBLAS burst"},
            "points": out}


def tp_decode_layer(rank, world, dev, hidden=8192, inter=22016, heads=64, batch=32, kvlen=1024, page=32, layers=80, iters=20):
    """BASELINE config #5: decode step of a Llama-65B-shaped W4A4 layer, tensor-parallel over `world` ranks: heads and MLP
    channels sharded, hidden state replicated, ONE all-reduce per column->row pair (two per layer), all captured in one
    CUDA graph per step.  Enough independent layer copies are chained that a rank's weights + KV exceed L2."""
    import torch.distributed as dist
    from atom_b200.kvcache import BatchedKvCacheInt4, KvCacheInt4, KvPoolInt4
    from atom_b200.llama import LlamaConfig
    from atom_b200.tp import TPLlamaDecoderLayer
    from atom_b200.comm import make_allreduce
    allreduce = make_allreduce(batch * hidden, dev) if world > 1 else None
    cfg = LlamaConfig(hidden_size=hidden, intermediate_size=inter, num_attention_heads=heads, num_hidden_layers=1)
    lh = heads // world
    w_bytes = (4 * hidden * hidden + 3 * hidden * inter) / 2 * 1.0625 / world
    kv_bytes = batch * lh * (kvlen + 1) * 136
    copies = max(2, int(2.4 * L2_BYTES // (w_bytes + kv_bytes)) + 1)
    mods, kvs = [], []
    for i in range(copies):
        mods.append(TPLlamaDecoderLayer(cfg, 0, rank, world, allreduce=allreduce).to(dev).init_random(i))
        pool = KvPoolInt4(1, lh, 128, capacity=batch * ((kvlen + page) // page + 1), block_len=page, device=dev)
        pool.buf.random_(0, 256); pool.param[..., 0].uniform_(0.01, 0.05); pool.param[..., 1].uniform_(0.0, 0.4)
        caches = [KvCacheInt4(pool, kvlen) for _ in range(batch)]
        for c in caches:
            c.acquire_one()
        kvs.append(BatchedKvCacheInt4(caches))
    x = torch.randn(batch, hidden, device=dev, dtype=torch.float16)

    def step():
        # consecutive layers hand their down projection over un-reduced: its all-reduce (like o_proj's) is formed inside the next
        # add+RMSNorm launch from what the GEMM epilogues pushed into the peers' receive buffers (push all-reduce only)
        y, pend = x, None
        for i, (l, kv) in enumerate(zip(mods, kvs)):
            y, pend = l.forward_chain(y, pend, kv, last=(i == len(mods) - 1))
        return y

    st = torch.cuda.Stream(dev)
    with torch.cuda.stream(st):
        for _ in range(3):
            step()
        st.synchronize()
        if world > 1:
            dist.barrier()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            step()
        for _ in range(3):
            g.replay()
        st.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(iters):
            g.replay()
        e1.record(st)
        e1.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters / copies
    t = torch.tensor([us], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    us = t.item()
    rec = {"metric": "llama_decode_tokens_per_s", "model_shape": {"hidden": hidden, "intermediate": inter, "heads": heads, "layers": layers},
           "tp": world, "batch": batch, "kv_len": kvlen, "us_per_layer": round(us, 1),
           "value": round(batch / (us * layers * 1e-6), 1), "unit": "tokens/s", "scaling": "strong",
           "allreduces_per_layer": 2 if world > 1 else 0, "allreduce": allreduce.name if allreduce is not None else None,
           "allreduce_fused_into_gemm_and_rmsnorm": bool(world > 1 and mods[0].o_proj.can_push(batch)),
           "allreduce_bytes": batch * hidden * 2 if world > 1 else 0,
           "launch": f"one CUDA graph per step over {copies} chained layer copies ({(w_bytes + kv_bytes) * copies / 1e6:.0f} MB of weights + KV per rank > L2), "
                     "collectives captured inside, device time, max over ranks",
           "hbm_bytes_per_layer_per_rank": int(w_bytes + kv_bytes),
           "hbm_frac": round((w_bytes + kv_bytes) / (us * 1e-6) * 1e-9 / 6573.2, 3)}
    g = None                 # a captured NCCL graph must be gone before the communicator is torn down
    del mods, kvs
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-tp", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    M, N, K = a.m, 4096, 4096
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: atom_b200 has no CPU path")
    ref_mode = a.impl == "reference"
    if ref_mode and world > 1:
        # the reference has no multi-GPU path: rank 0 alone measures it (single GPU), the other ranks leave at once
        if rank != 0:
            return
        world = 1
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    if ref_mode:
        from oracle import ref_gpu as R
        if not R.available():
            # no compiled reference on this box: time the CPU port instead (rank 0 only)
            if rank == 0:
                cb = cpu_baseline(M, N, K, budget_s=20.0)
                print(json.dumps({"impl": "reference", "metric": "gemm_i4_o16_throughput", "value": cb["value"], "unit": "TOP/s",
                                  "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "higher_is_better": True,
                                  "config": {"workload": f"gemm_i4_o16 M={M} N={N} K={K} group128 keeper128"}, "cpu_baseline": cb,
                                  "e2e": {"value": cb["value"], "unit": "TOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
            return
    from atom_b200 import ops, synth

    # ------------------------------------------------------------------ operands: R distinct sets > L2
    one = synth.gemm_operands(M, N, K, dev, seed=1234 + rank)
    per_set = sum(t.numel() * t.element_size() for t in one)
    R_sets = int(2.4 * L2_BYTES // per_set) + 1
    sets = [one] + [tuple(t.clone() for t in one) for _ in range(R_sets - 1)]
    outs = [torch.empty((M, N), dtype=torch.float16, device=dev) for _ in range(R_sets)]
    op_count = 2.0 * M * N * K
    # The reference launcher uses the LEGACY default stream (GEMM.cuh:763): its arm is enqueued, timed and synchronised on
    # exactly that stream (torch's default stream is the legacy stream), so the events bracket the kernels.  A non-blocking
    # side stream would not order against legacy-stream work at all and the events would time the CPU enqueue rate.
    stream = torch.cuda.default_stream(dev) if ref_mode else torch.cuda.Stream(dev)

    def run_batch():
        """Runs one step's GEMMs and returns the result of the last one."""
        if ref_mode:   # the reference launches on the legacy default stream (GEMM.cuh:763): not capturable, plain loop
            for i in range(R_sets):
                R.gemm_i4_o16(*sets[i], d=outs[i], sync=0)
            return outs[-1]
        # results are dropped as they come, so the allocator can hand one output buffer to every GEMM of the step
        for i in range(R_sets - 1):
            ops.dense_layer_gemm_i4_fp16(*sets[i])
        return ops.dense_layer_gemm_i4_fp16(*sets[-1])

    graph = None
    with torch.cuda.stream(stream):
        last_out = run_batch()
        stream.synchronize()
        torch.cuda.synchronize()
        if not ref_mode:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                last_out = run_batch()        # every replay rewrites this tensor

    launch_desc = "one CUDA graph replay per step" if graph is not None else "python loop on the legacy stream (reference launcher)"

    def step():
        if graph is not None:
            graph.replay()
        else:
            run_batch()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # nvidia-smi needs a few hundred ms to produce its first sample: start before the warm-up
    with torch.cuda.stream(stream):
        t_w = time.perf_counter()
        n_w = 0
        while n_w < max(a.warmup, 3) or time.perf_counter() - t_w < 0.4:     # same warm-up rule for both arms
            step(); n_w += 1
            if n_w % 50 == 0:
                stream.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        w0 = time.perf_counter()
        e0.record(stream)
        for _ in range(a.steps):
            step()
        e1.record(stream)
        barrier()
        wall_ms = (time.perf_counter() - w0) * 1e3
        ms = e0.elapsed_time(e1)
        # the events sit on the stream the kernels run on, so the device time they bracket must account for (nearly) all
        # of the host's wall clock between the two synchronising barriers; a large gap means they did not bracket the work
        assert ms >= 0.7 * wall_ms - 1.0, f"timing contract broken: events {ms:.3f} ms vs wall clock {wall_ms:.3f} ms"
    clocks = sampler.stop() if rank == 0 else None
    dumped = {"gemm_out": last_out.clone()} if a.dump_outputs and rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    ms_per_step = ms / a.steps
    value = op_count * R_sets * world / (ms_per_step * 1e-3) * 1e-12

    # ------------------------------------------------------------------ e2e: host activations in, host result out
    act_bytes = sum(one[i].numel() * one[i].element_size() for i in (0, 2, 4, 6))
    host_in = torch.empty(act_bytes + 64, dtype=torch.uint8).pin_memory()
    host_out = torch.empty((M, N), dtype=torch.float16).pin_memory()
    dev_in = torch.empty(act_bytes + 64, dtype=torch.uint8, device=dev)
    views, off = [], 0
    for i in (0, 2, 4, 6):   # a, a_scale, a_keeper, a_keeper_scale packed into one staging buffer (16-B aligned views)
        nb = one[i].numel() * one[i].element_size()
        host_in[off:off + nb] = one[i].reshape(-1).view(torch.uint8).cpu()
        views.append(dev_in[off:off + nb].view(one[i].dtype).view(one[i].shape))
        off += (nb + 15) // 16 * 16
    e2e_steps = min(a.steps, 200) if ref_mode else a.steps

    def e2e_step(i):
        w = sets[i % R_sets]
        dev_in.copy_(host_in, non_blocking=True)
        if ref_mode:
            torch.cuda.current_stream().synchronize()      # the reference kernel runs on the legacy stream
            d = R.gemm_i4_o16(views[0], w[1], views[1], w[3], views[2], w[5], views[3], w[7], d=outs[i % R_sets], sync=1)
        else:
            d = ops.dense_layer_gemm_i4_fp16(views[0], w[1], views[1], w[3], views[2], w[5], views[3], w[7])
        host_out.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()          # the caller reads the result

    # our arm: the whole step (pinned H2D copy node, GEMM kernel node, D2H copy node) is captured once in a CUDA graph --
    # the operator is capturable by design (no allocation / synchronisation inside the C ABI) -- and replayed per step;
    # the caller still synchronises every step to read the result.  The reference launches on the legacy stream and
    # cannot be captured: it runs the same three operations eagerly.
    e2e_graphs = None
    if not ref_mode:
        gs = torch.cuda.Stream(dev)
        with torch.cuda.stream(gs):
            for i in range(3):
                e2e_step(i)
            e2e_graphs = []
            for i in range(min(R_sets, 8)):           # a few weight sets, so consecutive steps do not hit L2
                g = torch.cuda.CUDAGraph()
                w = sets[i]
                with torch.cuda.graph(g, stream=gs):
                    dev_in.copy_(host_in, non_blocking=True)
                    d = ops.dense_layer_gemm_i4_fp16(views[0], w[1], views[1], w[3], views[2], w[5], views[3], w[7])
                    host_out.copy_(d, non_blocking=True)
                e2e_graphs.append(g)
            gs.synchronize()

        def e2e_step(i):   # noqa: F811
            e2e_graphs[i % len(e2e_graphs)].replay()
            gs.synchronize()

    for i in range(5):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_tops = op_count * e2e_steps * world / t.item() * 1e-12
    if dumped is not None:
        dumped["e2e_out"] = host_out.clone()
        dump_outputs(a.dump_outputs, dumped)
    # self-check of the timing contract: one device-timed launch cannot take longer than a whole synchronised e2e step
    # (H2D + the same launch + D2H + sync); if it does, the events did not bracket the kernels
    e2e_us_per_step = t.item() / e2e_steps * 1e6
    assert ms_per_step * 1e3 / R_sets <= e2e_us_per_step * 1.05, \
        f"timing contract broken: {ms_per_step * 1e3 / R_sets:.2f} us per launch (events) > {e2e_us_per_step:.2f} us per e2e step"

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    # ------------------------------------------------------------------ config #5: tensor-parallel decode layer (all ranks)
    tp_rec = None
    if not ref_mode and not a.no_tp:
        graph = e2e_graphs = None          # the captured graphs reference the operand sets freed next
        del sets, outs
        torch.cuda.empty_cache()
        try:
            tp_rec = tp_decode_layer(rank, world, dev)
        except Exception as e:  # noqa: BLE001  (the headline line must still be printed)
            tp_rec = {"error": str(e)[:300]}
    if rank != 0:
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            os._exit(0)
        return
    sweep = None
    if not ref_mode and not a.no_sweep:
        try:
            sweep = gemm_sweep(dev, peaks)
        except Exception as e:  # noqa: BLE001
            sweep = {"error": str(e)[:300]}
    # ------------------------------------------------------------------ roofline of the dominant kernel
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    us_per_launch = ms_per_step * 1e3 / R_sets
    alg = algorithmic_bytes(M, N, K)
    # HBM-bound up to the crossover M*~200 (BASELINE.md section 2); tensor-bound above it
    int8_peak_tops = 2.0 * peaks.get("bf16_tflops", 1590.0)
    t_hbm, t_tc = alg / (hbm_peak * 1e9), op_count / (int8_peak_tops * 1e12)
    if t_hbm >= t_tc:
        ach = alg / (us_per_launch * 1e-6) * 1e-9
        roof = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": ncu_traffic(M),
                "algorithmic_bytes_per_launch": alg, "us_per_launch": us_per_launch, "peak_source": peak_src}
    else:
        ach = op_count / (us_per_launch * 1e-6) * 1e-12
        roof = {"bound": "tensor", "achieved": ach, "peak": int8_peak_tops, "unit": "TOP/s", "frac": ach / int8_peak_tops,
                "traffic": ncu_traffic(M), "us_per_launch": us_per_launch,
                "peak_source": "2 x measured bf16 cuBLAS burst (INT8 tcgen05 = 2x bf16 rate; Blackwell has no INT4 MMA)"}
    line = {
        "metric": "gemm_i4_o16_throughput", "value": value, "unit": "TOP/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": (value / PUBLISHED_TOPS[M]) if M in PUBLISHED_TOPS else None, "dtype": "s4 x s4 -> s32 (via tcgen05 kind::i8), fp16 out",
        "data": "synthetic", "impl": a.impl,
        "config": {"workload": f"gemm_i4_o16 M={M} N={N} K={K} (K incl. 128 INT8 keeper) group_size=128", "gemms_per_step": R_sets,
                   "l2": f"{R_sets} distinct operand sets per step = {R_sets * per_set / 1e6:.0f} MB > 126 MB L2 (inputs larger than L2)",
                   "launch": launch_desc,
                   "parallelism": f"dp{world} for the GEMM line (independent GEMM problems per rank, no collective); "
                                  f"tp{world} with two all-reduces per layer for the `tp` record",
                   "published_baseline": (f"{PUBLISHED_TOPS[M]} TOP/s on one RTX 4090 (BASELINE.md section 1, bench_gemm.png)"
                                          if M in PUBLISHED_TOPS else None)},
        "e2e": {"value": e2e_tops, "unit": "TOP/s", "h2d_bytes_per_step": act_bytes, "d2h_bytes_per_step": M * N * 2,
                "steps": e2e_steps, "note": "one GEMM per step: pinned H2D of the activation tuple, op, D2H of D, stream sync" + ("" if ref_mode else "; the three nodes replayed from one CUDA graph")},
        "gpu_launches": a.steps * R_sets + e2e_steps + 5,
        "roofline": roof, "clocks": clocks, "sweep": sweep, "tp": tp_rec,
    }
    if ref_mode:
        line["cpu_baseline"] = {"value": value, "unit": "TOP/s", "cores": 0, "kind": "reference",
                                "sample": "the reference's own CUDA kernel (oracle/_ref, compiled unmodified for sm_100a) on this GPU; "
                                          "its CPU path is the fake-quant simulator, see cpu_baseline of the main arm"}
        line["gpu_launches"] = 0   # none of OUR kernels ran in this arm
    elif world == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(M, N, K)
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)          # captured NCCL work + communicator teardown can block: leave once every rank is here


if __name__ == "__main__":
    main()
