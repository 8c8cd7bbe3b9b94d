"""GPU-side diagnostics and timing (run under gpurun; writes JSON lines to stdout).

  python tools/gpu_check.py diag            structured GEMM probes (localise layout / descriptor bugs)
  python tools/gpu_check.py time [Ms...]    GEMM timing, ours (auto / tall / skinny) vs the reference kernel
"""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402
from oracle import ref_gpu as R  # noqa: E402
from atom_b200 import ops  # noqa: E402


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def ulp(a, b):
    def key(x):
        u = x.view(np.uint16).astype(np.int32)
        return np.where(u & 0x8000, 0x8000 - u, u)
    return np.abs(key(a) - key(b))


def diag():
    cases = [(16, 128, 256, 1), (16, 128, 512, 1), (16, 256, 4096, 1), (16, 256, 4096, 0), (7, 384, 1024, 32), (32, 256, 2048, 16),
             (64, 128, 1024, 1), (128, 128, 512, 2)]
    if len(sys.argv) > 2:
        cases = [tuple(int(x) for x in a.split(",")) for a in sys.argv[2:]]
    for (m, n, k, flags) in cases:
        for probe in ("ones", "int_only", "random"):
            t = list(O.make_gemm_inputs(m, n, k, seed=7))
            g = k // 128 - 1
            if probe == "ones":
                t[0] = O.pack_int4(np.ones((m, k - 128), np.int8)); t[1] = O.pack_int4(np.ones((n, k - 128), np.int8))
                t[4] = np.ones((m, 128), np.int8); t[5] = np.ones((n, 128), np.int8)
            if probe in ("ones", "int_only"):
                t[2] = O.a_scale_to_layout(np.ones((g, m))); t[3] = np.ones((g, n), np.float16)
                t[6] = O.a_scale_to_layout(np.ones((1, m)))[0]; t[7] = np.ones((n,), np.float16)
                if probe == "int_only":   # keep magnitudes inside fp16
                    t[2] = O.a_scale_to_layout(np.full((g, m), 2.0 ** -6)); t[6] = O.a_scale_to_layout(np.full((1, m), 2.0 ** -10))[0]
            try:
                d = ops.dense_layer_gemm_i4_fp16(*[T(x) for x in t], flags=flags)
                torch.cuda.synchronize()
                d = d.cpu().numpy()
            except Exception as e:  # noqa: BLE001
                print(json.dumps({"diag": [m, n, k, flags], "probe": probe, "error": str(e)[:300]}), flush=True)
                continue
            ref = O.gemm_i4_o16(*t)
            u = ulp(d, ref)
            rec = {"diag": [m, n, k, flags], "probe": probe, "max_ulp": int(u.max()), "mismatch_frac": float((u != 0).mean())}
            if u.max() != 0:
                bad = u != 0
                rec["bad_rows"] = np.nonzero(bad.any(1))[0][:16].tolist()
                rec["bad_cols"] = np.nonzero(bad.any(0))[0][:16].tolist()
                rec["got_sample"] = d[:2, :8].astype(float).tolist()
                rec["ref_sample"] = ref[:2, :8].astype(float).tolist()
            print(json.dumps(rec), flush=True)


def bench(fn, nrot, iters=50, warmup=5):
    """CUDA-event timing on the current stream; `fn(i)` must use buffer set i % nrot (rotating sets defeat L2)."""
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    ts = []
    for i in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(i); e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2], ts[len(ts) // 10], ts[(len(ts) * 9) // 10]


def timing(ms_list):
    n = k = 4096
    for m in ms_list:
        base = O.make_gemm_inputs(m, n, k, seed=1)
        per_set = sum(x.nbytes for x in base)
        nrot = max(3, int(300e6 // per_set) + 1)     # > 126 MB L2 in flight
        sets = [[T(x) for x in base] for _ in range(nrot)]
        outs = [torch.empty((m, n), dtype=torch.float16, device="cuda") for _ in range(nrot)]
        ops_count = 2.0 * m * n * k
        rec = {"time": [m, n, k], "rot_sets": nrot}
        variants = {"auto": 0, "nosplit": 1, "tall": 2}
        if m <= 128:
            variants["skinny_nosplit"] = 5
            variants["skinny"] = 4
        for name, flags in variants.items():
            try:
                med, p10, p90 = bench(lambda i: ops.dense_layer_gemm_i4_fp16(*sets[i % nrot], flags=flags), nrot)
                rec[name] = {"us": round(med, 2), "p10": round(p10, 2), "p90": round(p90, 2), "TOPS": round(ops_count / med * 1e-6, 1)}
            except Exception as e:  # noqa: BLE001
                rec[name] = {"error": str(e)[:200]}
        if R.available():
            med, p10, p90 = bench(lambda i: R.gemm_i4_o16(*sets[i % nrot], d=outs[i % nrot], sync=0), nrot)
            rec["reference_kernel"] = {"us": round(med, 2), "TOPS": round(ops_count / med * 1e-6, 1)}
        # launch-overhead-free estimate: many back-to-back launches inside one event pair
        reps = 20
        def burst(i):
            for j in range(reps):
                ops.dense_layer_gemm_i4_fp16(*sets[(i * reps + j) % nrot], flags=0)
        med, _, _ = bench(burst, nrot, iters=10, warmup=2)
        rec["auto_back_to_back_us"] = round(med / reps, 2)
        print(json.dumps(rec), flush=True)


def graph_time(fn, nrot, launches=20, reps=20):
    """GPU time per launch with launch overhead removed: `launches` calls captured in one CUDA graph, replayed."""
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for i in range(nrot):
            fn(i)                      # warm-up outside capture (func attributes, TMA descriptor cache)
        st.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for i in range(launches):
                fn(i)
        g.replay(); st.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); g.replay(); e1.record(st); e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / launches)
    ts.sort()
    return ts[len(ts) // 2]


def gtiming(ms_list, n=4096, k=4096):
    for m in ms_list:
        base = O.make_gemm_inputs(m, n, k, seed=1)
        per_set = sum(x.nbytes for x in base)
        nrot = max(3, int(300e6 // per_set) + 1)
        sets = [[T(x) for x in base] for _ in range(nrot)]
        outs = [torch.empty((m, n), dtype=torch.float16, device="cuda") for _ in range(nrot)]
        ops_count = 2.0 * m * n * k
        rec = {"graph_time": [m, n, k], "rot_sets": nrot}
        variants = {"auto": 0, "nosplit": 1}
        if 64 < m <= 128:
            variants["skinny"] = 4
        if m > 64:
            variants["tall128"] = 2           # 128 x 128 tiles
        launches = nrot if m <= 512 else 6
        for name, flags in variants.items():
            us = graph_time(lambda i: ops.dense_layer_gemm_i4_fp16(*sets[i % nrot], flags=flags), nrot, launches=launches)
            rec[name] = {"us": round(us, 2), "TOPS": round(ops_count / us * 1e-6, 1)}
        if R.available() and m in (16, 4096):
            us = graph_time(lambda i: R.gemm_i4_o16(*sets[i % nrot], d=outs[i % nrot], sync=0), nrot, launches=4, reps=5) \
                if False else None   # the reference launches on the legacy stream: not capturable; use event timing
            med, _, _ = bench(lambda i: R.gemm_i4_o16(*sets[i % nrot], d=outs[i % nrot], sync=0), nrot, iters=10)
            rec["reference_kernel_us"] = round(med, 1)
        print(json.dumps(rec), flush=True)


def trace(m, flags, n=4096, k=4096):
    from atom_b200 import _lib
    t = [T(x) for x in O.make_gemm_inputs(m, n, k, seed=1)]
    buf = torch.zeros((4096, 128), dtype=torch.int64, device="cuda")
    for _ in range(3):
        ops.dense_layer_gemm_i4_fp16(*t, flags=flags)
    # cold-ish run: flush L2 with a big write first
    junk = torch.empty(64 << 20, dtype=torch.int32, device="cuda"); junk.fill_(1)
    _lib.lib().atom_gemm_set_trace(buf.data_ptr())
    ops.dense_layer_gemm_i4_fp16(*t, flags=flags)
    torch.cuda.synchronize()
    _lib.lib().atom_gemm_set_trace(None)
    b = buf.cpu().numpy()
    used = np.nonzero(b[:, 0])[0]
    out = {"trace": [m, n, k, flags], "ctas": int(len(used))}
    for cta in used[[len(used) // 2]]:
        r = b[cta]; t0 = r[0]
        rel = lambda x: None if x == 0 else int(x - t0)
        names = ["producer", "conv_slot", "conv_data", "conv_stored", "conv_arrived", "mma_woke", "acc_ready"]
        d = {"setup": rel(r[1]), "epi_loop_done": rel(r[2]), "reduced": rel(r[3]), "end": rel(r[4]),
             "q_batch0_ready": rel(r[5]), "dependency_resolved": rel(r[6]), "scales_staged": rel(r[7])}
        for i, nm in enumerate(names):
            d[nm] = [rel(x) for x in r[8 + 16 * i:8 + 16 * i + 8]]
        d["mma_loop_top"] = [rel(x) for x in r[96:104]]       # decode kernel only (slots free there)
        d["mma_issued"] = [rel(x) for x in r[16:24]]
        d["mma_committed"] = [rel(x) for x in r[32:40]]
        d["epi_done"] = [rel(x) for x in r[120:128]]
        out[f"cta{cta}"] = d
    print(json.dumps(out), flush=True)


def trace_warm(m, flags, n=4096, k=4096):
    """Pipeline stamps of the LAST launch of a replayed graph of back-to-back GEMMs on rotating operand sets (steady state,
    programmatic dependent launch active): per-CTA intervals relative to the CTA's own start, median / p10 / p90 over CTAs."""
    from atom_b200 import _lib
    base = O.make_gemm_inputs(m, n, k, seed=1)
    per_set = sum(x.nbytes for x in base)
    nrot = max(3, int(300e6 // per_set) + 1)
    sets = [[T(x) for x in base] for _ in range(nrot)]
    buf = torch.zeros((4096, 128), dtype=torch.int64, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for i in range(3):
            ops.dense_layer_gemm_i4_fp16(*sets[i], flags=flags)
        st.synchronize()
        _lib.lib().atom_gemm_set_trace(buf.data_ptr())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for i in range(nrot):
                ops.dense_layer_gemm_i4_fp16(*sets[i], flags=flags)
        _lib.lib().atom_gemm_set_trace(None)
        for _ in range(3):
            g.replay()
        st.synchronize()
    b = buf.cpu().numpy()
    used = np.nonzero(b[:, 0])[0]
    rel = (b[used] - b[used, 0:1]).astype(np.float64)
    rel[b[used] == 0] = np.nan
    def q(col):
        v = rel[:, col]; v = v[~np.isnan(v)]
        return None if len(v) == 0 else [int(np.percentile(v, p)) for p in (10, 50, 90)]
    out = {"trace_warm": [m, n, k, flags], "ctas": int(len(used)), "p10_p50_p90_cycles_from_cta_start": {
        "setup_done": q(1), "dependency_resolved": q(6), "q_batch0_ready": q(5), "scales_staged": q(7),
        "first_weights_landed": q(40), "first_unit_converted": q(72), "mma_top_0": q(96), "mma_woke_0": q(88), "mma_issued_0": q(16), "mma_committed_0": q(32), "mma_top_1": q(97), "mma_woke_1": q(89),
        "mma_top_2": q(98), "mma_woke_2": q(90), "mma_top_3": q(99), "mma_woke_3": q(91),
        "acc_ready_0": q(104), "acc_ready_3": q(107), "epi_done_0": q(120), "epi_done_3": q(123),
        "epi_loop_done": q(2), "reduced": q(3), "end": q(4)}}
    # spread of CTA start times of the last launch (global clock64 differs per SM only by a constant offset: informative only)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    cmd = sys.argv[1]
    if cmd == "diag":
        diag()
    elif cmd == "gtime":
        gtiming([int(x) for x in sys.argv[2:]] or [16, 32, 64, 128, 256, 1024, 4096])
    elif cmd == "gshape":      # gshape [M N K] : compare split-K factors on one shape (default: the Llama-7B/13B decode shapes)
        shapes = [tuple(int(x) for x in sys.argv[2:5])] if len(sys.argv) >= 5 else [
            (16, 4096, 4096), (16, 11008, 4096), (16, 4096, 11008), (32, 5120, 5120), (32, 13824, 5120), (32, 5120, 13824),
            (64, 4096, 4096)]
        for m, n, k in shapes:
            base = O.make_gemm_inputs(m, n, k, seed=1)
            per_set = sum(x.nbytes for x in base)
            nrot = max(3, int(300e6 // per_set) + 1)
            sets = [[T(x) for x in base] for _ in range(nrot)]
            rec = {"gshape": [m, n, k]}
            for name, flags in {"auto": 0, "nosplit": 1, "split2": 16, "split4": 32, "split8": 64}.items():
                us = graph_time(lambda i: ops.dense_layer_gemm_i4_fp16(*sets[i % nrot], flags=flags), nrot, launches=nrot)
                rec[name] = round(us, 2)
            print(json.dumps(rec), flush=True)
            del sets
    elif cmd == "trace":       # trace M FLAGS [N K]
        trace(int(sys.argv[2]), int(sys.argv[3]), *[int(x) for x in sys.argv[4:6]])
    elif cmd == "tracew":
        trace_warm(int(sys.argv[2]), int(sys.argv[3]))
    elif cmd == "time":
        timing([int(x) for x in sys.argv[2:]] or [16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
