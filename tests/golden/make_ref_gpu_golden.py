"""Regenerates tests/golden/ref_gpu_kernels.npz: the reference's own CUDA kernels (oracle/_ref/libatom_ref.so, built by
`make -C oracle ref` from the reference tree) run on a B200 over the inputs of tests/test_gpu_vs_reference.py.

Run from the repository root on a machine with the GPU and oracle/_ref/libatom_ref.so:
    python tests/golden/make_ref_gpu_golden.py [OUT.npz]
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_gpu as R  # noqa: E402
from tests import test_gpu_vs_reference as V  # noqa: E402


def main(out):
    if not R.available():
        raise SystemExit(f"{R.SO} not built: run `make -C oracle ref` where the reference tree is present")
    g = {}
    for m in V.REORDER_M:
        x, idx = V.reorder_inputs(m)
        g.update(V.record(f"reorder.{m}", (x, idx), V.quant_outputs(R.reorder_fp16_i4(x, idx), m)))
    for m in V.RMSNORM_M:
        x, w, idx = V.rmsnorm_inputs(m)
        g.update(V.record(f"rmsnorm.{m}", (x, w, idx), V.quant_outputs(R.rmsnorm_fp16_i4(x, w, idx, 1e-5), m)))
    for m in V.ACTIVATE_M:
        a, b = V.activate_inputs(m)
        g.update(V.record(f"activate.{m}", (a, b), V.quant_outputs(R.activate_fp16_i4(a, b), m)))
    for m, n, k in sorted({c[:3] for c in V.GEMM_O16_CASES}):
        t = V.gemm_o16_inputs(m, n, k)
        g.update(V.record(V.gemm_o16_key(m, n, k), t, {"d": R.gemm_i4_o16(*t)}))
        del t
        torch.cuda.empty_cache()
    t = V.gemm_splitk_inputs()
    g.update(V.record("gemm_o16_splitk", t, {}))
    g["gemm_o16_splitk.d"] = R.gemm_i4_o16(*t).cpu().numpy()
    for m in sorted({c[0] for c in V.GEMM_O4_CASES}):
        t = V.gemm_o4_inputs(m)
        d, ds = R.gemm_i4_o4(*t)
        g.update(V.record(f"gemm_o4.{m}", t, {"ds": ds, "d": d}))
    from tests.test_gpu_parity import _KV
    (data, param, indptr, indices, last), qn = V.decode_inputs()
    g.update(V.record("decode", (data, param, indptr, indices, last, qn), {}))
    kv, q = _KV(data, param, indptr, indices, last), V.T(qn)
    g["decode.o"] = np.stack([R.batch_decode_i4(q, kv.data, kv.param, kv.indptr, kv.indicies, kv.last_page_offset, layer).cpu().numpy()
                              for layer in range(V.DECODE_LAYERS)])
    fixture, (k, v, kp, vp) = V.append_kv_inputs()
    b = _KV(*fixture)
    R.append_kv_i4(b.data, b.param, b.indptr, b.indicies, b.last_page_offset, k, v, kp, vp, 1)
    g.update(V.record("append_kv", (*fixture, k, v, kp, vp), {"data": b.data, "param": b.param}))
    torch.cuda.synchronize()
    np.savez_compressed(out, **g)
    print(f"wrote {out}: {len(g)} arrays, {os.path.getsize(out)} bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_gpu_kernels.npz"))
