"""GPU parity suite, part 2 (-m gpu): our kernels against what the REFERENCE'S OWN CUDA kernels return for the same inputs.

The reference's torch-extension sources, compiled unmodified for sm_100a (oracle/Makefile -> oracle/_ref/libatom_ref.so; the
INT4 mma.sync is emulated by ptxas on the INT8 pipe), were run on a B200 over exactly the inputs built below, and
tests/golden/ref_gpu_kernels.npz keeps what they returned (tests/golden/make_ref_gpu_golden.py regenerates it).  Outputs
compared bit for bit are stored as a SHA-256 digest of the whole array plus a fixed sample of its bytes; outputs compared
within a tolerance are stored whole.  This is the strongest available statement of drop-in parity, because the reference
ships no golden vectors for its GEMM or decode kernels (SURVEY.md 8c)."""
import functools
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gpu_kernels.npz")
SAMPLE_BYTES = 256

REORDER_M = [1, 7, 16, 100, 1024]
RMSNORM_M = [1, 7, 16, 100, 1024]
ACTIVATE_M = [1, 7, 16, 100]
GEMM_O16_CASES = [(16, 4096, 4096, 1), (7, 4096, 4096, 1), (128, 4096, 4096, 1), (128, 4096, 4096, 2), (1000, 4096, 4096, 0),
                  (4096, 4096, 4096, 0), (16, 11008, 4096, 1), (33, 4096, 11008, 1), (300, 4096, 11008, 0),
                  # Llama-13B (config #4) and Llama-65B TP-8 (config #5) projection shapes, decode batch 32
                  (32, 5120, 5120, 1), (32, 13824, 5120, 1), (32, 5120, 13824, 1), (32, 1024, 8192, 1),
                  (32, 8192, 2816, 1), (32, 8192, 2688, 1), (64, 8192, 1024, 1),
                  # prefill: the 7B MLP up-projection and config #3's 16 x 2048 tokens
                  (4096, 11008, 4096, 0), (32768, 4096, 4096, 0),
                  # the same prefill shapes forced through each of the two prefill kernels
                  (4096, 4096, 4096, 512), (4096, 4096, 4096, 1024), (1000, 11008, 4096, 512)]
GEMM_O4_CASES = [(16, 1), (16, 0), (33, 0), (100, 0), (1000, 0)]      # flags 0 = the default dispatch (o4 never splits K)
DECODE_LAYERS = 3


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


# ---------------------------------------------------------------------------------------------------- inputs (shared with
# make_ref_gpu_golden.py, which runs the reference kernels on them)

def reorder_inputs(m):
    rng = np.random.default_rng(m)
    return T((rng.standard_normal((m, 4096)) * 2).astype(np.float16)), T(rng.permutation(4096).astype(np.int16))


def rmsnorm_inputs(m):
    rng = np.random.default_rng(m + 1)
    x = T((rng.standard_normal((m, 4096)) * 2).astype(np.float16)); idx = T(rng.permutation(4096).astype(np.int16))
    return x, T((1 + 0.2 * rng.standard_normal(4096)).astype(np.float16)), idx


def activate_inputs(m):
    rng = np.random.default_rng(m + 2)
    return T((rng.standard_normal((m, 11008)) * 2).astype(np.float16)), T((rng.standard_normal((m, 11008)) * 2).astype(np.float16))


def gemm_o16_inputs(m, n, k):
    return [T(x) for x in O.make_gemm_inputs(m, n, k, seed=m + n + k, pair_shared=(m % 2 == 0))]


def gemm_splitk_inputs():
    return [T(x) for x in O.make_gemm_inputs(16, 4096, 4096, seed=3)]


def gemm_o4_inputs(m):
    return [T(x) for x in O.make_gemm_inputs(m, 4096, 4096, seed=m)]


def decode_inputs():
    from tests.test_gpu_parity import _kv_fixture
    rng = np.random.default_rng(0xabc)
    B, H, P, L = 7, 32, 16, DECODE_LAYERS
    lens = rng.integers(1, 500, B).tolist()
    fixture = _kv_fixture(rng, B, H, P, L, lens)
    return fixture, rng.standard_normal((B, H, 128)).astype(np.float16)


def append_kv_inputs():
    from tests.test_gpu_parity import _kv_fixture
    rng = np.random.default_rng(9)
    B, H, P, L = 4, 32, 16, 2
    fixture = _kv_fixture(rng, B, H, P, L, [1, 16, 17, 300])
    k = T(rng.integers(0, 256, (B, H, 64), dtype=np.uint8)); v = T(rng.integers(0, 256, (B, H, 64), dtype=np.uint8))
    kp = T(rng.random((B, H, 2)).astype(np.float16)); vp = T(rng.random((B, H, 2)).astype(np.float16))
    return fixture, (k, v, kp, vp)


# ---------------------------------------------------------------------------------------------------- stored reference outputs

def quant_outputs(out, m):
    """What the comparison covers of a quantiser's 4-tuple: both operands whole, the scales at the slots the layout uses."""
    idx = torch.tensor([O.scale_index(r) + 2 * j for r in range(m) for j in range(4)], device=out[2].device)
    return {"o8": out[0], "o4": out[1], "s8": out[2][idx], "s4": out[3][:, idx]}


def _bytes(a):
    if isinstance(a, torch.Tensor):
        a = a.contiguous().cpu().numpy()
    return np.ascontiguousarray(a).reshape(-1).view(np.uint8)


def _sample_index(nbytes):
    return np.random.default_rng(nbytes).integers(0, nbytes, min(SAMPLE_BYTES, nbytes))


def inputs_digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(_bytes(a))
    return np.frombuffer(h.digest(), np.uint8)


def record(key, inputs, outputs):
    """Golden entries of one case: the digest of its inputs and, per output, the digest of its bytes and a fixed sample."""
    rec = {f"{key}.inputs": inputs_digest(*inputs)}
    for name, a in outputs.items():
        b = _bytes(a)
        rec[f"{key}.{name}.sha256"] = np.frombuffer(hashlib.sha256(b).digest(), np.uint8)
        rec[f"{key}.{name}.sample"] = b[_sample_index(b.size)]
    return rec


@functools.lru_cache(maxsize=1)
def golden():
    with np.load(GOLDEN) as g:
        return {k: g[k] for k in g.files}


def check_inputs(key, inputs):
    assert np.array_equal(inputs_digest(*inputs), golden()[f"{key}.inputs"]), \
        f"{key}: the inputs are not the ones the reference outputs were recorded for (tests/golden/make_ref_gpu_golden.py)"


def assert_same_as_reference(key, inputs, outputs):
    """Bit-for-bit equality of every output with what the reference kernel returned for these inputs."""
    check_inputs(key, inputs)
    g = golden()
    for name, a in outputs.items():
        b = _bytes(a)
        want = g[f"{key}.{name}.sample"]
        got = b[_sample_index(b.size)]
        assert np.array_equal(got, want), f"{key}: {name}: {(got != want).sum()} of {want.size} sampled bytes differ from the reference"
        assert np.array_equal(np.frombuffer(hashlib.sha256(b).digest(), np.uint8), g[f"{key}.{name}.sha256"]), \
            f"{key}: {name} differs from the reference (outside the sampled bytes)"


def gemm_o16_key(m, n, k):
    return f"gemm_o16.{m}x{n}x{k}"


# ---------------------------------------------------------------------------------------------------- tests

@pytest.mark.parametrize("m", REORDER_M)
def test_reorder_equals_reference_kernel(m):
    from atom_b200 import ops
    x, idx = reorder_inputs(m)
    assert_same_as_reference(f"reorder.{m}", (x, idx), quant_outputs(ops.reorder_fp16_i4(x, idx), m))


@pytest.mark.parametrize("m", RMSNORM_M)
def test_rmsnorm_equals_reference_kernel(m):
    from atom_b200 import ops
    x, w, idx = rmsnorm_inputs(m)
    assert_same_as_reference(f"rmsnorm.{m}", (x, w, idx), quant_outputs(ops.rmsnorm_fp16_i4(x, w, idx, 1e-5), m))


@pytest.mark.parametrize("m", ACTIVATE_M)
def test_activate_equals_reference_kernel(m):
    from atom_b200 import ops
    a, b = activate_inputs(m)
    assert_same_as_reference(f"activate.{m}", (a, b), quant_outputs(ops.activate_fp16_i4(a, b), m))


@pytest.mark.parametrize("m,n,k,flags", GEMM_O16_CASES)
def test_gemm_o16_equals_reference_kernel(m, n, k, flags):
    from atom_b200 import ops
    t = gemm_o16_inputs(m, n, k)
    assert_same_as_reference(gemm_o16_key(m, n, k), t, {"d": ops.dense_layer_gemm_i4_fp16(*t, flags=flags)})


def test_gemm_o16_splitk_within_one_ulp_of_reference_kernel():
    from atom_b200 import ops
    t = gemm_splitk_inputs()
    check_inputs("gemm_o16_splitk", t)
    ours = ops.dense_layer_gemm_i4_fp16(*t, flags=0).float()
    ref = T(golden()["gemm_o16_splitk.d"]).float()
    assert torch.allclose(ours, ref, rtol=1e-3, atol=1e-3 * ref.abs().mean().item())
    assert (ours != ref).float().mean().item() < 0.02


@pytest.mark.parametrize("m,flags", GEMM_O4_CASES)
def test_gemm_o4_equals_reference_kernel(m, flags):
    from atom_b200 import ops
    t = gemm_o4_inputs(m)
    d, ds = ops.dense_layer_gemm_i4_o4(*t, flags=flags)
    assert_same_as_reference(f"gemm_o4.{m}", t, {"ds": ds, "d": d})


def test_batch_decode_at_least_as_close_to_the_oracle_as_the_reference_kernel():
    """Both kernels approximate transcendentals (the reference: __powf / __sincosf per element; ours: a rotation table and
    packed FP16 dequantisation), so neither is the other's bit pattern.  Judge both against the CPU oracle (float math,
    decode.cuh:480-689 restated): ours must meet rtol = atol = 5e-4 and must not be further from it than the reference is."""
    from atom_b200 import ops
    from tests.test_gpu_parity import _KV
    (data, param, indptr, indices, last), qn = decode_inputs()
    check_inputs("decode", (data, param, indptr, indices, last, qn))
    kv = _KV(data, param, indptr, indices, last)
    q = T(qn)
    for layer in range(DECODE_LAYERS):
        ours = ops.batch_decode_i4(q, kv, layer).float().cpu().numpy()
        ref = golden()["decode.o"][layer].astype(np.float32)
        orc = O.batch_decode_i4(qn, data, param, indptr, indices, last, layer).astype(np.float32)
        e_ours = (np.abs(ours - orc) - 5e-4 * np.abs(orc)).max()
        e_ref = (np.abs(ref - orc) - 5e-4 * np.abs(orc)).max()
        assert e_ours <= 5e-4, f"layer {layer}: ours exceeds 5e-4 by {e_ours:.2e} (reference kernel: {e_ref:.2e})"
        assert np.abs(ours - orc).max() <= max(np.abs(ref - orc).max() * 1.5, 2e-4), (np.abs(ours - orc).max(), np.abs(ref - orc).max())


def test_append_kv_equals_reference_kernel():
    from atom_b200 import ops
    from tests.test_gpu_parity import _KV
    fixture, (k, v, kp, vp) = append_kv_inputs()
    a = _KV(*fixture)
    ops.append_kv_i4(a, k, v, kp, vp, 1)
    assert_same_as_reference("append_kv", (*fixture, k, v, kp, vp), {"data": a.data, "param": a.param})
