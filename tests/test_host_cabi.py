"""CPU suite: the C-ABI library loads and exports every symbol include/atom_b200.h declares; host-side helpers
(scale layout, KV page table) behave like the reference's.  No compute call is made (there is no GPU here)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from atom_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "atom_b200.h")).read()
    declared = set(re.findall(r"ATOM_API\s+[\w\s\*]+?\b(atom_\w+)\s*\(", hdr))
    assert declared == set(_lib.symbols()), declared ^ set(_lib.symbols())
    l = _lib.lib()
    for name in declared:
        assert hasattr(l, name)
    assert l.atom_version() >= 100


def test_scale_layout_host_functions_match_reference_formula():
    from atom_b200 import _lib, ops
    from oracle import oracle as O
    l = _lib.lib()
    for m in list(range(1, 100)) + [128, 1000, 4096]:
        assert l.atom_scale_size(m) == ops.scale_size(m) == O.scale_size(m)
        assert l.atom_scale_index(m - 1) == O.scale_index(m - 1)


def test_ops_reject_cpu_tensors_loudly():
    from atom_b200 import ops
    with pytest.raises(RuntimeError):
        ops.reorder_fp16_i4(torch.zeros(2, 4096, dtype=torch.float16), torch.arange(4096, dtype=torch.int16))


def test_kv_page_table_matches_reference_semantics():
    from atom_b200.kvcache import KvPoolInt4, KvCacheInt4, BatchedKvCacheInt4
    pool = KvPoolInt4(num_layers=2, num_heads=4, head_dim=128, capacity=20, block_len=16, device=torch.device("cpu"))
    assert pool.buf.shape == (20, 2, 2, 4, 16, 64) and pool.param.shape == (20, 2, 2, 4, 16, 2)
    cs = [KvCacheInt4(pool, n) for n in (1, 16, 17, 40)]
    assert [len(c.indicies) for c in cs] == [1, 1, 2, 3] and pool.num_free_blocks == 13
    b = BatchedKvCacheInt4(cs)
    assert b.indptr.tolist() == [0, 1, 2, 4, 7] and b.last_page_offset.tolist() == [1, 16, 1, 8] and b.page_size == 16
    cs[1].acquire_one()       # 16 -> 17 needs a new page
    assert len(cs[1].indicies) == 2 and cs[1].seqlen == 17
    cs[0].acquire_one()
    assert len(cs[0].indicies) == 1
    cs[3].release()
    assert pool.num_free_blocks == 15
    with pytest.raises(ValueError):
        KvCacheInt4(pool, -1)


def test_gemm_rejects_unknown_flag_bits_before_touching_the_device():
    """A flag bit the library does not know (512 selected a GEMM kernel that has been removed) fails loudly instead of
    quietly running another kernel.  The check comes before any device work, so dummy pointers suffice."""
    from atom_b200 import _lib
    l = _lib.lib()
    p = [0x10000 + 0x100 * i for i in range(9)]          # 16-byte aligned, never dereferenced
    rc = l.atom_gemm_i4_o16(*p, 16, 256, 512, 512, None)
    assert rc == -1                                       # ATOM_E_INVALID
    assert "flags" in l.atom_last_error().decode()


def test_ops_reject_wrong_element_types_before_touching_the_device():
    """The C ABI takes raw pointers: the Python mirror refuses tensors whose element width cannot be what the kernel reads."""
    from atom_b200 import ops
    h16, idx = torch.zeros(2, 256, dtype=torch.float16), torch.arange(256, dtype=torch.int16)
    with pytest.raises(RuntimeError, match="hidden_states.*2-byte.*float16"):
        ops.reorder_fp16_i4(h16.float(), idx)
    with pytest.raises(RuntimeError, match="reorder_index"):
        ops.reorder_fp16_i4(h16, idx.int())
    with pytest.raises(RuntimeError, match="`b`"):
        ops.activate_fp16_i4(h16, h16.float())
    a, s, kp = torch.zeros(2, 64, dtype=torch.int8), torch.zeros(64, dtype=torch.float16), torch.zeros(2, 128, dtype=torch.int8)
    with pytest.raises(RuntimeError, match="a_scale"):
        ops.dense_layer_gemm_i4_fp16(a, a, s.float(), s, kp, kp, s, s)
    with pytest.raises(RuntimeError, match="CUDA device"):          # widths fine -> the next gate is the device
        ops.dense_layer_gemm_i4_fp16(a.view(torch.uint8), a, s, s, kp, kp, s, s)
    with pytest.raises(RuntimeError, match="CUDA device"):          # bfloat16 has the right width but is not float16
        ops.rmsnorm_fp16_i4(h16, torch.ones(256), idx, 1e-6)        # fp32 norm weight is converted, as for the reference model
    with pytest.raises(RuntimeError, match="float16"):
        ops.rmsnorm_fp16_i4(h16.bfloat16(), torch.ones(256), idx, 1e-6)
