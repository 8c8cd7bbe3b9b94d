"""Operator API -- mirrors /root/reference/e2e/punica-atom/punica/ops/__init__.py (names, argument order,
output allocation and return tuples) on top of the sm_100a kernels in libatom_b200.so.

Differences from the reference (all widening, none changes a result):
  * kernels run on torch's current CUDA stream (the reference uses the legacy default stream);
  * hidden_dim is any multiple of 128 (reference: 4096 for reorder/rmsnorm, 11008 for activate);
  * errors raise RuntimeError with the library's message instead of being silently ignored.
"""
import torch

from . import _lib

__all__ = [
    "batch_decode_i4", "append_kv_i4", "init_kv_i4", "activate_fp16_i4", "dense_layer_gemm_i4_fp16",
    "dense_layer_gemm_i4_o4", "rmsnorm_fp16_i4", "reorder_fp16_i4", "scale_size",
]

GEMM_AUTO, GEMM_NO_SPLITK, GEMM_FORCE_TALL, GEMM_FORCE_SKINNY = 0, 1, 2, 4
GEMM_SPLITK2, GEMM_SPLITK4 = 16, 32


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _req_cuda(*ts):
    for t in ts:
        if not (isinstance(t, torch.Tensor) and t.is_cuda):
            raise RuntimeError("atom_b200.ops: all tensors must live on a CUDA device (there is no CPU path)")
        if not t.is_contiguous():
            raise RuntimeError("atom_b200.ops: tensors must be contiguous")


def _req_width(what, **named):
    """Element-width checks (the C ABI takes raw pointers: a float32 tensor where float16 is meant would be silently
    misread).  Packed INT4 / INT8 operands may be int8 or uint8 views, so only the width is fixed for them."""
    for spec, t in named.items():
        name, width = spec.rsplit("_", 1)
        is_f16 = name.startswith("f16_")
        name = name[4:] if is_f16 else name
        ok = isinstance(t, torch.Tensor) and t.element_size() == int(width) and (not is_f16 or t.dtype == torch.float16)
        if not ok:
            raise RuntimeError(f"atom_b200.ops.{what}: `{name}` must be a tensor of {width}-byte elements"
                               f"{' (float16)' if is_f16 else ''}, got {getattr(t, 'dtype', type(t))}")


def scale_size(x):
    """ops/__init__.py:137-138"""
    return ((x) // 16 * 64 + 64 - (1 - (x % 16) // 8) * (8 - (x % 8)) * 8)


def _quant_outputs(bs, hidden_dim, device):
    group_size = 128
    o_outlier = torch.empty((bs, group_size), dtype=torch.int8, device=device)
    o_norms = torch.empty((bs, (hidden_dim - group_size) // 2), dtype=torch.int8, device=device)
    outlier_scales = torch.empty((scale_size(bs),), dtype=torch.float16, device=device)
    norm_scales = torch.empty((hidden_dim // group_size - 1, scale_size(bs)), dtype=torch.float16, device=device)
    return o_outlier, o_norms, outlier_scales, norm_scales


def reorder_fp16_i4(hidden_states, reorder_index):
    """ops/__init__.py:200-219"""
    _req_width("reorder_fp16_i4", f16_hidden_states_2=hidden_states, reorder_index_2=reorder_index)
    _req_cuda(hidden_states, reorder_index)
    bs, hidden_dim = hidden_states.shape
    out = _quant_outputs(bs, hidden_dim, hidden_states.device)
    with torch.cuda.device(hidden_states.device):
        _lib.check(_lib.lib().atom_reorder_fp16_i4(hidden_states.data_ptr(), reorder_index.data_ptr(), bs, hidden_dim,
                                                   out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                                   out[3].data_ptr(), _stream(hidden_states)), "reorder_fp16_i4")
    return out


def rmsnorm_fp16_i4(hidden_states, weight, reorder_index, eps):
    """ops/__init__.py:179-198.  `weight` may be fp32 (LlamaRMSNormInt4 keeps torch.ones fp32, llama.py:237); the
    reference reinterprets its storage as half -- here it is converted, which is what was meant."""
    if isinstance(weight, torch.Tensor) and weight.dtype != torch.float16:
        weight = weight.to(torch.float16)
    _req_width("rmsnorm_fp16_i4", f16_hidden_states_2=hidden_states, f16_weight_2=weight, reorder_index_2=reorder_index)
    _req_cuda(hidden_states, weight, reorder_index)
    bs, hidden_dim = hidden_states.shape
    out = _quant_outputs(bs, hidden_dim, hidden_states.device)
    with torch.cuda.device(hidden_states.device):
        _lib.check(_lib.lib().atom_rmsnorm_fp16_i4(hidden_states.data_ptr(), weight.data_ptr(), float(eps),
                                                   reorder_index.data_ptr(), bs, hidden_dim, out[0].data_ptr(),
                                                   out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(),
                                                   _stream(hidden_states)), "rmsnorm_fp16_i4")
    return out


def add_rmsnorm_fp16_i4(hidden_states, residual, weight, reorder_index, eps):
    """EXTENSION: (residual + hidden_states) and rmsnorm_fp16_i4 of the sum in one launch.  Returns (sum, 4-tuple);
    both bit-identical to `s = residual + hidden_states; rmsnorm_fp16_i4(s, ...)`."""
    if isinstance(weight, torch.Tensor) and weight.dtype != torch.float16:
        weight = weight.to(torch.float16)
    _req_width("add_rmsnorm_fp16_i4", f16_hidden_states_2=hidden_states, f16_residual_2=residual, f16_weight_2=weight,
               reorder_index_2=reorder_index)
    _req_cuda(hidden_states, residual, weight, reorder_index)
    if hidden_states.shape != residual.shape:
        raise RuntimeError("add_rmsnorm_fp16_i4: hidden_states and residual must have the same shape")
    bs, hidden_dim = hidden_states.shape
    out = _quant_outputs(bs, hidden_dim, hidden_states.device)
    s = torch.empty_like(hidden_states)
    with torch.cuda.device(hidden_states.device):
        _lib.check(_lib.lib().atom_add_rmsnorm_fp16_i4(hidden_states.data_ptr(), residual.data_ptr(), s.data_ptr(), weight.data_ptr(),
                                                       float(eps), reorder_index.data_ptr(), bs, hidden_dim, out[0].data_ptr(),
                                                       out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(),
                                                       _stream(hidden_states)), "add_rmsnorm_fp16_i4")
    return s, out


def activate_fp16_i4(a, b):
    """ops/__init__.py:141-157"""
    _req_width("activate_fp16_i4", f16_a_2=a, f16_b_2=b)
    _req_cuda(a, b)
    bs, hidden_dim = a.shape
    out = _quant_outputs(bs, hidden_dim, a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_activate_fp16_i4(a.data_ptr(), b.data_ptr(), bs, hidden_dim, out[0].data_ptr(),
                                                    out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(),
                                                    _stream(a)), "activate_fp16_i4")
    return out


def dense_layer_gemm_i4_fp16(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale, flags=GEMM_AUTO):
    """ops/__init__.py:160-168; dims as punica_ops.cc:236-237 (K = a.size(1)*2 + a_keeper.size(1))."""
    _req_width("dense_layer_gemm_i4_fp16", a_1=a, b_1=b, f16_a_scale_2=a_scale, f16_b_scale_2=b_scale, a_keeper_1=a_keeper,
               b_keeper_1=b_keeper, f16_a_keeper_scale_2=a_keeper_scale, f16_b_keeper_scale_2=b_keeper_scale)
    _req_cuda(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale)
    m, n = a.size(0), b.size(0)
    k = a.size(1) * 2 + a_keeper.size(1)
    d = torch.empty((m, n), dtype=torch.float16, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_gemm_i4_o16(a.data_ptr(), b.data_ptr(), a_scale.data_ptr(), b_scale.data_ptr(),
                                               a_keeper.data_ptr(), b_keeper.data_ptr(), a_keeper_scale.data_ptr(),
                                               b_keeper_scale.data_ptr(), d.data_ptr(), m, n, k, flags, _stream(a)),
                   "dense_layer_gemm_i4_fp16")
    return d


class ArHandle:
    """What the fused all-reduce entry points need of a comm.PushAllReduce: the device table of every rank's receive buffer, the
    local call-counter block, the slot size, and this rank's place in the group."""
    __slots__ = ("peer_ptrs", "state", "slot", "rank", "world")

    def __init__(self, peer_ptrs, state, slot, rank, world):
        self.peer_ptrs, self.state, self.slot, self.rank, self.world = int(peer_ptrs), state, int(slot), int(rank), int(world)


class PendingAllReduce:
    """Result of dense_layer_gemm_i4_fp16_push: the partial products sit in the receive buffers of all ranks; only
    reduce_add_rmsnorm_fp16_i4 (the very next consumer) can turn them into the all-reduced tensor."""
    __slots__ = ("ar", "shape", "device")

    def __init__(self, ar, shape, device):
        self.ar, self.shape, self.device = ar, tuple(shape), device


def dense_layer_gemm_i4_fp16_push(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale, ar, flags=GEMM_AUTO):
    """EXTENSION (tensor parallelism, decode batches M <= 64): dense_layer_gemm_i4_fp16 of a row-parallel shard whose epilogue pushes
    the FP16 partial into every rank's all-reduce receive buffer (csrc/comm_kernels.cuh).  Returns a PendingAllReduce."""
    _req_width("dense_layer_gemm_i4_fp16_push", a_1=a, b_1=b, f16_a_scale_2=a_scale, f16_b_scale_2=b_scale, a_keeper_1=a_keeper,
               b_keeper_1=b_keeper, f16_a_keeper_scale_2=a_keeper_scale, f16_b_keeper_scale_2=b_keeper_scale)
    _req_cuda(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale)
    m, n = a.size(0), b.size(0)
    k = a.size(1) * 2 + a_keeper.size(1)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_gemm_i4_o16_push(a.data_ptr(), b.data_ptr(), a_scale.data_ptr(), b_scale.data_ptr(),
                                                    a_keeper.data_ptr(), b_keeper.data_ptr(), a_keeper_scale.data_ptr(),
                                                    b_keeper_scale.data_ptr(), ar.peer_ptrs, ar.state.data_ptr(), ar.slot, ar.rank,
                                                    ar.world, m, n, k, flags, _stream(a)), "dense_layer_gemm_i4_fp16_push")
    return PendingAllReduce(ar, (m, n), a.device)


def reduce_add_rmsnorm_fp16_i4(pending, residual, weight, reorder_index, eps):
    """EXTENSION: add_rmsnorm_fp16_i4 whose `hidden_states` is the all-reduce of a PendingAllReduce, formed while the row is loaded.
    Returns (sum, 4-tuple), bit-identical to all-reducing first (rank-order FP32 sum, FP16 result) and calling add_rmsnorm_fp16_i4."""
    if isinstance(weight, torch.Tensor) and weight.dtype != torch.float16:
        weight = weight.to(torch.float16)
    _req_width("reduce_add_rmsnorm_fp16_i4", f16_residual_2=residual, f16_weight_2=weight, reorder_index_2=reorder_index)
    _req_cuda(residual, weight, reorder_index)
    if tuple(residual.shape) != pending.shape:
        raise RuntimeError("reduce_add_rmsnorm_fp16_i4: residual must have the shape of the pending all-reduce")
    bs, hidden_dim = residual.shape
    out = _quant_outputs(bs, hidden_dim, residual.device)
    s = torch.empty_like(residual)
    ar = pending.ar
    with torch.cuda.device(residual.device):
        _lib.check(_lib.lib().atom_reduce_add_rmsnorm_fp16_i4(ar.peer_ptrs, ar.state.data_ptr(), ar.slot, ar.rank, ar.world,
                                                              residual.data_ptr(), s.data_ptr(), weight.data_ptr(), float(eps),
                                                              reorder_index.data_ptr(), bs, hidden_dim, out[0].data_ptr(),
                                                              out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(),
                                                              _stream(residual)), "reduce_add_rmsnorm_fp16_i4")
    return s, out


def dense_layer_gemm_i4_o4(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale, flags=GEMM_AUTO):
    """ops/__init__.py:171-176"""
    _req_width("dense_layer_gemm_i4_o4", a_1=a, b_1=b, f16_a_scale_2=a_scale, f16_b_scale_2=b_scale, a_keeper_1=a_keeper,
               b_keeper_1=b_keeper, f16_a_keeper_scale_2=a_keeper_scale, f16_b_keeper_scale_2=b_keeper_scale)
    _req_cuda(a, b, a_scale, b_scale, a_keeper, b_keeper, a_keeper_scale, b_keeper_scale)
    m, n = a.size(0), b.size(0)
    k = a.size(1) * 2 + a_keeper.size(1)
    d = torch.empty((m, n // 2), dtype=torch.uint8, device=a.device)
    assert n % 128 == 0
    d_scale = torch.empty((m, n // 128 * 2), dtype=torch.float16, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_gemm_i4_o4(a.data_ptr(), b.data_ptr(), a_scale.data_ptr(), b_scale.data_ptr(),
                                              a_keeper.data_ptr(), b_keeper.data_ptr(), a_keeper_scale.data_ptr(),
                                              b_keeper_scale.data_ptr(), d.data_ptr(), d_scale.data_ptr(), m, n, k,
                                              flags, _stream(a)), "dense_layer_gemm_i4_o4")
    return d, d_scale


def dense_layer_gemm_i4_qkv(a, b_qkv, a_scale, b_scale_qkv, a_keeper, b_keeper_qkv, a_keeper_scale, b_keeper_scale_qkv, flags=GEMM_AUTO):
    """EXTENSION: q (fp16), k and v (o4) projections of one input over row-concatenated weights [3H, ...] in one launch for
    decode batches.  Returns (q, (k, k_scale), (v, v_scale)), bit-identical to the three separate operator calls."""
    _req_width("dense_layer_gemm_i4_qkv", a_1=a, b_qkv_1=b_qkv, f16_a_scale_2=a_scale, f16_b_scale_qkv_2=b_scale_qkv, a_keeper_1=a_keeper,
               b_keeper_qkv_1=b_keeper_qkv, f16_a_keeper_scale_2=a_keeper_scale, f16_b_keeper_scale_qkv_2=b_keeper_scale_qkv)
    _req_cuda(a, b_qkv, a_scale, b_scale_qkv, a_keeper, b_keeper_qkv, a_keeper_scale, b_keeper_scale_qkv)
    m, n3 = a.size(0), b_qkv.size(0)
    k = a.size(1) * 2 + a_keeper.size(1)
    if n3 % 384 != 0 or b_scale_qkv.numel() < (k // 128 - 1) * n3 or b_keeper_qkv.size(0) != n3:
        raise RuntimeError("dense_layer_gemm_i4_qkv: weights must be the row concatenation [q; k; v] with H % 128 == 0")
    h = n3 // 3
    q = torch.empty((m, h), dtype=torch.float16, device=a.device)
    kk = torch.empty((m, h // 2), dtype=torch.uint8, device=a.device)
    vv = torch.empty((m, h // 2), dtype=torch.uint8, device=a.device)
    ks = torch.empty((m, h // 128 * 2), dtype=torch.float16, device=a.device)
    vs = torch.empty((m, h // 128 * 2), dtype=torch.float16, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_gemm_i4_qkv(a.data_ptr(), b_qkv.data_ptr(), a_scale.data_ptr(), b_scale_qkv.data_ptr(),
                                               a_keeper.data_ptr(), b_keeper_qkv.data_ptr(), a_keeper_scale.data_ptr(),
                                               b_keeper_scale_qkv.data_ptr(), q.data_ptr(), kk.data_ptr(), ks.data_ptr(), vv.data_ptr(),
                                               vs.data_ptr(), m, h, k, flags, _stream(a)), "dense_layer_gemm_i4_qkv")
    return q, (kk, ks), (vv, vs)


def dense_layer_gemm_i4_gateup_act(a, b_gu, a_scale, b_scale_gu, a_keeper, b_keeper_gu, a_keeper_scale, b_keeper_scale_gu, flags=GEMM_AUTO):
    """EXTENSION: activate_fp16_i4(gate_proj(x), up_proj(x)) in one launch over row-concatenated weights [2I, ...] (decode
    batches, M <= 64).  Returns the activation 4-tuple, bit-identical to the three separate operator calls."""
    _req_width("dense_layer_gemm_i4_gateup_act", a_1=a, b_gu_1=b_gu, f16_a_scale_2=a_scale, f16_b_scale_gu_2=b_scale_gu, a_keeper_1=a_keeper,
               b_keeper_gu_1=b_keeper_gu, f16_a_keeper_scale_2=a_keeper_scale, f16_b_keeper_scale_gu_2=b_keeper_scale_gu)
    _req_cuda(a, b_gu, a_scale, b_scale_gu, a_keeper, b_keeper_gu, a_keeper_scale, b_keeper_scale_gu)
    m, n2 = a.size(0), b_gu.size(0)
    k = a.size(1) * 2 + a_keeper.size(1)
    if n2 % 256 != 0 or b_keeper_gu.size(0) != n2:
        raise RuntimeError("dense_layer_gemm_i4_gateup_act: weights must be the row concatenation [gate; up] with I % 128 == 0")
    inter = n2 // 2
    out = _quant_outputs(m, inter, a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().atom_gemm_i4_gateup_act(a.data_ptr(), b_gu.data_ptr(), a_scale.data_ptr(), b_scale_gu.data_ptr(),
                                                      a_keeper.data_ptr(), b_keeper_gu.data_ptr(), a_keeper_scale.data_ptr(),
                                                      b_keeper_scale_gu.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                                      out[3].data_ptr(), m, inter, k, flags, _stream(a)), "dense_layer_gemm_i4_gateup_act")
    return out


def _kv_dims(kv):
    # CHECK_DIM(6, kv_data) etc., punica_ops.cc:93-112
    if kv.data.dim() != 6 or kv.param.dim() != 6:
        raise RuntimeError("kv_data / kv_param must be 6-D [pages, L, 2, H, P, D]")
    if kv.data.dtype != torch.uint8 or kv.param.dtype != torch.float16:
        raise RuntimeError("kv_data must be uint8 and kv_param float16")
    if kv.data.size(5) * 2 != 128:
        raise RuntimeError("head_dim must be 128")
    return kv.data.size(1), kv.data.size(3), kv.data.size(4)


def batch_decode_i4(q, kv, layer_idx):
    """ops/__init__.py:21-32"""
    _req_cuda(q, kv.data, kv.param, kv.indptr, kv.indicies, kv.last_page_offset)
    L, H, P = _kv_dims(kv)
    if q.dim() != 3 or q.size(1) != H or q.size(2) != 128 or kv.indptr.size(0) != q.size(0) + 1 or \
            kv.last_page_offset.size(0) != q.size(0):
        raise RuntimeError("batch_decode_i4: shape mismatch")
    o = torch.empty(q.shape, dtype=q.dtype, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(_lib.lib().atom_batch_decode_i4(o.data_ptr(), q.data_ptr(), kv.data.data_ptr(), kv.param.data_ptr(),
                                                   kv.indptr.data_ptr(), kv.indicies.data_ptr(),
                                                   kv.last_page_offset.data_ptr(), L, layer_idx, H, P, q.size(0),
                                                   _stream(q)), "batch_decode_i4")
    return o


_rope_tables = {}


def rope_table(max_len, device):
    """(cos, sin)(pos * theta_i) for pos < max_len, i < 64, theta_i = 1e4^(-i/64), float32 [max_len, 64, 2] -- the factors of
    punica/models/llama.py:18-32 (`rotary_pos_emb`), computed the same way and cached per device."""
    size = max(256, 1 << (int(max_len) - 1).bit_length())
    key = (str(device), size)
    t = _rope_tables.get(key)
    if t is None:
        inv_freq = 1.0 / (10000 ** (torch.arange(0, 128, 2, device=device).float() / 128))
        freqs = torch.einsum("i,j->ij", torch.arange(0, size, device=device, dtype=torch.float32), inv_freq)
        t = torch.stack((freqs.cos(), freqs.sin()), dim=-1).contiguous()
        _rope_tables[key] = t
    return t


def prefill_attention_i4(q, k, k_param, v, v_param, seqlen_indptr, seqlens=None):
    """EXTENSION: causal prefill attention of every prompt over its own quantised K/V (the o4 projection outputs) with RoPE,
    one launch for all prompts and heads.  q f16 [T, H*128]; k, v u8 [T, H*64]; k_param, v_param f16 [T, H*2];
    seqlen_indptr i32 [B+1] (device); seqlens: the prompt lengths as host ints (avoids a device read).  Returns f16 [T, H*128]."""
    _req_width("prefill_attention_i4", f16_q_2=q, k_1=k, f16_k_param_2=k_param, v_1=v, f16_v_param_2=v_param)
    _req_cuda(q, k, k_param, v, v_param, seqlen_indptr)
    t, hd = q.shape
    h = hd // 128
    if hd % 128 or k.shape != (t, h * 64) or v.shape != k.shape or k_param.numel() != t * h * 2 or v_param.numel() != t * h * 2:
        raise RuntimeError("prefill_attention_i4: shape mismatch (head_dim must be 128)")
    if seqlens is None:
        ip = seqlen_indptr.cpu()
        seqlens = (ip[1:] - ip[:-1]).tolist()
    b, max_len = len(seqlens), max(seqlens)
    if sum(seqlens) != t or seqlen_indptr.numel() != b + 1:
        raise RuntimeError("prefill_attention_i4: seqlen_indptr does not cover the tokens")
    pos = torch.cat([torch.arange(n, dtype=torch.int32) for n in seqlens]).to(q.device, non_blocking=True)
    table = rope_table(max_len, q.device)
    kf, vf, out = torch.empty_like(q), torch.empty_like(q), torch.empty_like(q)
    with torch.cuda.device(q.device):
        _lib.check(_lib.lib().atom_prefill_attention_i4(q.data_ptr(), k.data_ptr(), k_param.data_ptr(), v.data_ptr(), v_param.data_ptr(),
                                                        seqlen_indptr.data_ptr(), pos.data_ptr(), table.data_ptr(), kf.data_ptr(),
                                                        vf.data_ptr(), out.data_ptr(), t, b, max_len, h, _stream(q)),
                   "prefill_attention_i4")
    return out


def init_kv_i4(kv, k, v, k_param, v_param, seqlen_indptr, layer_idx):
    """ops/__init__.py:35-46"""
    _req_cuda(kv.data, kv.param, kv.indptr, kv.indicies, kv.last_page_offset, k, v, k_param, v_param, seqlen_indptr)
    L, H, P = _kv_dims(kv)
    B = kv.last_page_offset.size(0)
    if kv.indptr.size(0) != B + 1 or seqlen_indptr.size(0) != B + 1:
        raise RuntimeError("init_kv_i4: indptr sizes do not match the batch")
    with torch.cuda.device(k.device):
        _lib.check(_lib.lib().atom_init_kv_i4(kv.data.data_ptr(), kv.param.data_ptr(), kv.indptr.data_ptr(),
                                              kv.indicies.data_ptr(), kv.last_page_offset.data_ptr(), k.data_ptr(),
                                              v.data_ptr(), k_param.data_ptr(), v_param.data_ptr(),
                                              seqlen_indptr.data_ptr(), k.size(0), L, layer_idx, H, P, B, _stream(k)),
                   "init_kv_i4")


def append_kv_i4(kv, k, v, k_param, v_param, layer_idx):
    """ops/__init__.py:49-59"""
    _req_cuda(kv.data, kv.param, kv.indptr, kv.indicies, kv.last_page_offset, k, v, k_param, v_param)
    L, H, P = _kv_dims(kv)
    B = k.size(0)
    if kv.indptr.size(0) != B + 1 or kv.last_page_offset.size(0) != B or k.shape != v.shape:
        raise RuntimeError("append_kv_i4: shape mismatch")
    with torch.cuda.device(k.device):
        _lib.check(_lib.lib().atom_append_kv_i4(kv.data.data_ptr(), kv.param.data_ptr(), kv.indptr.data_ptr(),
                                                kv.indicies.data_ptr(), kv.last_page_offset.data_ptr(), k.data_ptr(),
                                                v.data_ptr(), k_param.data_ptr(), v_param.data_ptr(), L, layer_idx, H,
                                                P, B, _stream(k)), "append_kv_i4")
