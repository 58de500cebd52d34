"""Python faces of the C-ABI kernels (raw ops; the autograd wiring lives in transformer.py / heads.py / rel_pos.py).

Every function here launches hand-written sm_100a kernels from libalm_b200.so on the current CUDA
stream.  No function has a CPU or stock-PyTorch implementation.
"""
from __future__ import annotations

import functools

import torch

from . import _lib

bf16 = torch.bfloat16
f32 = torch.float32


# ---- optional in-stream kernel timing (bench.py roofline): CUDA events bracket each tagged launch -----
_PROFILE = None
PROFILE_SHAPES = False  # per-shape GEMM classes (tools/profile_step.py)


def profile_start():
    """begin collecting (start_event, end_event, work) tuples per kernel class on the current stream."""
    global _PROFILE
    _PROFILE = {}


def profile_stop():
    """-> {cls: (total_ms, total_work, launches)}; synchronises the device."""
    global _PROFILE
    prof, _PROFILE = _PROFILE, None
    torch.cuda.synchronize()
    out = {}
    for cls, recs in (prof or {}).items():
        ms = sum(a.elapsed_time(b) for a, b, _ in recs)
        out[cls] = (ms, sum(w for _, _, w in recs), len(recs))
    return out


CLASS_UNIT = {}  # kernel class -> "flop" (tensor-bound classes) or "byte" (HBM-bound classes: algorithmic bytes)


class _timed:
    def __init__(self, cls, work, unit="flop"):
        self.cls, self.work = cls, work
        CLASS_UNIT[cls] = unit

    def __enter__(self):
        if _PROFILE is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if _PROFILE is not None:
            self.b.record()
            _PROFILE.setdefault(self.cls, []).append((self.a, self.b, self.work))
        return False


def _check_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.AlmError("audiolm_pytorch_b200 ops need CUDA tensors (no CPU fallback)")


def gemm(a, b, *, a_mn=False, b_mn=False, out=None, out_dtype=bf16, alpha=1.0, bias=None,
         acc_mode=0, split_k=1, cls="gemm_bf16_tcgen05"):
    """out[b,m,n] (op)= alpha * sum_k A(m,k) B(n,k) (+bias[n]).   bf16 operands, fp32 accumulate.

    a: [(batch,) M, K] (a_mn=False) or [(batch,) K, M] (a_mn=True); row stride must be a multiple of 8.
    b: [(batch,) N, K] (b_mn=False) or [(batch,) K, N] (b_mn=True).
    Reference counterpart: nn.Linear / einsum calls listed in include/alm_b200.h.
    """
    _check_cuda(a, b, out, bias)
    assert a.dtype == bf16 and b.dtype == bf16, "gemm operands must be bf16"
    batched = a.dim() == 3
    if not batched:
        a3, b3 = a.unsqueeze(0), b.unsqueeze(0)
    else:
        a3, b3 = a, b
    assert a3.stride(-1) == 1 and b3.stride(-1) == 1
    nb = a3.shape[0]
    assert b3.shape[0] == nb
    if a_mn:
        K, M = a3.shape[1], a3.shape[2]
    else:
        M, K = a3.shape[1], a3.shape[2]
    if b_mn:
        Kb, N = b3.shape[1], b3.shape[2]
    else:
        N, Kb = b3.shape[1], b3.shape[2]
    assert K == Kb, f"K mismatch {K} vs {Kb}"
    if out is None:
        out = torch.empty((nb, M, N) if batched else (M, N), device=a.device, dtype=out_dtype)
        assert acc_mode == 0
    o3 = out.unsqueeze(0) if out.dim() == 2 else out
    assert o3.shape == (nb, M, N) and o3.stride(-1) == 1
    assert o3.dtype in (bf16, f32)
    if bias is not None:
        assert bias.dtype == f32 and bias.numel() == N and bias.is_contiguous()
    if _PROFILE is not None and PROFILE_SHAPES:
        cls += f" M{M} N{N} K{K} b{nb} {'mn' if a_mn else 'k'}{'mn' if b_mn else 'k'} s{split_k}"
    with _timed(cls, 2.0 * M * N * K * nb):
        _lib.call(
            "alm_gemm_bf16",
            a3, int(a_mn), a3.stride(1), a3.stride(0) if nb > 1 else 0,
            b3, int(b_mn), b3.stride(1), b3.stride(0) if nb > 1 else 0,
            o3, int(o3.dtype == f32), o3.stride(1), o3.stride(0) if nb > 1 else 0,
            M, N, K, nb, float(alpha), bias, int(acc_mode), int(split_k),
        )
    return out


def _check_bias(bias, heads, n_q, n_k):
    """bias: fp32 [heads, n_q, ld] view with ld >= n_k, ld % 4 == 0 (see `pad_bias`)."""
    assert bias.dtype == f32 and bias.dim() == 3 and bias.shape[0] == heads and bias.shape[1] == n_q
    assert bias.shape[2] >= n_k and bias.stride(2) == 1 and bias.stride(1) % 4 == 0 and bias.stride(0) % 4 == 0
    return bias.stride(0), bias.stride(1)


def _ptr_array(tensors):
    import ctypes
    arr = (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


def embed_gather(src, tables, d):
    """src int32 [M, 2] ((table_id << 24) | row, -1 = none), tables: list of fp32 [rows_k, d] -> fp32 [M, d]"""
    _check_cuda(src, *tables)
    assert src.dtype == torch.int32 and src.is_contiguous() and src.shape[1] == 2
    assert all(t.dtype == f32 and t.is_contiguous() and t.shape[-1] == d for t in tables)
    M = src.shape[0]
    out = torch.empty(M, d, device=src.device, dtype=f32)
    import ctypes
    _lib.call("alm_embed_gather", ctypes.cast(_ptr_array(tables), ctypes.c_void_p), len(tables), src, out, M, d)
    return out


def embed_scatter(src, grad_tables, dout):
    """backward of embed_gather: grad_tables[id][row] += dout[m] (grad tables zeroed by the caller)"""
    _check_cuda(src, dout, *grad_tables)
    M, d = dout.shape
    assert dout.dtype == f32 and dout.is_contiguous()
    import ctypes
    _lib.call("alm_embed_scatter", ctypes.cast(_ptr_array(grad_tables), ctypes.c_void_p), len(grad_tables), src, dout,
              M, d)


class PackedKeyMask:
    """key mask in the bit layout the attention kernels read (alm_pack_key_mask): uint32 [b, 4 * ceil(n_k / 128)]"""

    def __init__(self, bits, n_k):
        self.bits, self.n_k = bits, n_k


def pack_key_mask(key_mask):
    """bool / uint8 [b, n_k] (True = attend) -> PackedKeyMask; pack once per forward and hand the result to every
    layer's mqa_attn_fwd / mqa_attn_bwd."""
    if key_mask is None or isinstance(key_mask, PackedKeyMask):
        return key_mask
    _check_cuda(key_mask)
    m = key_mask.to(torch.uint8).contiguous()
    b, n_k = m.shape
    bits = torch.empty(b, (n_k + 127) // 128 * 4, device=m.device, dtype=torch.int32)
    _lib.call("alm_pack_key_mask", m, bits, b, n_k)
    return PackedKeyMask(bits, n_k)


def mqa_attn_fwd(q, k, v, *, heads, key_mask=None, causal=True, scale=None, return_lse=True, bias=None):
    """Multi-query attention forward (attend.py:69-146).

    q: [b, n_q, heads*64] bf16 (last dim contiguous; may be a column slice of a wider buffer)
    k, v: [b, n_k, 64] bf16 (one shared head);  key_mask: [b, n_k] bool/uint8 (True = attend) or None.
    Queries are right-aligned against keys (query i sees keys <= i + n_k - n_q) when causal.
    bias: optional fp32 [heads, n_q, >=n_k] additive score bias shared by the batch (attend.py:122-124).
    Returns o [b, n_q, heads*64] bf16 and lse [b, heads, n_q] fp32.
    """
    _check_cuda(q, k, v, bias)
    assert q.dtype == bf16 and k.dtype == bf16 and v.dtype == bf16
    b, n_q, hd = q.shape
    n_k = k.shape[1]
    assert hd == heads * 64 and k.shape[-1] == 64 and v.shape[-1] == 64, "dim_head must be 64"
    assert q.stride(-1) == 1 and k.stride(-1) == 1 and v.stride(-1) == 1
    assert q.stride(0) == n_q * q.stride(1)
    o = torch.empty(b, n_q, hd, device=q.device, dtype=bf16)
    n_q_pad = (n_q + 127) // 128 * 128  # the backward stages lse rows with 512-B bulk copies
    lse = torch.empty(b, heads, n_q_pad, device=q.device, dtype=f32) if return_lse else None
    key_mask = pack_key_mask(key_mask)
    if key_mask is not None:
        assert key_mask.n_k == n_k and key_mask.bits.shape[0] == b
        key_mask = key_mask.bits
    if scale is None:
        scale = 64 ** -0.5
    # algorithmic FLOPs: QK^T + PV over the visible (lower-triangle) part only
    vis = (n_q * n_k - n_q * (n_q - 1) / 2) if causal else n_q * n_k
    bhs, brs = _check_bias(bias, heads, n_q, n_k) if bias is not None else (0, 0)
    with _timed("mqa_attn_fwd_tcgen05", 4.0 * b * heads * 64 * vis):
        _lib.call(
            "alm_mqa_attn_fwd",
            q, q.stride(1), k, k.stride(1), k.stride(0), v, v.stride(1), v.stride(0), key_mask,
            o, o.stride(1), lse, n_q_pad, bias, bhs, brs, b, heads, n_q, n_k, int(causal), float(scale),
        )
    return o, lse


def mqa_attn_bwd(q, k, v, o, d_o, lse, *, heads, key_mask=None, causal=True, scale=None, bias=None, dbias=None):
    """Backward of mqa_attn_fwd: returns dq [b,n_q,h*64], dk [b,n_k,64], dv [b,n_k,64] (bf16).

    lse is the padded [b, heads, n_q_pad] tensor returned by the forward.  With a bias, d(bias) is ACCUMULATED
    into `dbias` (fp32, same shape/strides as `bias`; the caller zeroes it once per step).
    """
    _check_cuda(q, k, v, o, d_o, lse, bias, dbias)
    b, n_q, hd = q.shape
    n_k = k.shape[1]
    n_q_pad = lse.shape[-1]
    assert d_o.dtype == bf16 and d_o.stride(-1) == 1 and o.stride(-1) == 1
    assert d_o.stride(0) == n_q * d_o.stride(1)
    delta = torch.empty(b, heads, n_q_pad, device=q.device, dtype=f32)
    _lib.call("alm_attn_delta", o, o.stride(1), d_o, d_o.stride(1), delta, n_q_pad, b, heads, n_q)
    key_mask = pack_key_mask(key_mask)
    if key_mask is not None:
        assert key_mask.n_k == n_k
        key_mask = key_mask.bits
    if scale is None:
        scale = 64 ** -0.5
    dq = torch.empty(b, n_q, hd, device=q.device, dtype=bf16)
    dk = torch.empty(b, n_k, 64, device=q.device, dtype=bf16)
    dv = torch.empty(b, n_k, 64, device=q.device, dtype=bf16)
    bhs, brs = _check_bias(bias, heads, n_q, n_k) if bias is not None else (0, 0)
    if dbias is not None:
        assert bias is not None and dbias.dtype == f32 and dbias.shape == bias.shape and dbias.stride() == bias.stride()
    vis = (n_q * n_k - n_q * (n_q - 1) / 2) if causal else n_q * n_k
    with _timed("mqa_attn_bwd_tcgen05", 10.0 * b * heads * 64 * vis):  # 5 matmuls (algorithmic; 7 executed)
        _lib.call(
            "alm_mqa_attn_bwd",
            q, q.stride(1), k, k.stride(1), k.stride(0), v, v.stride(1), v.stride(0), d_o, d_o.stride(1), key_mask,
            lse, delta, n_q_pad, dq, dq.stride(1), dk, dk.stride(1), dv, dv.stride(1),
            bias, dbias, bhs, brs, b, heads, n_q, n_k, int(causal), float(scale),
        )
    return dq, dk, dv


def gemv(x, w, *, out_dtype=bf16, bias=None):
    """x [rows <= 8, K] bf16, w [N, >=K (zero padded to a multiple of 8)] bf16 -> [rows, N] (decode-step Linear)."""
    _check_cuda(x, w, bias)
    rows, K = x.shape
    N = w.shape[0]
    assert x.dtype == bf16 and w.dtype == bf16 and x.stride(1) == 1 and w.stride(1) == 1 and rows <= 8
    assert w.shape[1] >= K and w.shape[1] % 8 == 0
    out = torch.empty(rows, N, device=x.device, dtype=out_dtype)
    _lib.call("alm_gemv_bf16", x, x.stride(0), w, w.stride(0), out, int(out_dtype == f32), out.stride(0),
              None if bias is None else bias.float().contiguous(), rows, N, K)
    return out


def kv_append(kv_new, k_cache, v_cache, cache_len):
    """k_cache[b, len] = kv_new[b, :64]; v_cache[b, len] = kv_new[b, 64:]  (len: int32 device scalar)."""
    _check_cuda(kv_new, k_cache, v_cache, cache_len)
    b, max_len, dh = k_cache.shape
    assert dh == 64 and v_cache.shape == k_cache.shape and kv_new.shape == (b, 128) and kv_new.dtype == bf16
    assert k_cache.dtype == bf16 and v_cache.dtype == bf16 and cache_len.dtype == torch.int32
    assert k_cache.stride(1) == 64 and v_cache.stride() == k_cache.stride() and kv_new.stride(1) == 1
    _lib.call("alm_kv_append", kv_new, kv_new.stride(0), k_cache, v_cache, k_cache.stride(0), cache_len, max_len, b)


def mqa_attn_decode(q, k_cache, v_cache, cache_len, *, heads, key_mask=None, scale=None, splits=None):
    """one new query per sequence against the static cache: q [b, heads*64] bf16 -> o [b, heads*64] bf16.
    Attends keys 0..cache_len (inclusive: the new token has just been appended at position cache_len)."""
    _check_cuda(q, k_cache, v_cache, cache_len, key_mask)
    b, max_len, _ = k_cache.shape
    assert q.shape == (b, heads * 64) and q.dtype == bf16 and q.stride(1) == 1
    o = torch.empty(b, heads * 64, device=q.device, dtype=bf16)
    if key_mask is not None:
        assert key_mask.dtype == torch.uint8 and key_mask.shape[0] == b and key_mask.shape[1] >= max_len
    if splits is None:  # enough CTAs to spread a long cache over the SMs, fixed per cache size (static launch)
        splits = max(1, min(32, max_len // 128, 148 // max(1, b)))
    ws = torch.empty(b, splits, heads, 66, device=q.device, dtype=f32) if splits > 1 else None
    _lib.call("alm_mqa_attn_decode", q, q.stride(0), k_cache, v_cache, k_cache.stride(0), cache_len, max_len, key_mask,
              0 if key_mask is None else key_mask.stride(0), o, o.stride(0), ws, splits, b, heads,
              float(64 ** -0.5 if scale is None else scale))
    return o


def head_ce_fwd(x, w, bias, labels, ignore_index):
    """fused logit head + cross entropy, forward: x [M, K] bf16, w [V, >=K] bf16 (+ bias [V] fp32), labels [M] int64
    -> (lse [M] fp32, loss_rows [M] fp32 = lse - logit[label], 0 where label == ignore_index).  No logits in HBM."""
    _check_cuda(x, w, bias, labels)
    M, K = x.shape
    V = w.shape[0]
    assert x.dtype == bf16 and w.dtype == bf16 and x.stride(1) == 1 and w.stride(1) == 1 and w.shape[1] >= K
    assert labels.dtype == torch.int64 and labels.is_contiguous() and labels.numel() == M
    tiles = int(_lib.load().alm_gemm_head_ce_tiles(V))
    part = torch.empty(M, tiles, 2, device=x.device, dtype=f32)
    lab = torch.empty(M, device=x.device, dtype=f32)
    lse = torch.empty(M, device=x.device, dtype=f32)
    rows = torch.empty(M, device=x.device, dtype=f32)
    with _timed("gemm_head_ce_fused", 2.0 * M * V * K):
        _lib.call("alm_gemm_head_ce", x, x.stride(0), w, w.stride(0), bias, labels, int(ignore_index), 1, part, lab, None,
                  None, None, None, 0, M, V, K)
    _lib.call("alm_ce_finish", part, tiles, lab, labels, int(ignore_index), lse, rows, M)
    return lse, rows


def head_ce_bwd(x, w, bias, labels, ignore_index, lse, scale_num, scale_den, dlogits):
    """fused logit head + cross entropy, backward: recomputes the logits tile by tile and writes
    dlogits [M, >=V] bf16 = (softmax - onehot) * scale_num / scale_den (device scalars), zero rows where ignored."""
    _check_cuda(x, w, bias, labels, lse, scale_num, scale_den, dlogits)
    M, K = x.shape
    V = w.shape[0]
    assert dlogits.dtype == bf16 and dlogits.shape[0] == M and dlogits.shape[1] >= V and dlogits.stride(1) == 1
    assert scale_num.dtype == f32 and scale_den.dtype == f32 and lse.dtype == f32
    # the recomputation is executed work, not algorithmic work: timed in the fused-head class with 0 algorithmic FLOPs
    with _timed("gemm_head_ce_fused", 0.0):
        _lib.call("alm_gemm_head_ce", x, x.stride(0), w, w.stride(0), bias, labels, int(ignore_index), 2, None, None, lse,
                  scale_num, scale_den, dlogits, dlogits.stride(0), M, V, K)
    return dlogits


DECODE_STEP_MAX_ROWS = 4


def decode_stack_scratch(b, d, heads, inner, device):
    """workspace of alm_decode_stack_step (barrier counter + error flag + the vectors that cross its barriers)."""
    n = int(_lib.load().alm_decode_stack_scratch_bytes(b, d, heads, inner))
    if n <= 0:
        raise _lib.AlmError(f"alm_decode_stack_step does not take b={b}, d={d}, heads={heads}, inner={inner}")
    return torch.zeros(n, device=device, dtype=torch.uint8)


def decode_stack_grid():
    """CTAs of the one-kernel decode step (= SMs); the engine regroups its operands for this count."""
    return int(_lib.load().alm_decode_stack_grid())


def regroup_rows(w, grid):
    """[N, K] -> [grid * pc, K] with row (c * pc + l) = w[c + l * grid] (zeros past N): CTA c's rows become contiguous."""
    N, K = w.shape
    pc = -(-N // grid)
    wp = torch.zeros(pc * grid, K, device=w.device, dtype=w.dtype)
    wp[:N] = w
    return wp.view(pc, grid, K).transpose(0, 1).contiguous().view(grid * pc, K)


def decode_stack_step(table, x, out, final_gamma, cache_len, k_cache, key_mask, scratch, *, heads, inner, grid,
                      value_residual=True, scale=None):
    """the whole hyper-connection stack for ONE new token per sequence in one cooperative kernel.
    table: int64 [L, 24] device pointers (see include/alm_b200.h); x fp32 [b, d]; out bf16 [b, d];
    k_cache: [L, b, max_len, 64] (only its strides / max_len are read here; the table holds the per-layer bases).
    Increments cache_len on the device."""
    _check_cuda(table, x, out, final_gamma, cache_len, key_mask, scratch)
    L, b, max_len, dh = k_cache.shape
    d = x.shape[1]
    assert table.dtype == torch.int64 and table.shape == (L, 24) and table.is_contiguous()
    assert x.dtype == f32 and x.is_contiguous() and out.dtype == bf16 and out.is_contiguous() and x.shape == (b, d)
    assert dh == 64 and k_cache.stride(2) == 64 and cache_len.dtype == torch.int32 and final_gamma.dtype == f32
    if key_mask is not None:
        assert key_mask.dtype == torch.uint8 and key_mask.shape[0] == b and key_mask.shape[1] >= max_len
    _lib.call("alm_decode_stack_step", table, L, x, out, final_gamma, cache_len, max_len, k_cache.stride(1), key_mask,
              0 if key_mask is None else key_mask.stride(0), scratch, scratch.numel(), b, d, heads, inner,
              int(bool(value_residual)), float(64 ** -0.5 if scale is None else scale), grid)
    return out


def bias_gather_fwd(table, idx, override, *, ld=None):
    """table [P, H] fp32, idx [n_q, n_k] int32 (-1 = override), override [H] fp32 or None -> bias [H, n_q, ld] fp32."""
    _check_cuda(table, idx, override)
    assert table.dtype == f32 and table.is_contiguous() and idx.dtype == torch.int32 and idx.is_contiguous()
    H = table.shape[1]
    n_q, n_k = idx.shape
    ld = (n_k + 3) // 4 * 4 if ld is None else ld
    out = torch.empty(H, n_q, ld, device=table.device, dtype=f32)
    _lib.call("alm_bias_gather_fwd", table, idx, None if override is None else override.contiguous(), out, H, n_q,
              n_k, ld)
    return out


def bias_gather_bwd(dbias, idx, table_rows, *, want_override):
    """scatter-add of d(bias) [H, n_q, ld] back to the table rows / the per-head override scalar."""
    _check_cuda(dbias, idx)
    assert dbias.dtype == f32 and dbias.is_contiguous()
    H, n_q, ld = dbias.shape
    n_k = idx.shape[1]
    dtable = torch.zeros(table_rows, H, device=dbias.device, dtype=f32)
    dover = torch.zeros(H, device=dbias.device, dtype=f32) if want_override else None
    _lib.call("alm_bias_gather_bwd", dbias, idx, dtable, dover, H, n_q, n_k, ld)
    return dtable, dover


HC_AUX = 54  # floats of per-token state kept for the backward (see csrc/hyper_conn.cu)


@functools.lru_cache(maxsize=None)
def _sm_count(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


def _hc_param_ptrs(hc, ln_gamma):
    return (hc["gamma"], hc["dyn_alpha"], hc["dyn_beta"], hc["static_alpha"], hc["static_beta"],
            hc["alpha_scale"], hc["beta_scale"], ln_gamma)


def hc_pre_fwd(hc, ln_gamma, *, R_in=None, Y=None, beta_prev=None, x_expand=None, M, d, streams=4):
    """depth(prev branch) + width(this branch) + pre-LayerNorm.  hc: dict of fp32 HC params.

    Returns R_out [M,S,d] bf16, bin [M,d] bf16, xn [M,d] bf16, beta [M,S] f32, aux [M,30] f32.
    """
    dev = ln_gamma.device
    R_out = torch.empty(M, streams, d, device=dev, dtype=bf16)
    bin_ = torch.empty(M, d, device=dev, dtype=bf16)
    xn = torch.empty(M, d, device=dev, dtype=bf16)
    beta = torch.empty(M, streams, device=dev, dtype=f32)
    aux = torch.empty(M, HC_AUX, device=dev, dtype=f32)
    with _timed("hc_pre_fwd", M * d * ((4 if x_expand is not None else 10) + 12), "byte"):
        _lib.call("alm_hc_pre_fwd", R_in, Y, beta_prev, x_expand, *_hc_param_ptrs(hc, ln_gamma),
                  R_out, bin_, xn, beta, aux, M, d, streams)
    return R_out, bin_, xn, beta, aux


def hc_pre_bwd(hc, ln_gamma, grads, g_ln_gamma, aux, dR_out, dxn, dbeta, *, dbin_extra=None, R_in=None, Y=None,
               beta_prev=None, x_expand=None, dx_scale=1.0, M, d, streams=4):
    """Backward of hc_pre_fwd.  `grads`: dict of fp32 accumulators shaped like `hc` (added to; for d <= 1024 in a
    fixed order, so the parameter gradients are bitwise reproducible).

    Returns (dR_in, dY, dbeta_prev) or dx_expand [M,d] f32 when the op expanded the streams.
    """
    dev = ln_gamma.device
    if x_expand is not None:
        dx = torch.empty(M, d, device=dev, dtype=f32)
        dR_in = dY = dbp = None
    else:
        dx = None
        dR_in = torch.empty(M, streams, d, device=dev, dtype=bf16)
        dY = torch.empty(M, d, device=dev, dtype=bf16)
        dbp = torch.empty(M, streams, device=dev, dtype=f32)
    # per-CTA parameter-gradient partial sums of the d <= 1024 kernel (at most 3 CTAs per SM), reduced in a fixed order
    blocks = 3 * _sm_count(dev)
    partial = torch.empty(blocks * (8 * d + 32), device=dev, dtype=f32) if d <= 1024 else None
    nbytes = M * d * ((4 + 8 + 2 + 4 if x_expand is not None else 8 + 2 + 8 + 2 + 8 + 2) + (2 if dbin_extra is not None else 0))
    with _timed("hc_pre_bwd", nbytes, "byte"):
        _lib.call("alm_hc_pre_bwd", R_in, Y, beta_prev, x_expand, *_hc_param_ptrs(hc, ln_gamma), aux, dR_out, dxn,
                  dbin_extra, dbeta, dR_in, dY, dbp, dx, float(dx_scale),
                  grads["gamma"], grads["dyn_alpha"], grads["dyn_beta"], grads["static_alpha"], grads["static_beta"],
                  grads["alpha_scale"], grads["beta_scale"], g_ln_gamma, partial, blocks, M, d, streams)
    return dx if x_expand is not None else (dR_in, dY, dbp)


def hc_post_fwd(R_in, Y, beta_prev, ln_gamma, *, M, d, streams=4):
    out = torch.empty(M, d, device=R_in.device, dtype=bf16)
    stats = torch.empty(M, 2, device=R_in.device, dtype=f32)
    _lib.call("alm_hc_post_fwd", R_in, Y, beta_prev, ln_gamma, out, stats, M, d, streams)
    return out, stats


def hc_post_bwd(R_in, Y, beta_prev, ln_gamma, stats, dout, g_ln_gamma, *, M, d, streams=4):
    dR_in = torch.empty(M, streams, d, device=R_in.device, dtype=bf16)
    dY = torch.empty(M, d, device=R_in.device, dtype=bf16)
    dbp = torch.empty(M, streams, device=R_in.device, dtype=f32)
    _lib.call("alm_hc_post_bwd", R_in, Y, beta_prev, ln_gamma, stats, dout, dR_in, dY, dbp, g_ln_gamma, M, d, streams)
    return dR_in, dY, dbp


def geglu_ln_fwd(h, gamma, *, inner, inner_pad):
    """h [M, 2*inner_pad] bf16 (a | gate) -> gn [M, inner_pad] bf16 = LN(gelu(gate)*a)*gamma, stats [M,2]."""
    M = h.shape[0]
    gn = torch.empty(M, inner_pad, device=h.device, dtype=bf16)
    stats = torch.empty(M, 2, device=h.device, dtype=f32)
    with _timed("geglu_ln_fwd", M * inner_pad * 6, "byte"):
        _lib.call("alm_geglu_ln_fwd", h, h.stride(0), inner_pad, gamma, gn, gn.stride(0), stats, M, inner, inner_pad)
    return gn, stats


def geglu_ln_bwd(h, gamma, stats, dgn, g_gamma, *, inner, inner_pad):
    M = h.shape[0]
    dh = torch.empty_like(h)
    assert dh.stride(0) == h.stride(0)
    with _timed("geglu_ln_bwd", M * inner_pad * 10, "byte"):
        _lib.call("alm_geglu_ln_bwd", h, h.stride(0), inner_pad, gamma, stats, dgn, dgn.stride(0), dh, g_gamma, M,
                  inner, inner_pad)
    return dh


def ce_fwd_bwd(logits, labels, *, ignore_index=-1, scale_num=None, scale_den=None, want_grad=True):
    """logits [R, V] f32 (row stride free), labels [R] int64 -> loss_rows [R] f32, dlogits [R, Vpad] bf16."""
    R, V = logits.shape
    Vpad = (V + 7) // 8 * 8
    loss_rows = torch.empty(R, device=logits.device, dtype=f32)
    dlogits = torch.empty(R, Vpad, device=logits.device, dtype=bf16) if want_grad else None
    _lib.call("alm_ce_fwd_bwd", logits, logits.stride(0), labels, int(ignore_index), loss_rows, dlogits,
              Vpad, scale_num, scale_den, R, V, Vpad)
    return loss_rows, dlogits


def axpby(x, alpha, y, beta, out=None):
    """out = alpha*x + beta*y on 2-D bf16 views (last dim contiguous)."""
    rows, cols = x.shape
    if out is None:
        out = torch.empty(rows, cols, device=x.device, dtype=bf16)
    _lib.call("alm_axpby_bf16", x, x.stride(0), float(alpha), y, y.stride(0) if y is not None else 0, float(beta),
              out, out.stride(0), rows, cols)
    return out


def cast_pad(src, cols_pad=None, out=None):
    """fp32 [R, C] (last dim contiguous) -> bf16 [R, cols_pad] zero padded."""
    rows, cols = src.shape
    cols_pad = cols if cols_pad is None else cols_pad
    if out is None:
        out = torch.empty(rows, cols_pad, device=src.device, dtype=bf16)
    _lib.call("alm_cast_pad_bf16", src, src.stride(0), out, out.stride(0), rows, cols, cols_pad)
    return out


def cast_pad_multi(desc):
    """desc: device int64 [n, 7] rows {src ptr, dst ptr, rows, cols, cols_pad, lds, ldd}: all casts in one launch"""
    _check_cuda(desc)
    assert desc.dtype == torch.int64 and desc.is_contiguous() and desc.shape[1] == 7
    _lib.call("alm_cast_pad_multi", desc, desc.shape[0])


def scale_by_scalar(x, s):
    _lib.call("alm_scale_by_scalar_bf16", x, s, x.numel())
    return x


# ---- SoundStream codec -------------------------------------------------------------------------------
PAD_MODES = {"reflect": 0, "constant": 1, "zeros": 1, "replicate": 2}


# (K, stride, dilation) shapes with a register-tiled specialisation (csrc/conv_tiled.cuh)
CONV_TILED_SHAPES = {(7, 1, 1), (7, 1, 3), (7, 1, 9), (1, 1, 1), (3, 1, 1), (4, 2, 1), (6, 3, 1), (8, 4, 1), (10, 5, 1),
                     (16, 8, 1)}


def causal_conv1d(x, weight, bias=None, *, stride=1, dilation=1, pad_mode="reflect", elu=False, residual=None,
                  weight_packed=None):
    """CausalConv1d forward (soundstream.py:332-345) with optional fused ELU and skip add. fp32 [B,C,T].

    weight [Cout, Cin, K] (torch layout); weight_packed: optional cached copy [Cin, K, Cout] (weight.permute(1, 2, 0))
    that lets the register-tiled kernel stage weights with coalesced loads."""
    _check_cuda(x, weight, bias, residual, weight_packed)
    assert x.dtype == f32 and weight.dtype == f32
    x = x.contiguous()
    B, Cin, T = x.shape
    Cout, Cin_w, K = weight.shape
    assert Cin_w == Cin, "groups != 1 is not supported"
    pad = dilation * (K - 1) + 1 - stride
    Tout = (T + pad - dilation * (K - 1) - 1) // stride + 1
    y = torch.empty(B, Cout, Tout, device=x.device, dtype=f32)
    if residual is not None:
        residual = residual.contiguous()
        assert residual.shape == y.shape
    packed = weight_packed is not None and (K, stride, dilation) in CONV_TILED_SHAPES
    if packed:
        assert weight_packed.shape == (Cin, K, Cout) and weight_packed.is_contiguous() and weight_packed.dtype == f32
    cls = "causal_conv1d"
    if _PROFILE is not None and PROFILE_SHAPES:
        cls += f" Cin{Cin} Cout{Cout} K{K} s{stride} d{dilation} T{T}"
    with _timed(cls, 2.0 * B * Cout * Tout * Cin * K):
        _lib.call("alm_causal_conv1d_fwd", x, weight_packed if packed else weight.contiguous(),
                  None if bias is None else bias.contiguous(), residual, y, B, Cin, Cout, T, K, stride, dilation,
                  PAD_MODES[pad_mode], int(elu), int(packed))
    return y


RU_FUSED_CHANNELS = {32, 64, 128, 256}
RU_FUSED_DILATIONS = {1, 3, 9}


def residual_unit(x, w7_packed, b7, w1_packed, b1, *, dilation, pad_mode="reflect"):
    """fused ResidualUnit forward (soundstream.py:362-369); packed weights [C,7,C] / [C,1,C], fp32 [B,C,T]."""
    _check_cuda(x, w7_packed, b7, w1_packed, b1)
    x = x.contiguous()
    B, C, T = x.shape
    assert w7_packed.shape == (C, 7, C) and w1_packed.shape == (C, 1, C) and x.dtype == f32
    y = torch.empty_like(x)
    with _timed("residual_unit_fused", 2.0 * B * C * T * C * 8):
        _lib.call("alm_residual_unit_fwd", x, w7_packed, b7.contiguous(), w1_packed, b1.contiguous(), y, B, C, T,
                  dilation, PAD_MODES[pad_mode])
    return y


def causal_conv_transpose1d(x, weight, bias=None, *, stride):
    """CausalConvTranspose1d forward (soundstream.py:347-360): weight [Cin, Cout, 2*stride]."""
    _check_cuda(x, weight, bias)
    x = x.contiguous()
    B, Cin, n = x.shape
    Cin_w, Cout, K = weight.shape
    assert Cin_w == Cin and K == 2 * stride
    y = torch.empty(B, Cout, n * stride, device=x.device, dtype=f32)
    _lib.call("alm_causal_convT1d_fwd", x, weight.contiguous(), None if bias is None else bias.contiguous(), y, B,
              Cin, Cout, n, stride)
    return y


# ---- SoundStream encoder on the tensor cores (csrc/codec_tc.cu) ---------------------------------------
def c8s_pack(x, phases=1):
    """fp32 [B, C, T] -> C8S bf16 [B, 2C/8, P, T/P, 8] (torch ops; boundaries and tests only)."""
    B, C, T = x.shape
    assert C % 8 == 0 and T % phases == 0
    hi = x.to(bf16)
    lo = (x - hi.float()).to(bf16)

    def arr(t):
        return t.reshape(B, C // 8, 8, T // phases, phases).permute(0, 1, 4, 3, 2)

    return torch.cat((arr(hi), arr(lo)), dim=1).contiguous()


def c8s_unpack(a):
    """C8S bf16 [B, 2C/8, P, T/P, 8] -> fp32 [B, C, T]."""
    B, nch2, P, Tp, _ = a.shape
    nch = nch2 // 2
    v = a[:, :nch].float() + a[:, nch:].float()
    return v.permute(0, 1, 4, 3, 2).reshape(B, nch * 8, Tp * P)


def _split_units(w, bn=None):
    """w fp32 [Cout, Cin, K] -> bf16 [K, Cin/16, 2 (hi, lo), 2, Cout, 8] (optionally tiled over Cout by bn)."""
    Cout, Cin, K = w.shape
    assert Cin % 16 == 0
    hi = w.to(bf16)
    lo = (w - hi.float()).to(bf16)

    def arr(t):
        return t.permute(2, 1, 0).reshape(K, Cin // 16, 2, 8, Cout).permute(0, 1, 2, 4, 3)

    st = torch.stack((arr(hi), arr(lo)), dim=2)                      # [K, kk, part, cc, Cout, 8]
    if bn is not None:
        st = st.reshape(K, Cin // 16, 2, 2, Cout // bn, bn, 8).permute(4, 0, 1, 2, 3, 5, 6)
    return st.contiguous()


def pack_ru_weights(w7, w1):
    """ResidualUnit weights [C, C, 7], [C, C, 1] -> the unit layout alm_codec_ru_tc streams (tap 7 = the 1x1 conv)."""
    return _split_units(torch.cat((w7.detach().float(), w1.detach().float()), dim=2))


def conv_tc_bn(cout):
    return 256 if cout % 256 == 0 else (128 if cout % 128 == 0 else 64)


def pack_conv_weights(w):
    return _split_units(w.detach().float(), bn=conv_tc_bn(w.shape[0]))


def pack_convT_weights(w, stride):
    """CausalConvTranspose1d weight [Cin, Cout, 2s] -> (units for alm_codec_conv_tc, Cout' = s * Cout): the transposed conv
    is the 2-tap causal conv  out[i, (r, o)] = W[c, o, r + s] x[i - 1, c] + W[c, o, r] x[i, c]  (soundstream.py:347-360)."""
    cin, cout, k = w.shape
    assert k == 2 * stride
    wf = w.detach().float()
    taps = torch.stack((wf[..., stride:], wf[..., :stride]), dim=-1)          # [c, o, r, j]: j = 0 -> x[i-1], 1 -> x[i]
    wp = taps.permute(2, 1, 0, 3).reshape(stride * cout, cin, 2)               # [(r, o), c, j]
    return pack_conv_weights(wp)


def codec_pack_c8s(x):
    """fp32 channels-last [B, n, C] -> C8S [B, 2C/8, 1, n, 8] (entry of the tensor-core decoder)."""
    _check_cuda(x)
    B, n, C = x.shape
    x = x.to(f32).contiguous()
    y = torch.empty(B, 2 * C // 8, 1, n, 8, device=x.device, dtype=bf16)
    _lib.call("alm_codec_pack_c8s", x, y, B, n, C)
    return y


def codec_last_conv(x, weight, bias, *, pad_mode="reflect"):
    """CausalConv1d(Cin, 1, K) on C8S (P = 1) -> fp32 [B, 1, T] (soundstream.py:626)."""
    _check_cuda(x, weight, bias)
    B, nch2, P, T, _ = x.shape
    assert P == 1 and weight.shape[0] == 1 and weight.shape[1] == nch2 * 4
    y = torch.empty(B, 1, T, device=x.device, dtype=f32)
    with _timed("codec_last_conv", 4.0 * B * T * (nch2 * 4 + 1), "byte"):
        _lib.call("alm_codec_last_conv", x, weight.detach().contiguous(),
                  None if bias is None else bias.detach().contiguous(), y, B, T, nch2 * 4, weight.shape[2],
                  PAD_MODES[pad_mode])
    return y


def codec_first_conv(wave, weight, bias, *, pad_mode="reflect"):
    """CausalConv1d(1, Cout, K) on fp32 [B, T] -> C8S [B, 2Cout/8, 1, T, 8] (soundstream.py:520)."""
    _check_cuda(wave, weight, bias)
    B, T = wave.shape
    Cout, cin, K = weight.shape
    assert cin == 1 and wave.dtype == f32
    y = torch.empty(B, 2 * Cout // 8, 1, T, 8, device=wave.device, dtype=bf16)
    with _timed("codec_first_conv", (B * T * 4 + B * Cout * T * 4), "byte"):
        _lib.call("alm_codec_first_conv", wave.contiguous(), weight.detach().contiguous(),
                  None if bias is None else bias.detach().contiguous(), y, B, T, Cout, K, PAD_MODES[pad_mode])
    return y


def codec_ru_tc(x, w_units, b7, b1, *, dilation, pad_mode="reflect", out_phases=1):
    """fused ResidualUnit on C8S activations (P = 1 in, `out_phases` planes out)."""
    _check_cuda(x, w_units, b7, b1)
    B, nch2, P, T, _ = x.shape
    C = nch2 * 4
    assert P == 1 and x.dtype == bf16 and x.is_contiguous() and w_units.dtype == bf16 and w_units.is_contiguous()
    assert w_units.numel() == 8 * (C // 16) * 2 * 2 * C * 8
    y = torch.empty(B, nch2, out_phases, T // out_phases, 8, device=x.device, dtype=bf16)
    cls = "codec_ru_tc"
    if _PROFILE is not None and PROFILE_SHAPES:
        cls += f" C{C} T{T} d{dilation} P{out_phases}"
    with _timed(cls, 2.0 * B * C * T * 4, "byte"):
        _lib.call("alm_codec_ru_tc", x, y, w_units, b7, b1, B, C, T, int(dilation), PAD_MODES[pad_mode],
                  int(out_phases))
    return y


def codec_conv_tc(x, w_units, bias, *, cout, kernel_size, stride, pad_mode="reflect", out_phases=1, out_fp32=False,
                  upsample=1):
    """CausalConv1d(Cin, cout, kernel_size, stride) on C8S activations with P = stride planes.  upsample = s > 1: the
    transposed-conv form (see pack_convT_weights): cout = s * C' columns become s time steps of C' channels."""
    _check_cuda(x, w_units, bias)
    B, nch2, P, Tp, _ = x.shape
    Cin, Tin = nch2 * 4, P * Tp
    assert P == stride and x.is_contiguous() and w_units.is_contiguous()
    n_out = Tin // stride
    if out_fp32:
        y = torch.empty(B, n_out, cout, device=x.device, dtype=f32)
    elif upsample > 1:
        y = torch.empty(B, 2 * (cout // upsample) // 8, 1, n_out * upsample, 8, device=x.device, dtype=bf16)
    else:
        y = torch.empty(B, 2 * cout // 8, out_phases, n_out // out_phases, 8, device=x.device, dtype=bf16)
    cls = "codec_conv_tc"
    if _PROFILE is not None and PROFILE_SHAPES:
        cls += f" Cin{Cin} Cout{cout} K{kernel_size} s{stride} T{Tin}"
    with _timed(cls, 4.0 * B * (Cin * Tin + cout * n_out), "byte"):
        _lib.call("alm_codec_conv_tc", x, y, w_units, bias, B, Cin, cout, Tin, int(kernel_size), int(stride),
                  PAD_MODES[pad_mode], int(out_phases), int(out_fp32), int(upsample))
    return y


def rvq_encode(x, codebooks):
    """x [N, D] fp32, codebooks [Q, C, D] fp32 -> (quantized [N, D] fp32, indices [N, Q] int64)."""
    _check_cuda(x, codebooks)
    assert x.dtype == f32 and codebooks.dtype == f32 and x.stride(-1) == 1
    N, D = x.shape
    Q, C, D2 = codebooks.shape
    assert D == D2
    codebooks = codebooks.contiguous()
    quant = torch.empty(N, D, device=x.device, dtype=f32)
    idx = torch.empty(N, Q, device=x.device, dtype=torch.int64)
    ws = torch.empty(Q * C, device=x.device, dtype=f32)
    with _timed("rvq_encode", 2.0 * N * Q * C * D):
        _lib.call("alm_rvq_encode", x, x.stride(0), codebooks, ws, quant, D, idx, Q, N, D, C, Q)
    return quant, idx


def rvq_pack_codebooks(codebooks):
    """codebooks fp32 [Q, C, D] -> (packed bf16 [Q, C, 3D] = [hi | hi | lo], e2 fp32 [Q, C]) for rvq_encode_tc."""
    _check_cuda(codebooks)
    Q, C, D = codebooks.shape
    cb = codebooks.to(f32).contiguous()
    packed = torch.empty(Q, C, 3 * D, device=cb.device, dtype=bf16)
    e2 = torch.empty(Q, C, device=cb.device, dtype=f32)
    _lib.call("alm_rvq_pack_codebooks", cb, packed, e2, Q * C, D)
    return cb, packed, e2


def rvq_encode_tc(x, packed_codebooks):
    """x [N, D] fp32 -> (quantized [N, D] fp32, indices [N, Q] int64); distance GEMMs on the tensor cores, the
    winner of every stage chosen by exact fp32 re-evaluation of the candidates (csrc/rvq_tc.cu)."""
    cb, packed, e2 = packed_codebooks
    _check_cuda(x, cb)
    assert x.dtype == f32 and x.stride(-1) == 1
    N, D = x.shape
    Q, C, _ = cb.shape
    assert D % 8 == 0
    dev = x.device
    r = torch.empty(N, D, device=dev, dtype=f32)
    quant = torch.empty(N, D, device=dev, dtype=f32)
    rp = torch.empty(N, 3 * D, device=dev, dtype=bf16)
    scores = torch.empty(N, C, device=dev, dtype=f32)
    idx = torch.empty(N, Q, device=dev, dtype=torch.int64)
    with _timed("rvq_encode_tc", 2.0 * N * Q * C * D):
        _lib.call("alm_rvq_prepare", x, x.stride(0), r, quant, D, rp, N, D)
        for q in range(Q):
            gemm(rp, packed[q], out=scores, cls="rvq_score_gemm")
            _lib.call("alm_rvq_select", scores, C, e2[q], cb[q], r, quant, D, rp, idx[:, q:], Q, N, D, C,
                      int(q + 1 < Q))
    return quant, idx


def nearest_centroid(x, packed_centroids):
    """cluster assignment of HubertWithKmeans.forward (hubert_kmeans.py:114-116: `(-torch.cdist(embed, centers)).argmax(-1)`):
    x [N, D] fp32, packed_centroids = rvq_pack_codebooks(centers[None]) -> ids [N] int64.  Same kernels as one RVQ stage:
    the distance GEMM on the tensor cores, then the exact fp32 re-rank (lowest index on ties, as argmax does)."""
    _, idx = rvq_encode_tc(x, packed_centroids)
    return idx[:, 0]


def rvq_decode(indices, codebooks):
    """indices [N, Q] int64 (-1 = dropped) -> sum of selected codes [N, D] fp32."""
    _check_cuda(indices, codebooks)
    indices = indices.to(torch.int64).contiguous()
    N, Q = indices.shape
    Qc, C, D = codebooks.shape
    assert Q <= Qc
    out = torch.empty(N, D, device=indices.device, dtype=f32)
    _lib.call("alm_rvq_decode", indices, Q, codebooks.contiguous(), out, D, N, D, C, Q)
    return out


def topk_gumbel_sample(logits, uniform, *, k, temperature=1.0):
    """ids [R] = Gumbel-max sample over the k largest logits of each row (noise supplied by the caller)."""
    _check_cuda(logits, uniform)
    assert logits.dtype == f32 and uniform.dtype == f32 and logits.shape == uniform.shape
    assert logits.stride(-1) == 1 and uniform.stride(-1) == 1
    R, V = logits.shape
    ids = torch.empty(R, device=logits.device, dtype=torch.int64)
    _lib.call("alm_topk_gumbel_sample", logits, logits.stride(0), uniform, uniform.stride(0), ids, R, V, int(k),
              float(temperature))
    return ids


def resid_ln_fwd(r, y, gamma, *, want_r_new=True, want_raw=False):
    """plain residual + LayerNorm (num_residual_streams == 1).  r [M,d] fp32, y [M,d] bf16 or None.

    Returns r_new [M,d] fp32 (== r when y is None and want_r_new False), xn bf16, raw bf16 copy (optional), stats."""
    M, d = r.shape
    r_new = torch.empty_like(r) if (want_r_new and y is not None) else None
    xn = torch.empty(M, d, device=r.device, dtype=bf16)
    raw = torch.empty(M, d, device=r.device, dtype=bf16) if want_raw else None
    stats = torch.empty(M, 2, device=r.device, dtype=f32)
    _lib.call("alm_resid_ln_fwd", r, y, gamma, r_new, xn, raw, stats, M, d)
    return (r_new if r_new is not None else r), xn, raw, stats


def resid_ln_bwd(r_new, gamma, stats, dr_out, dxn, dextra, g_gamma, *, out_scale=1.0, want_bf16=True):
    """dr = out_scale * (dr_out + LN_bwd(dxn) + dextra) as fp32 (and bf16 for the next GEMMs)."""
    M, d = r_new.shape
    dr = torch.empty(M, d, device=r_new.device, dtype=f32)
    dr_b = torch.empty(M, d, device=r_new.device, dtype=bf16) if want_bf16 else None
    _lib.call("alm_resid_ln_bwd", r_new, gamma, stats, dr_out, dxn, dextra, dr, dr_b, g_gamma, float(out_scale), M, d)
    return dr, dr_b
