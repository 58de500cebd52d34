"""CPU: drop-in surface — constructor kwargs, state_dict keys/shapes, C-ABI symbols, host-side helpers."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
G = ROOT / "tests" / "golden"


def load(name):
    return torch.load(G / name, map_location="cpu", weights_only=False)


@pytest.mark.parametrize("fixture,cls_name", [("semantic.pt", "SemanticTransformer"), ("coarse.pt", "CoarseTransformer"),
                                              ("fine.pt", "FineTransformer"),
                                              ("semantic_plain.pt", "SemanticTransformer")])
def test_state_dict_keys_match_reference(fixture, cls_name):
    from audiolm_pytorch_b200 import audiolm

    g = load(fixture)
    m = getattr(audiolm, cls_name)(**g["kwargs"])
    mine = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    ref = {k: tuple(v.shape) for k, v in g["state"].items()}
    assert mine == ref
    m.load_state_dict(g["state"], strict=True)


@pytest.mark.parametrize("which,cls_name", [("semantic", "SemanticTransformer"), ("coarse", "CoarseTransformer"),
                                            ("fine", "FineTransformer")])
def test_state_dict_keys_match_reference_rel_pos_bias(which, cls_name):
    """flash_attn=False: rel_pos_bias.net.*, cross_attn_bias, pos_bias_mlp.*, null_pos_bias (SURVEY §8 a7)."""
    from audiolm_pytorch_b200 import audiolm

    g = load("relpos.pt")[which]
    m = getattr(audiolm, cls_name)(**g["kwargs"])
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == {k: tuple(v.shape) for k, v in g["state"].items()}
    m.load_state_dict(g["state"], strict=True)


def test_fine_pos_bias_index_matches_oracle():
    """the int32 index map + MLP inputs the gather kernel consumes reproduce the oracle's dense bias."""
    from audiolm_pytorch_b200 import audiolm
    from oracle import transformer as ot

    g = load("relpos.pt")["fine"]
    m = audiolm.FineTransformer(**g["kwargs"])
    m.load_state_dict(g["state"])
    st = g["state"]
    n, nf = 12, 18
    idx, mlp_in = m._pos_bias_index(n, nf, "cpu")
    t = torch.nn.functional.silu(mlp_in @ st["pos_bias_mlp.0.weight"].t() + st["pos_bias_mlp.0.bias"])
    t = torch.nn.functional.silu(t @ st["pos_bias_mlp.2.weight"].t() + st["pos_bias_mlp.2.bias"])
    t = t @ st["pos_bias_mlp.4.weight"].t() + st["pos_bias_mlp.4.bias"]
    dense = torch.where((idx < 0)[None], st["null_pos_bias"], t[idx.clamp(min=0).long()].permute(2, 0, 1))
    assert torch.allclose(dense, ot.fine_pos_bias(st, n, nf, 3, 5, "cpu"), atol=1e-6)


def test_c_abi_exports_every_declared_symbol():
    lib_path = ROOT / "audiolm_pytorch_b200" / "libalm_b200.so"
    if not lib_path.exists():
        from audiolm_pytorch_b200 import build

        build.build()
    lib = ctypes.CDLL(str(lib_path))
    header = (ROOT / "include" / "alm_b200.h").read_text()
    names = set(re.findall(r"\b(alm_[A-Za-z0-9_]+)\s*\(", header))
    assert len(names) >= 15
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/alm_b200.h but not exported"
    from audiolm_pytorch_b200 import _lib

    for n in _lib.SIGNATURES:
        assert n in names, f"{n} bound in _lib.py but not declared in the header"
    assert lib.alm_version() >= 100


def test_ops_refuse_cpu_tensors():
    from audiolm_pytorch_b200 import _lib, ops

    a = torch.zeros(8, 8, dtype=torch.bfloat16)
    with pytest.raises(_lib.AlmError):
        ops.gemm(a, a)


def test_fcm_mask_and_eos_helpers():
    from audiolm_pytorch_b200 import heads

    m = heads.generate_mask_with_prob((4, 100), 0.15, "cpu")
    assert m[:, 0].all() and (~m).sum(-1).eq(15).all()
    g = load("sampling.pt")
    assert torch.equal(heads.top_k(g["logits"], thres=0.9), g["filtered"])
    assert torch.equal(heads.mask_out_after_eos_id(g["seq"], 64, keep_eos=False), g["seq_masked"])


def test_split_k_heuristic_bounds():
    from audiolm_pytorch_b200.transformer import best_split_k

    for (M, N, K) in [(512, 1024, 32768), (128, 1024, 32768), (5460, 1024, 32768), (1024, 2730, 32768), (64, 64, 64)]:
        s = best_split_k(M, N, K)
        assert 1 <= s <= max(1, -(-K // 64))


def test_kernel_bias_layout_helper():
    """as_kernel_bias: any [h, i, j] bias becomes an fp32 tensor whose row stride is a multiple of 4 elements,
    without a copy when the caller already holds the padded buffer (rel_pos.gather_bias slices it)."""
    from audiolm_pytorch_b200.rel_pos import as_kernel_bias

    b = torch.randn(2, 5, 7)
    k = as_kernel_bias(b)
    assert k.shape == (2, 5, 8) and k.is_contiguous() and torch.equal(k[..., :7], b) and (k[..., 7] == 0).all()
    padded = torch.randn(2, 5, 8)
    view = padded[..., :7]
    assert as_kernel_bias(view).data_ptr() == padded.data_ptr()   # the padded base is reused
    full = torch.randn(2, 4, 12)
    assert as_kernel_bias(full) is full


def test_tile_rows_equals_modulo_indexing():
    from audiolm_pytorch_b200.audiolm import _tile_rows

    w = torch.randn(3, 6, requires_grad=True)
    for n in (0, 1, 3, 7, 12):
        idx = torch.arange(n) % 3
        assert torch.equal(_tile_rows(w, n), w[idx])
    _tile_rows(w, 7).sum().backward()
    assert torch.equal(w.grad, torch.tensor([[3.0] * 6, [2.0] * 6, [2.0] * 6]))


def test_flat_bucket_ranges():
    from audiolm_pytorch_b200.parallel import FlatGradBucket

    m = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
    b = FlatGradBucket(m.parameters())
    assert b.range_of(list(m[0].parameters())) == (0, 15) and b.range_of(list(m[1].parameters())) == (15, 23)
    with pytest.raises(AssertionError):
        b.range_of([m[0].weight, m[1].weight])   # not adjacent in the bucket
    b.reduce_range_async(0, 15)                  # no process group: no-op
    b.finish()


def test_bench_dump_outputs_are_seeded_and_bounded(tmp_path):
    """bench.py --dump-outputs: float32 / float64 .npy files, the same sample positions on every call, under 64 MB."""
    import numpy as np

    import bench
    from audiolm_pytorch_b200.parallel import FlatGradBucket

    m = torch.nn.Sequential(torch.nn.Linear(300, 200), torch.nn.Linear(200, 10))
    b = FlatGradBucket(m.parameters())
    b.flat.copy_(torch.arange(b.numel, dtype=torch.float32))
    out = bench.last_step_outputs(torch.tensor(2.5), b)
    bench.write_outputs(tmp_path / "a", out)
    bench.write_outputs(tmp_path / "b", bench.last_step_outputs(torch.tensor(2.5), b))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grad_norm.npy", "grad_sample.npy", "loss.npy"]
    for name in files:
        a, c = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, c), name
    assert float(np.load(tmp_path / "a" / "loss.npy")) == 2.5
    sample = np.load(tmp_path / "a" / "grad_sample.npy")
    assert np.array_equal(sample, np.sort(sample)) and sample.max() < b.numel   # positions of the flat gradient
    norms = np.load(tmp_path / "a" / "grad_norm.npy")
    assert np.allclose(norms, [p.grad.double().norm().item() for p in b.params])
    assert bench.DUMP_GRAD_SAMPLES * 4 + 142 * 8 + 4 < 64 << 20   # the benchmarked model has 142 parameters


def test_batch_unique_consecutive_matches_per_row_loop():
    """vectorised version vs the reference construction (audiolm_pytorch.py:162-164)"""
    from torch import nn

    from audiolm_pytorch_b200.audiolm import batch_unique_consecutive

    def ref(t, pad_value):
        rows = [torch.unique_consecutive(r) for r in t.unbind(0)]
        return nn.utils.rnn.pad_sequence(rows, batch_first=True, padding_value=pad_value)

    torch.manual_seed(0)
    for shape, hi in [((4, 50), 3), ((3, 1), 5), ((2, 17), 100), ((5, 200), 2), ((1, 9), 1)]:
        t = torch.randint(0, hi, shape)
        assert torch.equal(batch_unique_consecutive(t, -1), ref(t, -1)), shape
    t = torch.tensor([[1, 1, 2, -1, -1], [3, 4, 5, 6, 7]])
    assert torch.equal(batch_unique_consecutive(t, -1), ref(t, -1))


def test_flat_grad_bucket_survives_zero_grad_set_to_none():
    """optimizer.zero_grad(set_to_none=True) detaches .grad from the bucket; sync_views() copies the fresh gradients in
    and restores the aliasing before any collective / clip (ADVICE r1, parallel.py)."""
    from audiolm_pytorch_b200.parallel import FlatGradBucket

    m = torch.nn.Linear(4, 3)
    b = FlatGradBucket(m.parameters())
    opt = torch.optim.SGD(m.parameters(), lr=0.1)
    opt.zero_grad()                      # set_to_none=True by default
    assert m.weight.grad is None
    m(torch.ones(2, 4)).sum().backward()
    assert m.weight.grad.data_ptr() != b.flat.data_ptr()
    n = b.grad_norm()                    # -> sync_views
    assert m.weight.grad.data_ptr() == b.flat[:12].data_ptr()
    assert torch.allclose(n, torch.cat([p.grad.flatten() for p in m.parameters()]).norm())
    assert torch.equal(b.flat[:12].view(3, 4), torch.full((3, 4), 2.0))
    b.zero_()
    assert float(m.weight.grad.abs().sum()) == 0.0


def test_regroup_rows_layout_of_the_decode_step_operands():
    """ops.regroup_rows: row (c * pc + l) of the copy is row (c + l * grid) of the operand, zero rows past N - the layout
    alm_decode_stack_step documents in include/alm_b200.h (CTA c's rows of a projection become one contiguous block)."""
    from audiolm_pytorch_b200 import ops

    for N, K, grid in [(640, 16, 148), (5472, 8, 148), (7, 8, 4), (148, 8, 148), (149, 8, 148)]:
        w = torch.arange(N * K, dtype=torch.float32).view(N, K)
        wp = ops.regroup_rows(w, grid)
        pc = -(-N // grid)
        assert wp.shape == (grid * pc, K) and wp.is_contiguous()
        for c in (0, 1, grid // 2, grid - 1):
            for l in range(pc):
                n = c + l * grid
                want = w[n] if n < N else torch.zeros(K)
                assert torch.equal(wp[c * pc + l], want), (N, grid, c, l)


def test_deferred_heads_flag_is_scoped_to_the_loss_forward():
    """the wrappers switch the transformers to LazyLogits only while they compute a loss; the flag is reset on exit and
    on exceptions, and heads.FUSED_HEAD_CE = False disables it (public forward signatures stay the reference's)."""
    from audiolm_pytorch_b200 import audiolm, heads

    class T:
        _defer_heads = False

    t = T()
    with audiolm._deferred_heads(t, True):
        assert t._defer_heads is True
    assert t._defer_heads is False
    with audiolm._deferred_heads(t, False):
        assert t._defer_heads is False
    try:
        with audiolm._deferred_heads(t, True):
            raise RuntimeError("x")
    except RuntimeError:
        pass
    assert t._defer_heads is False
    heads.FUSED_HEAD_CE = False
    try:
        with audiolm._deferred_heads(t, True):
            assert t._defer_heads is False
    finally:
        heads.FUSED_HEAD_CE = True
    import inspect
    for cls in (audiolm.SemanticTransformer, audiolm.CoarseTransformer, audiolm.FineTransformer):
        assert not any(name.startswith("_") for name in inspect.signature(cls.forward).parameters if name != "self")
