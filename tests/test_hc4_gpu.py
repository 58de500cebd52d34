"""Hyper-connection pre-branch kernels for d <= 1024 (csrc/hyper_conn_v4.cuh) at awkward token counts and widths,
both input forms, against the fp32 restatement + autograd; parameter gradients are bitwise reproducible."""
import pytest
import torch

from test_ops_gpu import DEV, bf16, hc_ref, make_hc, rel_err

pytestmark = pytest.mark.gpu

SHAPES = [(32768, 1024)] + [(M, d) for M in (1, 3, 37, 300, 32768 + 5) for d in (64, 128, 520, 1024)]


def _run(M, d, expand, seed):
    from audiolm_pytorch_b200 import ops

    torch.manual_seed(seed)
    S = 4
    hc, ln_gamma = make_hc(d, seed=d)
    if expand:
        x = torch.randn(M, d, device=DEV)
        inputs = dict(x_expand=x)
    else:
        R_in = torch.randn(M, S, d, device=DEV).to(bf16)
        Y = torch.randn(M, d, device=DEV).to(bf16)
        bp = 1 + 0.2 * torch.randn(M, S, device=DEV)
        inputs = dict(R_in=R_in, Y=Y, beta_prev=bp)
    outs = ops.hc_pre_fwd(hc, ln_gamma, **inputs, M=M, d=d)
    up = (torch.randn(M, S, d, device=DEV).to(bf16), torch.randn(M, d, device=DEV).to(bf16),
          torch.randn(M, d, device=DEV).to(bf16), torch.randn(M, S, device=DEV))
    return hc, ln_gamma, inputs, outs, up


def _bwd(hc, ln_gamma, inputs, aux, up, M, d):
    from audiolm_pytorch_b200 import ops

    w1, w2, w3, w4 = up
    grads = {k: torch.zeros_like(v) for k, v in hc.items()}
    g_ln = torch.zeros_like(ln_gamma)
    extra = dict(dx_scale=0.1) if "x_expand" in inputs else {}
    res = ops.hc_pre_bwd(hc, ln_gamma, grads, g_ln, aux, w1, w2, w4, dbin_extra=w3, **inputs, **extra, M=M, d=d)
    return res, grads, g_ln


@pytest.mark.parametrize("expand", [False, True])
@pytest.mark.parametrize("M,d", SHAPES)
def test_hc4_pre_fwd_bwd(M, d, expand):
    hc, ln_gamma, inputs, outs, up = _run(M, d, expand, seed=M + d)
    S = 4
    hc_leaf = {k: v.clone().requires_grad_(True) for k, v in hc.items()}
    lng_leaf = ln_gamma.clone().requires_grad_(True)
    if expand:
        x_leaf = inputs["x_expand"].clone().requires_grad_(True)
        R = x_leaf[:, None, :].expand(M, S, d)
    else:
        Ri, Yl, bpl = (t.float().clone().requires_grad_(True) for t in inputs.values())
        R = Ri + bpl[..., None] * Yl[:, None, :]
    R_out, bin_, xn, beta, aux = outs
    r_out, r_bin, r_xn, r_beta = hc_ref(hc_leaf, lng_leaf, R, d)
    assert rel_err(R_out, r_out) < 1e-2
    assert rel_err(bin_, r_bin) < 1e-2
    assert rel_err(xn, r_xn) < 1.5e-2
    assert rel_err(beta, r_beta) < 1e-3

    w1, w2, w3, w4 = up
    loss = (r_out * w1.float()).sum() + (r_xn * w2.float()).sum() + (r_bin * w3.float()).sum() + (r_beta * w4).sum()
    loss.backward()
    res, grads, g_ln = _bwd(hc, ln_gamma, inputs, aux, up, M, d)
    if expand:
        assert rel_err(res, 0.1 * x_leaf.grad) < 2e-2
    else:
        for got, ref in zip(res, (Ri.grad, Yl.grad, bpl.grad)):
            assert rel_err(got, ref) < 2e-2
    torch.cuda.synchronize()
    for k in hc:
        assert rel_err(grads[k], hc_leaf[k].grad) < 3e-2, k
    assert rel_err(g_ln, lng_leaf.grad) < 3e-2


@pytest.mark.parametrize("expand", [False, True])
@pytest.mark.parametrize("M,d", [(300, 520), (32768, 1024)])
def test_hc4_param_grads_bitwise_reproducible(M, d, expand):
    hc, ln_gamma, inputs, outs, up = _run(M, d, expand, seed=7)
    _, g_a, ln_a = _bwd(hc, ln_gamma, inputs, outs[4], up, M, d)
    _, g_b, ln_b = _bwd(hc, ln_gamma, inputs, outs[4], up, M, d)
    for k in hc:
        assert torch.equal(g_a[k], g_b[k]), k
    assert torch.equal(ln_a, ln_b)
