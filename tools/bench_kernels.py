#!/usr/bin/env python
"""Stand-alone timings of the HBM-bound row kernels at C3 sizes (CUDA events, L2 flushed between iterations).
usage: python tools/bench_kernels.py [geglu] [hc] [attn] ..."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from audiolm_pytorch_b200 import ops  # noqa: E402

dev = "cuda"
bf16, f32 = torch.bfloat16, torch.float32
torch.manual_seed(0)
M, d, H = 16 * 2048, 1024, 8
which = set(sys.argv[1:]) or {"geglu", "hc", "attn"}
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)


def rnd(*s, dt=bf16, k=1.0):
    return (torch.randn(*s, device=dev) * k).to(dt)


def timeit(name, fn, nbytes=None, flops=None, iters=8):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = sorted(ts)[len(ts) // 2]
    extra = ""
    if nbytes:
        extra += f"  {nbytes / ms / 1e6:8.0f} GB/s"
    if flops:
        extra += f"  {flops / ms / 1e9:8.0f} TFLOP/s"
    print(f"{name:34s} {ms * 1e3:9.1f} us{extra}", flush=True)


if "geglu" in which:
    ip = 2736
    h = rnd(M, 2 * ip)
    g = rnd(2730, dt=f32)
    gn, st = ops.geglu_ln_fwd(h, g, inner=2730, inner_pad=ip)
    dgn = rnd(M, ip)
    gg = torch.zeros_like(g)
    timeit("geglu_ln_fwd", lambda: ops.geglu_ln_fwd(h, g, inner=2730, inner_pad=ip), nbytes=M * ip * 6)
    timeit("geglu_ln_bwd", lambda: ops.geglu_ln_bwd(h, g, st, dgn, gg, inner=2730, inner_pad=ip), nbytes=M * ip * 10)

if "hc" in which:
    hc = dict(gamma=rnd(d, dt=f32, k=0.1), dyn_alpha=rnd(d, 5, dt=f32, k=0.05), dyn_beta=rnd(d, dt=f32, k=0.05),
              static_alpha=rnd(4, 5, dt=f32), static_beta=rnd(4, dt=f32), alpha_scale=torch.tensor(0.3, device=dev),
              beta_scale=torch.tensor(0.3, device=dev))
    lng = rnd(d, dt=f32)
    R, Y, bp = rnd(M, 4, d), rnd(M, d), rnd(M, 4, dt=f32)
    timeit("hc_pre_fwd", lambda: ops.hc_pre_fwd(hc, lng, R_in=R, Y=Y, beta_prev=bp, M=M, d=d), nbytes=M * d * 22)
    R_out, bin_, xn, beta, aux = ops.hc_pre_fwd(hc, lng, R_in=R, Y=Y, beta_prev=bp, M=M, d=d)
    dR, dxn, dbe, dbin = rnd(M, 4, d), rnd(M, d), rnd(M, 4, dt=f32), rnd(M, d)
    grads = {k_: torch.zeros_like(v_) for k_, v_ in hc.items()}
    gl = torch.zeros_like(lng)

    def hcb():
        return ops.hc_pre_bwd(hc, lng, grads, gl, aux, dR, dxn, dbe, dbin_extra=dbin, R_in=R, Y=Y, beta_prev=bp, M=M, d=d)

    timeit("hc_pre_bwd (+ param finish)", hcb, nbytes=M * d * 32)
    x = rnd(M, d, dt=f32)
    timeit("hc_pre_fwd x_expand", lambda: ops.hc_pre_fwd(hc, lng, x_expand=x, M=M, d=d), nbytes=M * d * 16)
    aux_x = ops.hc_pre_fwd(hc, lng, x_expand=x, M=M, d=d)[4]
    timeit("hc_pre_bwd x_expand (+ param finish)",
           lambda: ops.hc_pre_bwd(hc, lng, grads, gl, aux_x, dR, dxn, dbe, dbin_extra=dbin, x_expand=x, M=M, d=d),
           nbytes=M * d * 20)

if "attn" in which:
    q, k, v = rnd(16, 2048, 512), rnd(16, 2048, 64), rnd(16, 2048, 64)
    fl = 4.0 * 16 * 8 * 64 * (2048 * 2049 / 2)
    timeit("attn fwd", lambda: ops.mqa_attn_fwd(q, k, v, heads=8), flops=fl)
    o, lse = ops.mqa_attn_fwd(q, k, v, heads=8)
    do = rnd(16, 2048, 512)
    timeit("attn bwd (delta + dkv + dq)", lambda: ops.mqa_attn_bwd(q, k, v, o, do, lse, heads=8), flops=2.5 * fl)
