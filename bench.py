#!/usr/bin/env python
"""Headline benchmark: CoarseTransformer fwd+bwd tokens/s at seq 2048 (BASELINE.json configs[2], "C3").

    python bench.py --gpus N --steps K --warmup W             # our CUDA path (one rank per GPU via torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores
    python bench.py --gpus 1 --steps K --dump-outputs DIR     # + loss / gradients of the last timed step as .npy

One step = what CoarseTransformerTrainer.train_step runs (trainer.py:1242-1252): the training wrapper
`CoarseTransformerWrapper.forward(semantic_token_ids, coarse_token_ids, return_loss=True)` with its defaults
(unique_consecutive=True, mask_prob=0.15: EOS handling, the key-padding mask it ALWAYS passes and the forgetful
causal mask, audiolm_pytorch.py:1742-1854) around CoarseTransformer(dim 1024, depth 6, heads 8, 4 hyper-connection
streams, flash path) on a batch of 16 sequences of 2048 positions (371 semantic ids + EOS, 558 frames x 3 coarse
ids, 2 start tokens), backward to every parameter, and (N > 1) the flat-bucket gradient all-reduce.
`variants.direct_causal` times the bare transformer without any key mask (SURVEY 8(d) variant a) for comparison.
At N=1 the line also carries the other BASELINE.json configs (C1 codec, C2, C4, C5) as extra keys.
Synthetic ids, random-init weights.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CFG = dict(num_semantic_tokens=500, codebook_size=1024, num_coarse_quantizers=3, dim=1024, depth=6, heads=8,
           flash_attn=True)
BATCH, N_SEM, N_COARSE = 16, 372, 1674  # direct variant: 1 + 372 + 1 + 1674 = 2048 positions
SEQ = 1 + N_SEM + 1 + N_COARSE
W_SEM, W_FRAMES = 371, 558  # wrapper path: 1 + (371 + EOS) + 1 + (558*3 + EOS - 1) = 2048 positions
METRIC = "CoarseTransformer tokens/sec fwd+bwd seq2048"


def synth_ids(batch, seed):
    g = torch.Generator().manual_seed(seed)
    sem = torch.randint(0, CFG["num_semantic_tokens"], (batch, N_SEM), generator=g)
    coarse = torch.randint(0, CFG["codebook_size"], (batch, N_COARSE), generator=g)
    return sem, coarse


def synth_wrapper_ids(batch, seed):
    """ids for the wrapper path; no two equal neighbours among the semantic ids, so unique_consecutive=True (the wrapper
    default) leaves every row at full length and the step always covers exactly 2048 positions per sequence"""
    g = torch.Generator().manual_seed(1000 + seed)
    sem = torch.randint(0, CFG["num_semantic_tokens"], (batch, W_SEM), generator=g)
    for i in range(1, W_SEM):
        same = sem[:, i] == sem[:, i - 1]
        sem[:, i] = torch.where(same, (sem[:, i] + 1) % CFG["num_semantic_tokens"], sem[:, i])
    coarse = torch.randint(0, CFG["codebook_size"], (batch, W_FRAMES, CFG["num_coarse_quantizers"]), generator=g)
    return sem, coarse


class _CodecStub:
    """the wrapper constructors read these two attributes of the codec; the codec itself is benchmarked separately"""
    rq_groups = 1
    num_quantizers = 8


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region: NVML every 10 ms (pynvml ships with the image as
    nvidia-ml-py); falls back to polling nvidia-smi when NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()
        self.max_mhz = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may remap indices; the UUID of the torch device is authoritative
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            h = None
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                u = pynvml.nvmlDeviceGetUUID(hi)
                u = u.decode() if isinstance(u, bytes) else u
                if uuid in u:
                    h = hi
            self._h = h if h is not None else pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        mhz = n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        names = []
        for name, bit in (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
                          ("sw_power_cap", 0x4)):
            if r & bit:
                names.append(name)
        self.samples.append((mhz, names))

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    if len(f) >= 7 and f[0].replace(".", "").isdigit():
                        names = [nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                      "sw_power_cap"), f[3:7]) if v.lower().startswith("active")]
                        self.samples.append((int(float(f[0])), names))
                        self.max_mhz = int(float(f[1]))
            except Exception:
                pass
            self._stop_evt.wait(0.01 if self._nvml is not None else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(s[0] for s in self.samples)
        reasons = sorted({r for s in self.samples for r in s[1]})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_min_mhz=sm[0] if sm else None,
                    sm_max_mhz=self.max_mhz, reasons=reasons, samples=len(self.samples),
                    source="nvml" if self._nvml is not None else "nvidia-smi")


# ------------------------------------------------------------------------------------------------
# reference algorithm on the CPU (oracle port of the reference path; the real package cannot be
# installed offline and /root/reference does not exist on the GPU box)
# ------------------------------------------------------------------------------------------------
def cpu_step_fn(batch):
    from oracle import transformer as ot
    from audiolm_pytorch_b200.audiolm import CoarseTransformer

    torch.manual_seed(1234)
    model = CoarseTransformer(**CFG)
    state = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    del model
    # the wrapper's arithmetic (audiolm_pytorch.py:1785-1854) restated over the oracle: EOS appended to both id
    # streams, semantic EOS masked as a key, forgetful causal mask, the two cross entropies mixed by logit count
    sem, coarse = synth_wrapper_ids(batch, 0)
    sem_l = torch.cat((sem, torch.full((batch, 1), CFG["num_semantic_tokens"])), dim=1)
    co_l = torch.cat((coarse.reshape(batch, -1), torch.full((batch, 1), CFG["codebook_size"])), dim=1)
    keep = torch.nn.functional.pad(sem_l != CFG["num_semantic_tokens"], (1, co_l.shape[1]), value=True)
    hk = dict(heads=CFG["heads"], depth=CFG["depth"], codebook_size=CFG["codebook_size"],
              num_coarse_quantizers=CFG["num_coarse_quantizers"])

    def step():
        for v in state.values():
            v.grad = None
        mask = keep & ot.fcm_mask(tuple(keep.shape), 0.15)
        (sl, cl), _ = ot.coarse_forward(state, sem_l.masked_fill(sem_l == CFG["num_semantic_tokens"], 0), co_l[:, :-1],
                                        self_attn_mask=mask, **hk)
        loss = ot.coarse_wrapper_loss(sl, cl, sem_l, co_l)
        loss.backward()
        return float(loss.detach())

    return step


def run_cpu(steps, warmup, batch=1):
    # more than ~32 intra-op threads makes torch's CPU kernels slower at these sizes (measured: 128 threads ->
    # 113 s/step vs 11 s/step with 8), so the baseline uses min(cores, 32) threads and says so in `cores`
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    step = cpu_step_fn(batch)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * SEQ * steps / dt, dt / steps * 1e3, torch.get_num_threads()


WORKLOAD = ("C3 CoarseTransformerWrapper.forward(return_loss=True) [key mask + FCM mask, wrapper defaults] around "
            "CoarseTransformer d1024 L6 h8 4-stream hyper-connections, flash path, batch 16/GPU x seq 2048, "
            "fwd + CE + bwd")


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else this process (or NCCL) prints went to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tps, ms, cores = run_cpu(args.steps, args.warmup)
    sample = f"batch 1 x {SEQ} tokens per step, fp32, oracle port of the reference path (torch CPU, {cores} threads)"
    emit({
        "impl": "reference", "metric": METRIC, "value": tps, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD + " (CPU arm: bounded sample, see cpu_baseline.sample)", "seq_len": SEQ,
                   "global_batch": BATCH * args.gpus, "parallelism": f"dp{args.gpus}"},
        "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ------------------------------------------------------------------------------------------------
# second half of BASELINE.json's metric: SoundStream frames/s encode (config C1 shapes, batch of clips)
# ------------------------------------------------------------------------------------------------
ENC_BYTES_PER_CLIP = 133.8e6  # SURVEY 8(d): sum over encoder layers of (C_in T_in + C_out T_out) * 4 B, fused RU = 1 layer


def _timed_cuda(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def codec_bench(dev, clips=32, iters=5):
    """C1: encoder conv stack + 8-stage RVQ (and the decoder) on `clips` x 2 s @ 24 kHz (48000 samples -> 150 frames)."""
    from audiolm_pytorch_b200 import ops
    from audiolm_pytorch_b200.soundstream import SoundStream

    torch.manual_seed(7)
    ss = SoundStream(codebook_size=1024, rq_num_quantizers=8, target_sample_hz=24000, use_local_attn=False)
    for rvq in ss.rq.rvqs:
        for layer in rvq.layers:
            layer._codebook.embed.normal_()
            layer._codebook.initted.fill_(True)
    ss = ss.to(dev).eval()
    wave = torch.randn(clips, 48000, device=dev)
    pk = peaks()
    with torch.no_grad():
        ms = _timed_cuda(lambda: ss(wave, return_encoded=True), iters)
        _, idx, _ = ss(wave, return_encoded=True)
        ms_dec = _timed_cuda(lambda: ss.decode_from_codebook_indices(idx), iters)
        ops.profile_start()
        ss(wave, return_encoded=True)
        prof = ops.profile_stop()
    # the constructor's default configuration: LocalTransformer bottleneck (use_local_attn=True) before the quantizer
    try:
        torch.manual_seed(7)
        ssd = SoundStream(codebook_size=1024, rq_num_quantizers=8, target_sample_hz=24000)
        for rvq in ssd.rq.rvqs:
            for layer in rvq.layers:
                layer._codebook.embed.normal_()
                layer._codebook.initted.fill_(True)
        ssd = ssd.to(dev).eval()
        with torch.no_grad():
            ms_default = _timed_cuda(lambda: ssd(wave, return_encoded=True), iters)
        del ssd
    except Exception as e:  # pragma: no cover
        ms_default = None
    frames = clips * 150
    kern = {cls: {"ms_per_call": ms_, "launches": n_,
                  ("gbps" if ops.CLASS_UNIT.get(cls) == "byte" else "tflops"): work / (ms_ * 1e-3) / (1e9 if ops.CLASS_UNIT.get(cls) == "byte" else 1e12) if ms_ else 0.0}
            for cls, (ms_, work, n_) in prof.items()}
    conv_ms = sum(v["ms_per_call"] for k, v in kern.items() if not k.startswith("rvq"))
    enc_gbps = ENC_BYTES_PER_CLIP * clips / (conv_ms * 1e-3) / 1e9 if conv_ms else 0.0
    return {"metric": "SoundStream frames/sec encode", "value": frames / (ms * 1e-3), "unit": "frames/s",
            "ms_per_call": ms, "clips": clips, "samples_per_clip": 48000, "kernels": kern,
            "encoder_convs": {"ms": conv_ms, "algorithmic_gbps": enc_gbps, "frac_of_hbm_peak": enc_gbps / pk["hbm"],
                              "algorithmic_bytes": ENC_BYTES_PER_CLIP * clips},
            "decode": {"frames_per_s": frames / (ms_dec * 1e-3), "ms_per_call": ms_dec},
            "default_ctor_with_local_attn": None if ms_default is None else
            {"frames_per_s": frames / (ms_default * 1e-3), "ms_per_call": ms_default},
            "config": "use_local_attn=False (the kernels the north star names); default_ctor_with_local_attn adds the "
                      "LocalTransformer bottleneck"}


# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configs (extra keys of the N=1 line)
# ------------------------------------------------------------------------------------------------
def _no_repeat(ids, vocab):
    for i in range(1, ids.shape[1]):
        same = ids[:, i] == ids[:, i - 1]
        ids[:, i] = torch.where(same, (ids[:, i] + 1) % vocab, ids[:, i])
    return ids


def _train_bench(wrapper, model, call, positions, steps, dev):
    from audiolm_pytorch_b200.parallel import FlatGradBucket

    bucket = FlatGradBucket(model.parameters()).attach(model)

    def step():
        bucket.zero_()
        model.transformer.invalidate_weight_cache()
        model._heads.clear()
        call(wrapper).backward()

    ms = _timed_cuda(step, steps, warm=3)
    return {"tokens_per_s": positions / (ms * 1e-3), "ms_per_step": ms, "positions_per_step": positions}


def config_c2(dev, steps=5):
    """C2: SemanticTransformerWrapper.forward(return_loss=True), batch 8 x 1024 positions (wrapper defaults)."""
    from audiolm_pytorch_b200 import SemanticTransformer, SemanticTransformerWrapper

    torch.manual_seed(2)
    m = SemanticTransformer(num_semantic_tokens=500, dim=1024, depth=6, heads=8, flash_attn=True).to(dev)
    w = SemanticTransformerWrapper(transformer=m).train()
    ids = _no_repeat(torch.randint(0, 500, (8, 1023)), 500).to(dev)
    return _train_bench(w, m, lambda w_: w_(semantic_token_ids=ids, return_loss=True), 8 * 1024, steps, dev)


def config_c4(dev, steps=5):
    """C4: FineTransformerWrapper.forward(return_loss=True), batch 16 x (1 + 768 + 1 + 1279 = 2049) positions."""
    from audiolm_pytorch_b200 import FineTransformer, FineTransformerWrapper

    torch.manual_seed(4)
    m = FineTransformer(num_coarse_quantizers=3, num_fine_quantizers=5, codebook_size=1024, dim=1024, depth=6, heads=8,
                        flash_attn=True).to(dev)
    w = FineTransformerWrapper(transformer=m, codec=_CodecStub()).train()
    coarse = torch.randint(0, 1024, (16, 256, 3), device=dev)
    fine = torch.randint(0, 1024, (16, 256, 5), device=dev)
    return _train_bench(w, m, lambda w_: w_(coarse_token_ids=coarse, fine_token_ids=fine, return_loss=True),
                        16 * 2049, steps, dev)


def config_c5(dev, window=120):
    """C5: KV-cache decode latency, batch 1: ms per generated token of the three generate() loops (wall clock around
    the public call, one warm-up call that also captures the decode graphs), median of 3."""
    from audiolm_pytorch_b200 import (CoarseTransformer, CoarseTransformerWrapper, FineTransformer,
                                      FineTransformerWrapper, SemanticTransformer, SemanticTransformerWrapper)

    torch.manual_seed(5)
    kw = dict(dim=1024, depth=6, heads=8, flash_attn=True)
    out = {}

    def timed(name, fn, count):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3 / max(count(r), 1))
        out[name] = {"ms_per_token": sorted(ts)[1]}

    sem = SemanticTransformerWrapper(transformer=SemanticTransformer(num_semantic_tokens=500, **kw).to(dev),
                                     unique_consecutive=False)
    timed("semantic", lambda: sem.generate(max_length=window, batch_size=1), lambda r: int(r.shape[1]))
    del sem
    coarse = CoarseTransformerWrapper(transformer=CoarseTransformer(num_semantic_tokens=500, codebook_size=1024,
                                                                    num_coarse_quantizers=3, **kw).to(dev),
                                      codec=_CodecStub(), unique_consecutive=False)
    sem_ids = torch.randint(0, 500, (1, 500), device=dev)
    timed("coarse", lambda: coarse.generate(semantic_token_ids=sem_ids, max_time_steps=window // 3),
          lambda r: window // 3 * 3)
    del coarse
    fine = FineTransformerWrapper(transformer=FineTransformer(num_coarse_quantizers=3, num_fine_quantizers=5,
                                                              codebook_size=1024, **kw).to(dev), codec=_CodecStub())
    c_ids = torch.randint(0, 1024, (1, window // 5, 3), device=dev)
    timed("fine", lambda: fine.generate(coarse_token_ids=c_ids), lambda r: window // 5 * 5)
    out["window_tokens"] = window
    out["stack_step"] = decode_stack_step_us(dev)
    return out


def decode_stack_step_us(dev, cache_len=600):
    """device time of ONE decode step of the d1024 L6 stack (batch 1, 600 cached positions), replayed from a CUDA graph:
    the one-kernel step (alm_decode_stack_step) beside the multi-kernel step it replaced."""
    from audiolm_pytorch_b200 import decode
    from audiolm_pytorch_b200.transformer import Transformer

    tr = Transformer(dim=1024, depth=6, heads=8, flash_attn=True).to(dev).eval()
    res = {"cache_len": cache_len}
    for fused in (False, True):
        decode.FUSED_STACK_STEP = fused
        try:
            dec = decode.StackDecoder(tr, 1, 2048)
            dec.load_cache(torch.randn(6, 2, 1, cache_len, 64, device=dev))
            x = torch.randn(1, 1024, device=dev)
            y = torch.zeros(1, 1024, device=dev, dtype=torch.bfloat16)
            g = decode.GraphedStep(lambda: y.copy_(dec.step(x)), [dec.len, y])
            for _ in range(10):
                g()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(100):
                g()
            e1.record()
            torch.cuda.synchronize()
            res["one_kernel_us" if fused else "multi_kernel_us"] = round(e0.elapsed_time(e1) * 10, 1)
        finally:
            decode.FUSED_STACK_STEP = True
    return res


def gemm_traffic_from_profile():
    """DRAM bytes (read + write) per GEMM launch from the committed ncu capture of this command's step
    (`--metrics dram__bytes_read.sum,dram__bytes_write.sum`): parsed at run time from profiles/, newest round first."""
    import csv
    for name in ("r02_ncu_gemm_dram_bytes_per_launch_one_step.csv", "r01_ncu_gemm_dram_bytes_per_launch_one_step.csv"):
        f = ROOT / "profiles" / name
        if not f.exists():
            continue
        total, ids = 0.0, set()
        for row in csv.reader(open(f, errors="replace")):
            # (the fused head + cross-entropy instantiation <BN, 0, 0, 1> is its own class, `gemm_head_ce_fused`)
            if len(row) >= 15 and row[0].isdigit() and "gemm_bf16_tcgen05" in row[4] and ", 1>(" not in row[4] \
                    and row[12].startswith("dram__bytes"):
                total += float(row[14])
                ids.add(row[0])
        if ids:
            return total / len(ids), f"profiles/{name} ({len(ids)} launches)"
    return None, None


DUMP_GRAD_SAMPLES = 1 << 22  # 16 MB of the ~260 MB fp32 gradient; the whole dump stays far below 64 MB


def last_step_outputs(loss, bucket):
    """what a caller of the timed step gets back: the loss and every parameter's .grad.  The gradients are dumped as
    one float64 L2 norm per parameter (in model.parameters() order) and the flat fp32 gradient at a fixed, seeded
    sample of positions, so two builds can be compared element by element without writing all of it."""
    bucket.sync_views()
    g = torch.Generator().manual_seed(0)
    n = min(DUMP_GRAD_SAMPLES, bucket.numel)
    idx = torch.randint(0, bucket.numel, (n,), generator=g).sort().values.to(bucket.flat.device)
    norms = torch.stack([torch.linalg.vector_norm(p.grad, dtype=torch.float64) for p in bucket.params])
    return {"loss": loss.float().cpu().numpy(),
            "grad_norm": norms.cpu().numpy(),
            "grad_sample": bucket.flat[idx].cpu().numpy()}


def write_outputs(out_dir, arrays):
    import numpy as np

    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)


# ------------------------------------------------------------------------------------------------
# our CUDA path
# ------------------------------------------------------------------------------------------------
def main_ours(args):
    import torch.distributed as dist

    from audiolm_pytorch_b200 import _lib, ops
    from audiolm_pytorch_b200.audiolm import CoarseTransformer, CoarseTransformerWrapper
    from audiolm_pytorch_b200.heads import cross_entropy
    from audiolm_pytorch_b200.parallel import FlatGradBucket

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    torch.manual_seed(1234)
    model = CoarseTransformer(**CFG).to(dev).train()
    wrapper = CoarseTransformerWrapper(transformer=model, codec=_CodecStub()).train()  # reference defaults
    bucket = FlatGradBucket(model.parameters()).attach(model)
    # default: ONE ncclAvg all-reduce of the flat bucket after the backward.  Overlapping (half / per layer) was measured
    # at N=2 on B200 and lost both times (profiles/r02_allreduce_n2.md): the persistent GEMMs own all 148 SMs
    overlap = world > 1 and os.environ.get("ALM_OVERLAP_ALLREDUCE", "0") != "0"
    if overlap:
        # the upper half of the stack (layers depth/2 .. depth-1: ~half of the bucket) is all-reduced on NCCL's stream
        # as soon as its gradients are final, under the backward of the lower half; finish() sends the rest.
        # (ALM_OVERLAP_ALLREDUCE=layers: one collective per layer - measured slower in round 1; =0: single all-reduce)
        layers = model.transformer.layers
        ranges = [bucket.range_of(list(layer.parameters())) for layer in layers]
        if os.environ.get("ALM_OVERLAP_ALLREDUCE") == "layers":
            model.transformer.grad_ready_hook = lambda i: bucket.reduce_range_async(*ranges[i])
        else:
            mid = len(layers) // 2
            lo, hi = ranges[mid][0], ranges[-1][1]
            model.transformer.grad_ready_hook = lambda i: bucket.reduce_range_async(lo, hi) if i == mid else None
    n_params = bucket.numel

    wsem_h, wco_h = synth_wrapper_ids(BATCH, rank)
    wsem_pin, wco_pin = wsem_h.pin_memory(), wco_h.pin_memory()
    wsem_d, wco_d = wsem_h.to(dev), wco_h.to(dev)
    sem_d, coarse_d = (t.to(dev) for t in synth_ids(BATCH, rank))
    eos = torch.full((BATCH, 1), CFG["codebook_size"], device=dev)

    NO_COLLECTIVE = os.environ.get("ALM_BENCH_NO_COLLECTIVE") is not None  # diagnostic only: N ranks, no exchange

    def prep():
        bucket.zero_()
        # a real training step sees new weights every iteration: rebuild the bf16 operand copies inside the
        # timed region (what bf16 autocast does at every Linear) instead of reusing last step's cache
        model.transformer.invalidate_weight_cache()
        model._heads.clear()

    def step(sem, coarse):
        """the trainer's step: wrapper forward with its key mask + forgetful causal mask, loss, backward, all-reduce"""
        prep()
        loss = wrapper(semantic_token_ids=sem, coarse_token_ids=coarse, return_loss=True)
        loss.backward()
        if not NO_COLLECTIVE:
            bucket.finish()  # N > 1: all-reduce of the flat bucket (whatever the overlap hook has not sent yet), mean
        return loss

    def step_direct():
        """variant (a): bare CoarseTransformer.forward, pure causal attention (no key mask)"""
        prep()
        coarse_labels = torch.cat((coarse_d, eos), dim=1)
        sl, cl = model(semantic_token_ids=sem_d, coarse_token_ids=coarse_d)
        n_s, n_c = sl.shape[1], cl.shape[1]
        loss = (cross_entropy(sl, sem_d) * n_s + cross_entropy(cl, coarse_labels) * n_c) / (n_s + n_c)
        loss.backward()
        bucket.finish()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for _ in range(max(args.warmup, 3)):
        step(wsem_d, wco_d)

    # ---- device-resident timing ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    _lib.reset_launch_count()
    last_loss = [None]

    def headline_step():
        last_loss[0] = step(wsem_d, wco_d).detach()

    ms_total = timed(headline_step, args.steps)
    launches = _lib.launch_count() / args.steps
    outputs = last_step_outputs(last_loss[0], bucket) if args.dump_outputs and rank == 0 else None

    # ---- end to end: pinned host ids -> device, loss -> host, every step ----
    def e2e_step():
        s = wsem_pin.to(dev, non_blocking=True)
        c = wco_pin.to(dev, non_blocking=True)
        return step(s, c).item()

    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    clocks = sampler.stop() if sampler else None   # sampled over both timed regions (device-resident + end-to-end)

    # ---- variant (a): no key mask ----
    for _ in range(2):
        step_direct()
    n_direct = max(3, args.steps // 2)
    ms_direct = timed(step_direct, n_direct) / n_direct

    # ---- collective alone (N > 1): the flat-bucket all-reduce timed on its own, max over ranks ----
    ms_allreduce = None
    if world > 1:
        bucket.all_reduce_mean()
        ms_allreduce = timed(lambda: bucket.all_reduce_mean(), 5) / 5

    # ---- roofline of the dominant kernel class (tcgen05 GEMM), events on the launching stream ----
    barrier()
    ops.profile_start()
    for _ in range(2):
        step(wsem_d, wco_d)
    prof = ops.profile_stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    tokens = world * BATCH * SEQ
    ms_step = ms_total / args.steps
    g_ms, g_flops, g_n = prof.get("gemm_bf16_tcgen05", (0.0, 0.0, 0))
    achieved = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    kern = {}
    for cls, (ms_, work, n_) in prof.items():
        rate = work / (ms_ * 1e-3) if ms_ else 0.0
        kern[cls] = {"ms_per_step": ms_ / 2, "launches_per_step": n_ / 2}
        if ops.CLASS_UNIT.get(cls) == "byte":  # HBM-bound classes: algorithmic bytes / time vs the measured copy peak
            kern[cls].update(gbps=rate / 1e9, frac_of_hbm_peak=rate / 1e9 / pk["hbm"] if pk.get("hbm") else None)
        else:
            kern[cls]["tflops"] = rate / 1e12
    traffic, traffic_src = gemm_traffic_from_profile()
    step_tflop = 388e6 * BATCH * SEQ / 1e12  # SURVEY 8(d): 388 MFLOP/token fwd+bwd

    line = {
        "metric": METRIC, "value": tokens / (ms_step * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD + ((" + grad all-reduce" + (" (overlapped with the backward)" if overlap else "")) if world > 1 else ""),
                   "global_batch": world * BATCH, "seq_len": SEQ, "parallelism": f"dp{world}", "params": n_params,
                   "l2": "working set (~9 GB of saved activations per step) far exceeds the 126 MB L2"},
        "e2e": {"value": tokens / (ms_e2e / args.steps * 1e-3), "unit": "tokens/s",
                "h2d_bytes_per_step": (wsem_pin.numel() + wco_pin.numel()) * 8, "d2h_bytes_per_step": 4},
        "gpu_launches": launches,
        **({"diagnostic": "ALM_BENCH_NO_COLLECTIVE: gradient exchange skipped, NOT a valid multi-GPU number"} if NO_COLLECTIVE else {}),
        "clocks": clocks,
        "variants": {"direct_causal": {"tokens_per_s": tokens / (ms_direct * 1e-3), "ms_per_step": ms_direct,
                                       "what": "CoarseTransformer.forward without key mask + the same two CE + bwd"}},
        "step_mfu": {"algorithmic_tflop_per_step_per_gpu": step_tflop,
                     "achieved_tflops": step_tflop / (ms_step * 1e-3), "peak": pk["tf_sustained"],
                     "frac": step_tflop / (ms_step * 1e-3) / pk["tf_sustained"]},
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel (all fwd/dgrad/wgrad launches of a step)",
                     "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / pk["tf_sustained"] if pk["tf_sustained"] else None,
                     "traffic": traffic, "traffic_unit": "DRAM bytes (read + write) per launch, class average",
                     "traffic_source": traffic_src,
                     "algorithmic_flops_per_launch": g_flops / g_n if g_n else None,
                     "peak_source": pk["src"] + ", sustained figure (kernel timed inside a long step)"},
        "kernels": kern,
    }
    if ms_allreduce is not None:
        line["collective"] = {"what": f"all-reduce of the {n_params * 4 / 1e6:.0f} MB fp32 flat gradient bucket + 1/N",
                              "ms_alone": ms_allreduce,
                              "busbw_gbps": 2 * (world - 1) / world * n_params * 4 / (ms_allreduce * 1e-3) / 1e9}
    if world == 1 and not args.headline_only:
        del wrapper, model, bucket
        torch.cuda.empty_cache()
        cfgs = {}
        for name, fn in (("C1_soundstream", codec_bench), ("C2_semantic_b8_n1024", config_c2),
                         ("C4_fine_b16_n2049", config_c4), ("C5_decode_b1", config_c5)):
            try:
                cfgs[name] = fn(dev)
            except Exception as e:  # pragma: no cover
                cfgs[name] = {"error": repr(e)}
            torch.cuda.empty_cache()
        line["configs"] = cfgs
        line["soundstream_encode"] = cfgs["C1_soundstream"]
    if not args.no_cpu:
        try:
            tps, ms_cpu, cores = run_cpu(steps=1, warmup=1)
            line["cpu_baseline"] = {"value": tps, "unit": "tokens/s", "cores": cores, "kind": "port",
                                    "sample": f"1 warm-up + 1 timed fwd+bwd of batch 1 x {SEQ} tokens, fp32 oracle port "
                                              "(restatement of the reference's modules; /root/reference is absent on the GPU box)"}
        except Exception as e:  # pragma: no cover
            line["cpu_baseline"] = {"error": repr(e)}
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the bounded CPU baseline leg")
    ap.add_argument("--headline-only", action="store_true", help="skip the extra C1/C2/C4/C5 legs of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of the last timed step as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
    # NCCL / torch may print banners ("NCCL version ...") on fd 1: keep stdout for the JSON line only
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        main_reference(a)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback); "
                             "use --impl reference for the CPU arm")
        main_ours(a)
