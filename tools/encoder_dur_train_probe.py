"""Times one trainable rcvrptw DistAngleFusion (three-way duration gate, attn_freenet.py:242-289) at 101 nodes: the inference
kernel, the backward kernels (rrnco_train_nab_dur_backward) on their own, forward + backward through autograd with the peak
memory of it, at 1024 and 4096 instances; then upstream's op sequence (oracle/encoder.py) in torch autograd, fp32, at the
largest of 1024 / 512 / 256 instances that fits.   python tools/encoder_dur_train_probe.py [output file]"""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rrnco_b200 as rb  # noqa: E402
from rrnco_b200 import encoder_ops, train_ops  # noqa: E402
from oracle import encoder as oenc  # noqa: E402

dev = torch.device("cuda", 0)
N = 101
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def peak_rise(fn):
    """Largest rise of allocated device memory over what was allocated before the call, bytes."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = "nvidia-smi unavailable"
say(f"# {torch.cuda.get_device_name(dev)} | nvidia-smi: {card} | torch {torch.__version__}")
say("# CUDA events; every shape warmed up; times are per call of one module, N = 101 (10201 pairs per instance)")

torch.manual_seed(0)
m = rb.DistAngleFusion(128, use_duration_matrix=True, trainable=True, train_duration_gate=True).to(dev)
g = torch.Generator(device=dev).manual_seed(1)
for B in (1024, 4096):
    coords = torch.rand(B, N, 2, device=dev, generator=g)
    cost = torch.rand(B, N, N, device=dev, generator=g) * 1.4
    dur = torch.rand(B, N, N, device=dev, generator=g) * 2.0
    G = torch.randn(B, N, N, device=dev, generator=g)
    reps = 10 if B <= 1024 else 4
    with torch.no_grad():
        t_fwd = timed(lambda: m(coords, cost, dur), reps)
    packed = m._packed_duration()
    flat = torch.cat([p.detach().reshape(-1) for p in encoder_ops._dur_params(m)])
    t_bwd = timed(lambda: encoder_ops.nab_dur_gating_backward(coords, cost, dur, 0, packed, flat, 1.0, G), reps)

    def fwd_bwd():
        m(coords, cost, dur).backward(G)
    t_fb = timed(fwd_bwd, reps)
    rise = peak_rise(fwd_bwd)
    ws = train_ops.lib().rrnco_train_nab_dur_workspace_bytes(B, N)
    unit = B * N * N * 4
    say(f"B {B:5d}: forward kernel {t_fwd:8.3f} ms | backward kernels {t_bwd:8.3f} ms ({t_bwd / t_fwd:4.2f} x forward) | "
        f"forward + backward (autograd) {t_fb:8.3f} ms | peak rise {rise / 1e6:9.1f} MB = {rise / unit:4.2f} x B N^2 fp32 "
        f"(workspace {ws / 1e6:.2f} MB)")
    del coords, cost, dur, G
    torch.cuda.empty_cache()

# upstream's op sequence in torch autograd (fp32), largest batch that fits
ref = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
for B in (1024, 512, 256):
    try:
        coords = torch.rand(B, N, 2, device=dev, generator=g)
        cost = torch.rand(B, N, N, device=dev, generator=g) * 1.4
        dur = torch.rand(B, N, N, device=dev, generator=g) * 2.0
        G = torch.randn(B, N, N, device=dev, generator=g)

        def up():
            for v in ref.values():
                v.grad = None
            oenc.dist_angle_fusion(ref, coords, cost, dur).backward(G)
        rise = peak_rise(up)
        t_up = timed(up, 3)
    except torch.cuda.OutOfMemoryError:
        say(f"upstream op sequence, B {B:5d}: out of memory")
        coords = cost = dur = G = None
        torch.cuda.empty_cache()
        continue
    say(f"upstream op sequence, B {B:5d}: forward + backward {t_up:9.3f} ms | peak rise {rise / 1e9:7.2f} GB "
        f"= {rise / (B * N * N * 4):5.1f} x B N^2 fp32")
    break

if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write("\n".join(lines) + "\n")
