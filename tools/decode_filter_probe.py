"""Cost of the top-k / top-p logit filters in the decode kernels: whole multistart sampling rollouts (RRNetPolicy.forward
with a fixed encoder output), unfiltered vs top_k=10 vs top_p=0.9, timed with CUDA events after a warm-up of every shape.
  * config C3's shape, RCVRPTW n=100, 1024 instances x 100 starts, and RCVRP n=100, 1024 x 100 (lean engine);
  * ATSP n=200, 64 x 100 starts: filtered calls run the per-step pipeline, unfiltered ones the key-tiled fused kernel.
   python tools/decode_filter_probe.py [--reps 5]"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rrnco_b200 as rb  # noqa: E402
from oracle import synth, model as omodel  # noqa: E402  (input generator + default-initialised weights only)

dev = torch.device("cuda", 0)
SHAPES = [("rcvrptw", 100, 1024, 100), ("rcvrp", 100, 1024, 100), ("atsp", 200, 64, 100)]
FILTERS = [("unfiltered", {}), ("top_k=10", dict(top_k=10)), ("top_p=0.9", dict(top_p=0.9))]


def gpu_label():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{torch.cuda.get_device_name(dev)}, power limit {pl}"


def setup(name, n, B):
    raw = synth.make_instances(name, B, n, seed=1)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(rb.TensorDictLite({k: v.to(dev) for k, v in raw.items()}, batch_size=[B]))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=2)
    row, col = row.to(dev), col.to(dev)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col

    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(omodel.init_decoder_params(name, seed=1234))
    return env, td, pol


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decode_filter_probe needs a CUDA device")
    rb.set_precision(3)
    print(f"# decode_filter_probe on {gpu_label()}; multistart sampling rollouts, median of {args.reps} after 2 warm-up calls")
    for name, n, B, S in SHAPES:
        env, td, pol = setup(name, n, B)
        base = None
        for label, fk in FILTERS:
            run = lambda: pol(td, env, phase="val", decode_type="multistart_sampling", num_starts=S, seed=7, **fk)
            with torch.no_grad():
                for _ in range(2):
                    run()
                times = []
                for _ in range(args.reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    out = run()
                    e1.record()
                    torch.cuda.synchronize()
                    times.append(e0.elapsed_time(e1))
            ms = sorted(times)[len(times) // 2]
            base = ms if base is None else base
            path = "per-step pipeline" if (fk and n + (name != "atsp") > 128) else "fused kernel"
            print(f"{name} n={n} {B}x{S}: {label:10s} {ms:9.2f} ms ({ms / base:5.2f}x unfiltered; {path}; "
                  f"spread {min(times):.2f}-{max(times):.2f} ms; mean reward {out['reward'].float().mean().item():.4f})")


if __name__ == "__main__":
    main()
