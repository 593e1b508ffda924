"""Cost of beam search: whole RRNetPolicy.forward calls with a fixed encoder output, beam_search (all beams kept,
select_best=False) against multistart greedy at the same instances x width, timed with CUDA events after a warm-up of
every shape.  Beam search runs the per-step kernel pipeline (rrnco_decoder_logits[_large] -> rrnco_beam_select -> env
step, then rrnco_beam_backtrack); multistart greedy runs the fused rollout kernel.  On the first decode step's inputs it
also times one decoder step (RRNetDecoder.forward) and rrnco_beam_select alone, median of 20 calls each.
  * RCVRPTW n=100 and RCVRP n=100, 1024 instances x 100 beams / starts;
  * ATSP n=200, 64 x 100.
   python tools/beam_search_probe.py [--reps 5]"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rrnco_b200 as rb  # noqa: E402
from rrnco_b200 import models  # noqa: E402
from oracle import synth, model as omodel  # noqa: E402  (input generator + default-initialised weights only)

dev = torch.device("cuda", 0)
SHAPES = [("rcvrptw", 100, 1024, 100), ("rcvrp", 100, 1024, 100), ("atsp", 200, 64, 100)]


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


def step_times(env, td, pol, name, W, reps=20):
    """(decoder step ms, beam select ms) on the inputs of the first decode step after the starts."""
    B = td["action_mask"].shape[0]
    keys = models._ROLLOUT_STATE_KEYS[name]
    with torch.no_grad():
        cache = pol.decoder._precompute_cache(pol.encoder(td), num_starts=W)
        roll = rb.TensorDictLite({k: (rb.batchify(td[k], W) if k in keys else td[k]) for k in td.keys() if k != "done"},
                                 batch_size=[B * W])
        roll.set("action", env.select_start_nodes(td, W))
        roll = env.step(roll)["next"]
        logits, mask = pol.decoder(roll, cache, W)
        score = torch.zeros(B * W, device=dev)
        out = []
        for fn in (lambda: pol.decoder(roll, cache, W), lambda: rb.beam_select(logits, mask, score, W)):
            fn()
            times = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            out.append(sorted(times)[len(times) // 2])
    return out


def timed(run, reps):
    with torch.no_grad():
        for _ in range(2):
            run()
        times = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    return sorted(times)[len(times) // 2], times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("beam_search_probe needs a CUDA device")
    rb.set_precision(3)
    print(f"# beam_search_probe on {gpu_label()}; median of {args.reps} after 2 warm-up calls")
    for name, n, B, W in SHAPES:
        env, td, pol = setup(name, n, B)
        ms_g, t_g, out_g = timed(lambda: pol(td, env, phase="test", decode_type="multistart_greedy", num_starts=W), args.reps)
        ms_b, t_b, out_b = timed(lambda: pol(td, env, phase="test", decode_type="beam_search", beam_width=W,
                                             select_best=False), args.reps)
        best_g = out_g["reward"].view(W, B).max(0)[0].mean().item()
        best_b = out_b["reward"].view(W, B).max(0)[0].mean().item()
        T = out_b["actions"].shape[1]
        print(f"{name} n={n} {B}x{W}: multistart greedy {ms_g:9.2f} ms (fused kernel; spread {min(t_g):.2f}-{max(t_g):.2f}); "
              f"beam search {ms_b:9.2f} ms (per-step pipeline, {T} steps, {ms_b / T * 1e3:.0f} us/step; spread "
              f"{min(t_b):.2f}-{max(t_b):.2f}); {ms_b / ms_g:6.2f}x; mean best reward greedy {best_g:.4f}, beam {best_b:.4f}")
        t_dec, t_sel = step_times(env, td, pol, name, W)
        print(f"{name} n={n} {B}x{W}: first beam step: decoder {t_dec * 1e3:7.0f} us, rrnco_beam_select {t_sel * 1e3:7.0f} us "
              f"({t_sel / (t_dec + t_sel):.0%} of the two)")


if __name__ == "__main__":
    main()
