"""One full training step (fused sampling rollout, differentiable batched replay, backward; rrnco_b200/training.py) at instance
sizes beyond the single-tile replay kernels, on the kernels and, where its estimated peak memory fits, on the plain-torch (ATen)
form; then the key-tiled and the single-tile attention kernels at N = 101, forward and backward, timed with CUDA events.
   python tools/train_large_n_probe.py"""
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rrnco_b200 as rb  # noqa: E402
from rrnco_b200 import training, train_ops  # noqa: E402
from oracle import synth, model as omodel  # noqa: E402  (input generator + default-initialised weights only)

dev = torch.device("cuda", 0)
SHAPES = [("rcvrp", 100, 512, 101), ("rcvrp", 200, 128, 201), ("atsp", 1000, 32, 100)]
# ATen replay, measured at N = 101 (profiles/r2_train_step_probe_final.txt): 47 GiB for 512 x 101 starts x ~125 steps; most of it
# is [rows, N] fp32 intermediates, so the estimate scales the bytes per row with N (an upper estimate: part does not grow with N)
ATEN_BYTES_PER_ROW_AT_101 = 47 * 2 ** 30 / (512 * 101 * 125)


def gpu_label():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{torch.cuda.get_device_name(dev)}, power limit {pl}"


def sync_time():
    torch.cuda.synchronize()
    return time.perf_counter()


def setup(name, n, B):
    raw = synth.make_instances(name, B, n, seed=1)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(rb.TensorDictLite({k: v.to(dev) for k, v in raw.items()}, batch_size=[B]))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=2)
    row, col = row.to(dev).requires_grad_(True), col.to(dev).requires_grad_(True)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col

    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(omodel.init_decoder_params(name, seed=1234))
    return env, td, pol, row, col, N


def step(env, td, pol, row, col, S, name):
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    t0 = sync_time()
    with torch.no_grad():
        out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S)
    t1 = sync_time()
    inputs = rb.iter_decode_inputs(pol.decoder, env, td, out["actions"], S)   # consumed chunk by chunk: env replay overlaps
    dur = td["duration_matrix"].float() if name == "rcvrptw" else None
    logp = rb.batched_logprobs(pol.decoder, row, col, td["distance_matrix"].float(), dur, inputs, out["actions"], S)
    ll = logp.sum(1)
    loss = rb.pomo_shared_baseline_loss(out["reward"], ll, S)
    t2 = sync_time()
    loss.backward()
    t3 = sync_time()
    err = (ll - out["log_likelihood"]).abs().max().item()
    peak = torch.cuda.max_memory_allocated(dev) - base
    pol.zero_grad(set_to_none=True)
    row.grad = col.grad = None
    return dict(sample=t1 - t0, fwd=t2 - t1, bwd=t3 - t2, total=t3 - t0, err=err, peak=peak, T=out["actions"].shape[1])


def run_shapes():
    for name, n, B, S in SHAPES:
        env, td, pol, row, col, N = setup(name, n, B)
        for impl in ("fused", "aten"):
            training.REPLAY_IMPL = impl
            try:
                if impl == "aten":
                    est = ATEN_BYTES_PER_ROW_AT_101 * N / 101 * B * S * (last["T"] - 1)
                    free, total = torch.cuda.mem_get_info(dev)
                    if est > 0.7 * free:
                        print(f"{name} n={n} B={B} S={S} aten replay: not run (estimated peak {est / 2 ** 30:.0f} GiB, "
                              f"{free / 2 ** 30:.0f} GiB free)")
                        continue
                step(env, td, pol, row, col, S, name)          # warm-up
                runs = [step(env, td, pol, row, col, S, name) for _ in range(2)]
            finally:
                training.REPLAY_IMPL = "fused"
            r = min(runs, key=lambda x: x["total"])
            last = r
            print(f"{name} n={n} B={B} S={S} T={r['T']} {impl} replay: sample {1e3 * r['sample']:7.1f} ms | env replay + fwd "
                  f"{1e3 * r['fwd']:7.1f} | bwd {1e3 * r['bwd']:7.1f} | total {1e3 * r['total']:7.1f} ms = {B / r['total']:7.1f} "
                  f"instances/s | peak rise {r['peak'] / 2 ** 30:6.1f} GiB | max |ll - kernel ll| {r['err']:.1e}")
        del env, td, pol, row, col
        torch.cuda.empty_cache()


def time_attention_101(reps=20):
    """Single-tile vs key-tiled attention kernels at N = 101 on one replay chunk of the C5 shape (512 instances x 32 steps x 101
    starts), forward and backward, CUDA events over `reps` launches after a warm-up."""
    n_inst, L, N = 512, 32 * 101, 101
    g = torch.Generator(device=dev).manual_seed(0)
    q = torch.randn(n_inst, L, 128, device=dev, generator=g)
    k = torch.randn(n_inst, N, 128, device=dev, generator=g)
    v = torch.randn(n_inst, N, 128, device=dev, generator=g)
    mask = torch.rand(n_inst, L, N, device=dev, generator=g) < 0.5
    mask[..., 0] = True
    d_out = torch.randn(n_inst, L, 128, device=dev, generator=g) * 1e-6
    h, st = train_ops.lib(), train_ops._stream(dev)
    P = train_ops._p
    m8 = mask.view(torch.uint8)
    res = {}
    for form in ("single", "tiled"):
        out, lse = torch.empty_like(q), torch.empty(n_inst, L, 8, device=dev)
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        ws = torch.empty(max(1, h.rrnco_train_attention_tiled_workspace_bytes(n_inst, L, N)), dtype=torch.uint8, device=dev)
        if form == "single":
            fwd = lambda: h.rrnco_train_attention_fwd(n_inst, L, N, P(q), P(k), P(v), P(m8), 1, P(out), P(lse), st)  # noqa: E731
            bwd = lambda: h.rrnco_train_attention_bwd(n_inst, L, N, P(q), P(k), P(v), P(m8), P(out), 1, P(lse), P(d_out),  # noqa: E731
                                                      P(dq), P(dk), P(dv), st)
        else:
            fwd = lambda: h.rrnco_train_attention_tiled_fwd(n_inst, L, N, P(q), P(k), P(v), P(m8), 1, P(out), P(lse), st)  # noqa: E731
            bwd = lambda: h.rrnco_train_attention_tiled_bwd(n_inst, L, N, P(q), P(k), P(v), P(m8), P(out), 1, P(lse),  # noqa: E731
                                                            P(d_out), P(ws), P(dq), P(dk), P(dv), st)
        for which, fn in (("fwd", fwd), ("bwd", bwd)):
            assert fn() == 0
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[form, which] = e0.elapsed_time(e1) / reps
        res[form, "out"] = (out.clone(), dq.clone(), dk.clone(), dv.clone())
    same = [bool(torch.equal(a, b)) for a, b in zip(res["single", "out"], res["tiled", "out"])]
    rel = [float((a - b).abs().max() / b.abs().max()) for a, b in zip(res["tiled", "out"], res["single", "out"])]
    print(f"attention at N = 101, {n_inst} x {L} rows: single-tile fwd {res['single', 'fwd']:.2f} ms, bwd {res['single', 'bwd']:.2f} ms | "
          f"key-tiled fwd {res['tiled', 'fwd']:.2f} ms, bwd {res['tiled', 'bwd']:.2f} ms | bitwise equal (out, dq, dk, dv) {same} | "
          f"max rel diff {', '.join(f'{x:.1e}' for x in rel)}")


if __name__ == "__main__":
    print(gpu_label())
    time_attention_101()
    run_shapes()
    train_ops.check_status(dev)
