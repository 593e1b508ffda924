#!/usr/bin/env python
"""bench.py -- RCVRP n=100 POMO rollout throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path (fused construction rollout: decode loop + env step + reward) over one
batch of BASELINE config[1]: RCVRP n=100, 1024 instances x 8 augmentations x 101 POMO starts, greedy.
Instances are independent, so each rank owns its own 1024 instances (weak scaling, no data-path collective);
the only collective is one all-gather of the best costs per step.

Printed JSON line (rank 0): see the contract in the task statement; extra keys
  roofline      dominant kernel (rollout_lean_kernel): bound "tensor" -- algorithmic FLOP/s (SURVEY.md 8(d): 373 kFLOP per
                rollout-step x the rollout-steps the tiles actually ran) against the measured bf16 peak, the issued-MMA
                figure (three-term split, padded rows / keys) beside it, and the HBM-algorithmic figure of the north star
                (3.2 KB per rollout-step) as `hbm_algorithmic`; `traffic` = measured DRAM bytes of this build (ncu)
  cpu_baseline  the CPU oracle (= line-faithful restatement of the reference's eager rollout) on this box's cores
  e2e           same metric through RRNetPolicy.forward with HOST (pinned) inputs, H2D/D2H inside the timing
  configs       one short measured line per other BASELINE config: C1 ATSP n=100 batch 32 x8 aug, C3 RCVRPTW n=100
                sampling batch 1024, C4 ATSP n=1000 batch 64, C5 RCVRP training rollouts (global batch 4096 sharded over
                the ranks = strong scaling, instances generated on the device from 1000-node city matrices)
`--impl reference` times the reference's own CPU path (oracle port; rl4co cannot be installed offline).
`--workload c5` makes config C5 the headline line (strong scaling of the fixed global batch).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_LOC, N_AUG, N_START = 100, 8, 101
BYTES_PER_ROLLOUT_STEP = 737 + 404 + 512 + 12 + 1536   # SURVEY.md 8(d): env step + bias row + ctx gather + out + K/V/Lk / S
FLOPS_PER_ROLLOUT_STEP = 373_000                        # SURVEY.md 8(d)


def algorithmic_per_rollout_step(env_name, N, S):
    """(bytes, flops) per rollout-step, SURVEY.md 8(d): env-step bytes + bias row(s) + context gather + 12 B out +
    K/V/Lk amortised over the S starts that share them; context proj + QK + PV + FFN + logits."""
    E = 128
    env_b = {"atsp": 2 * N + 50, "rcvrp": 7 * N + 30, "rcvrptw": 39 * N + 100}[env_name]
    bias_b = (8 if env_name == "rcvrptw" else 4) * N
    ctx_b = (8 if env_name == "atsp" else 4) * E
    k = {"atsp": E, "rcvrp": 1, "rcvrptw": 4}[env_name]
    flops = 2 * (E + k) * E + 3 * 2 * N * E + 2 * 2 * E * 4 * E
    return env_b + bias_b + ctx_b + 12 + 12 * N * E / S, flops


def issued_mma_flops_per_tile_step(N, passes=3):
    """Tensor-pipe FLOPs one 128-row tile issues per decode step in the fused kernel: operand terms of the fp16 split x
    padded shapes (128 rows, keys rounded up to 16): QK 8 heads, PV 8 heads x R16/16 K steps (N=16), FFN 64 K steps of
    128x128x16, logits 8 K steps."""
    R16 = (N + 15) // 16 * 16
    mma = lambda n: 2 * 128 * n * 16
    return passes * (8 * mma(R16) + 8 * (R16 // 16) * mma(16) + 64 * mma(128) + 8 * mma(R16))


def profile_stamp():
    """Measured DRAM bytes per launch from the ncu captures of THIS build (profiles/r2_traffic.json, stamped with the
    digest of the CUDA sources): a number taken from another build is not reported."""
    try:
        from rrnco_b200.build import build_digest
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        return d if d.get("build_digest") == build_digest() else {}
    except Exception:
        return {}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of the headline workload (the per-config block "
                                                          "times a fixed number of steps per config: C1 5, C3 5, C4 2, C5 5)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before the headline's timed steps")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="instances per GPU per step")
    ap.add_argument("--precision", type=int, default=3, choices=[1, 3], help="3 = three-term fp16-split contractions, fp32-faithful (headline); 1 = single fp16 pass")
    ap.add_argument("--cpu-sample", type=int, default=16, help="instances in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block (C1, C3, C4, C5)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"], help="headline workload: BASELINE config[1] (default) or config[4]")
    ap.add_argument("--c5-global-batch", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rollout outputs of the last timed headline step (rank 0) "
                                                          "to DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d["hbm_gbs"], d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md 8(d)): city-like asymmetric 1000-node matrix -> sub-sampled instances
# --------------------------------------------------------------------------------------------------
def make_city(city_id=0, length=1000):
    rng = np.random.default_rng(1000 + city_id)
    pts = rng.uniform(0.0, 3.0, size=(length, 2))
    eu = np.linalg.norm(pts[:, None, :] - pts[None, :, :], axis=-1)
    dist = eu * (1.2 + 0.4 * rng.uniform(size=(length, length)))
    np.fill_diagonal(dist, 0.0)
    speed = rng.uniform(20.0, 50.0, size=(length, length))  # km/h
    return {"points": pts, "distance": dist, "duration": dist / speed * 60.0}


def host_instances(batch, seed):
    """Raw instance batch on the HOST (what a DataLoader hands to env.reset): fp32, pinned."""
    city = make_city(seed % 10)
    rng = np.random.RandomState(seed)
    idx = np.array([rng.choice(1000, N_LOC + 1, replace=False) for _ in range(batch)])
    dm = torch.from_numpy(city["distance"][idx[:, :, None], idx[:, None, :]].astype(np.float32))
    pts = torch.from_numpy(city["points"][idx].astype(np.float32))
    g = torch.Generator().manual_seed(seed)
    demand = torch.randint(1, 10, (batch, N_LOC), generator=g).float() / 50.0
    return {"locs": pts[:, 1:].contiguous(), "depot": pts[:, :1].contiguous(), "demand": demand, "distance_matrix": dm}


def stand_in_embeddings(n_inst, seed):
    """Encoder output stand-in (the encoder stays the reference's PyTorch module and is not on this path):
    unit-variance embeddings, as an instance-normalised encoder produces."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n_inst, N_LOC + 1, 128, generator=g), torch.randn(n_inst, N_LOC + 1, 128, generator=g)


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        """NVML from a Python thread (pynvml, ~20 Hz): no process start-up or driver re-initialisation inside the timed
        region, which an `nvidia-smi -lms` child costs.  Falls back to that child if NVML cannot be loaded."""
        self.rows, self.p, self.thread, self.stop_flag = [], None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES: map the CUDA ordinal to the NVML handle through the PCI bus id
            bus = torch.cuda.get_device_properties(gpu_index)
            h = None
            try:
                h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{bus.pci_domain_id:08x}:{bus.pci_bus_id:02x}:{bus.pci_device_id:02x}.0")
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self.stop_flag:
                    try:
                        self.rows.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                          pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons_fn(h))))
                    except Exception:
                        pass
                    time.sleep(0.05)
            import threading
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            try:
                self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                           "-i", str(gpu_index), "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
            except Exception:
                self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if not self.rows:
                return out
            sm = sorted(r[0] for r in self.rows)
            bits = 0
            for r in self.rows:
                bits |= r[2]
            # nvml.h: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            out.update({"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "power_w_max": max(r[1] for r in self.rows),
                        "reasons": [n for b, n in names.items() if bits & b], "samples": len(self.rows), "source": "nvml"})
            return out
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = float(rows[0][2])
        out["power_w_max"] = max(float(r[3]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out["reasons"] = [n for i, n in enumerate(names) if any("Active" in r[5 + i] and "Not" not in r[5 + i] for r in rows)]
        out["samples"] = len(rows)
        out["source"] = "nvidia-smi"
        return out


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle (line-faithful restatement of the reference's eager rollout) on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_rollout_rate(n_inst_sample, threads, seed=4242):
    from oracle import envs as oenvs, model as omodel
    from oracle.td import TD, batchify
    torch.set_num_threads(threads)
    raw = host_instances(n_inst_sample, seed)
    env = oenvs.RCVRPEnv(N_LOC, check_solution=False)
    p = omodel.init_decoder_params("rcvrp", seed=1234)
    row, col = stand_in_embeddings(n_inst_sample * N_AUG, seed)
    with torch.inference_mode():
        t0 = time.perf_counter()
        td = env.reset(TD(raw, batch_size=[n_inst_sample]))
        td = batchify(td, N_AUG)  # StateAugmentation = batchify(td, 8) (distance matrices identical across augs)
        out = omodel.policy_forward(p, env, td, row, col, decode_type="multistart_greedy", num_starts=N_START)
        best = out["reward"].view(N_START, N_AUG, n_inst_sample).amax(0).amax(0)
        dt = time.perf_counter() - t0
    return n_inst_sample / dt, dt, float(-best.mean()), int(out["actions"].shape[1])


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rates = []
    for i in range(args.warmup + args.steps):
        rate, dt, cost, T = cpu_rollout_rate(args.cpu_sample, threads, seed=4242 + i)
        if i >= args.warmup:
            rates.append((rate, dt))
    value = sum(args.cpu_sample for _ in rates) / sum(dt for _, dt in rates)
    sample = f"{args.cpu_sample} instances x {N_AUG} aug x {N_START} starts per step (bounded sample of the 1024-instance batch)"
    line = {
        "impl": "reference", "metric": "RCVRP n100 POMO rollout instances/s", "value": value, "unit": "instances/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(dt for _, dt in rates) / len(rates), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "RCVRP n=100 POMO multi-start x8 aug greedy rollout (BASELINE config[1])",
                   "num_starts": N_START, "n_aug": N_AUG, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "instances/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = CPU oracle port of the reference's eager rollout (rl4co/tensordict not installable offline)",
    }
    print(json.dumps(line), flush=True)


# (row-index file, outputs it selects, row budget): per-rollout vectors are whole up to 2^20 rollouts (the default 827 392
# fit); tours ([R, T] actions, T <= 2N) are a fixed sample of 2^14 rollouts (<= 13 MB at N = 101)
DUMP_GROUPS = (("rollout_rows", ("reward", "normalized_reward", "log_likelihood"), 1 << 20),
               ("tour_rows", ("actions",), 1 << 14))


def dump_outputs(out_dir, out):
    """What `fused_rollout` handed back in the last timed step, as float32 `.npy` files (node indices are exact in
    float32); at most ~33 MB.  Each group's rows are written beside it (`rollout_rows.npy`, `tour_rows.npy`, float64): all
    R rollouts in order, or, above the group's budget, a sorted sample drawn with a fixed seed.  Every file of an earlier
    dump in `out_dir` is removed first, so an output this rollout does not return is absent rather than stale."""
    os.makedirs(out_dir, exist_ok=True)
    for rows_name, names, _ in DUMP_GROUPS:
        for name in (rows_name, *names):
            if os.path.exists(os.path.join(out_dir, name + ".npy")):
                os.remove(os.path.join(out_dir, name + ".npy"))
    R = out["actions"].shape[0]
    for rows_name, names, k in DUMP_GROUPS:
        idx = torch.arange(R) if R <= k else torch.randperm(R, generator=torch.Generator().manual_seed(0))[:k].sort().values
        np.save(os.path.join(out_dir, rows_name + ".npy"), idx.numpy().astype(np.float64))
        for name in names:
            if name in out:
                np.save(os.path.join(out_dir, name + ".npy"), out[name][idx.to(out[name].device)].float().cpu().numpy())


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import rrnco_b200 as rb
    from rrnco_b200 import _lib
    from rrnco_b200.sharding import gather_costs

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        # NCCL prints its version banner to stdout when the first communicator is created; stdout carries exactly one
        # JSON line, so the file descriptor points at stderr until the communicator exists
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    rb.set_precision(args.precision)
    B, Bp = args.batch, args.batch * N_AUG
    env = rb.RCVRPEnv(generator_params={"num_loc": N_LOC}, check_solution=False, device=dev)

    # decoder weights: default-initialised RRNetDecoder, seed 1234 (experiment/rrnet.yaml:55)
    torch.manual_seed(1234)
    decoder = rb.RRNetDecoder(env_name="rcvrp").to(dev)

    class HostEncoder(torch.nn.Module):
        """Hands the (host, pinned) encoder output of the current batch to the policy."""
        def __init__(self):
            super().__init__()
            self.row = self.col = None

        def forward(self, td, phase=None):
            return self.row.to(dev, non_blocking=True), self.col.to(dev, non_blocking=True)

    enc = HostEncoder()
    policy = rb.RRNetPolicy(encoder=enc, decoder=decoder, env_name="rcvrp").to(dev)

    # StateAugmentation(dihedral8) of test.py:28,188 with the [N,N] matrices / demand rows left un-replicated (the kernels
    # read row r % data_rows): no 8-fold device copy of the instance data
    augment = rb.StateAugmentation(num_augment=N_AUG, augment_fn="dihedral8", no_aug_coords=False, share_instance_data=True)

    # two alternating batches so that consecutive steps never see the same inputs (and > L2: 1.7 GB of cache each)
    n_sets = 2
    host_sets, dev_sets = [], []
    for i in range(n_sets):
        raw = host_instances(B, seed=100 * (rank + 1) + i)
        row, col = stand_in_embeddings(Bp, seed=200 * (rank + 1) + i)
        raw = {k: v.pin_memory() for k, v in raw.items()}
        host_sets.append((raw, row.pin_memory(), col.pin_memory()))
        td_aug = env.reset(augment(rb.TensorDictLite({k: v.to(dev) for k, v in raw.items()}, batch_size=[B])))
        cache = decoder._precompute_cache((row.to(dev), col.to(dev)))
        dev_sets.append((td_aug, cache))
    torch.cuda.synchronize()

    def step_resident(i):
        td_aug, cache = dev_sets[i % n_sets]
        out = rb.fused_rollout(decoder, cache, env, td_aug, N_START, True, "greedy", check=False)
        best = rb.unbatchify(out["reward"], (N_AUG, N_START)).amax(-1).amax(-1)  # [B]  test.py:210-212
        if dist_on:
            gather_costs(best, world * B)  # the path's only collective (NCCL all-gather of [B] fp32 per rank)
        return out

    # e2e: every step copies its own batch from pinned host memory; the copy of step i+1 is issued on the copy stream
    # before step i's kernels (rrnco_b200.HostPrefetcher), so in steady state it overlaps the rollout of step i
    prefetch = rb.HostPrefetcher(dev)
    tickets = {}

    def host_batch(i):
        raw, row, col = host_sets[i % n_sets]
        return {**raw, "__row_emb": row, "__col_emb": col}

    def step_e2e(i):
        if i not in tickets:
            tickets[i] = prefetch.submit(host_batch(i))              # first call only
        tickets[i + 1] = prefetch.submit(host_batch(i + 1))          # H2D of the next step's batch
        ticket = tickets.pop(i)
        d = prefetch.acquire(ticket)
        enc.row, enc.col = d["__row_emb"], d["__col_emb"]
        td_aug = env.reset(augment(rb.TensorDictLite({k: v for k, v in d.items() if not k.startswith("__")}, batch_size=[B])))
        out = policy(td_aug, env, phase="val", decode_type="multistart_greedy", num_starts=N_START)
        best = rb.unbatchify(out["reward"], (N_AUG, N_START)).amax(-1).amax(-1)
        prefetch.release(ticket)
        return best.cpu()                                            # D2H of the result

    def barrier():
        torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        last = None
        for i in range(warmup):
            # keep the previous result alive while the next step runs, exactly as the timed loop does: otherwise the
            # second output set (867 MB of int64 actions) is first needed - and cudaMalloc'ed, ~100 ms - inside the
            # second timed step (seen as a 90-105 ms outlier there in three of six round-1 runs)
            last = fn(i)
        # no generation-2 pass of Python's cyclic collector inside the timed region either
        gc.collect()
        gc.disable()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        last = None
        marks = []
        for i in range(steps):
            last = fn(warmup + i)
            marks.append(torch.cuda.Event(enable_timing=True))
            marks[-1].record()
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        gc.enable()
        ms = max(e0.elapsed_time(e1), 0.0)
        if rank == 0:  # per-step device times (diagnostic only, stderr)
            ts = [e0.elapsed_time(m) for m in marks]
            print(f"[bench] {fn.__name__}: per-step ms " + " ".join(f"{b - a:.1f}" for a, b in zip([0.0] + ts[:-1], ts)), file=sys.stderr)
        if isinstance(last, torch.Tensor) and not last.is_cuda:
            ms = max(ms, wall * 1e3)  # e2e ends with a host-visible result: the wall clock bounds it
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist_on:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / steps, last

    if args.workload == "c5":
        # BASELINE config[4] as the headline: fixed GLOBAL batch sharded over the ranks (strong scaling)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        launches0 = _lib.kernel_count
        entry = measure_configs(args, rb, dev, rank, world, dist_on, timed, only=("C5",), steps=args.steps,
                                warmup=args.warmup, dump_dir=args.dump_outputs)["C5"]
        launches = (_lib.kernel_count - launches0) // (args.steps + args.warmup) * args.steps
        clocks = sampler.stop() if sampler else None
        if rank == 0:
            hbm_peak, tf_peak, peak_src = peaks()
            r = entry["roofline"]
            line = {"metric": "RCVRP n100 POMO training-rollout instances/s (global batch %d)" % args.c5_global_batch,
                    "value": entry["value"], "unit": "instances/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": entry["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "f32 (fp32-faithful: three-term fp16-split tcgen05 contractions, fp32 accumulate)",
                    "data": "synthetic (8 city-like asymmetric 1000-node matrices in HBM, instances sub-sampled on the device; "
                            "random-init decoder seed 1234; encoder output = stand-in embeddings)",
                    "config": {"workload": entry["workload"], "global_batch": args.c5_global_batch,
                               "instances_per_gpu": entry["instances_per_gpu"], "num_starts": entry["num_starts"],
                               "decode": entry["decode"], "l2_policy": "a fresh batch is generated every step (key cache 4 x 212 MB per 4096 instances >> L2)"},
                    "clocks": clocks, "gpu_launches": int(launches), "e2e": entry["e2e"],
                    "roofline": {"bound": "tensor", "achieved": r["tensor_algorithmic"]["achieved"], "peak": tf_peak,
                                 "unit": "TFLOP/s", "frac": r["tensor_algorithmic"]["frac"], "traffic": None,
                                 "peak_source": peak_src, "hbm_algorithmic": r["hbm_algorithmic"]},
                    "cpu_baseline": entry.get("cpu_baseline")}
            print(json.dumps(line), flush=True)
        if dist_on:
            dist.destroy_process_group()
        return

    # ---- value: inputs resident in HBM -------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = _lib.kernel_count
    ms_step, out = timed(step_resident, args.steps, args.warmup)
    launches = (_lib.kernel_count - launches0) // (args.steps + args.warmup) * args.steps
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    T = int(out["actions"].shape[1])
    tile_steps = out["tile_steps"].clone()
    value = world * B / (ms_step * 1e-3)

    # ---- dominant kernel alone (rollout + finalize), CUDA events on the launching stream -------------
    def kernel_only(i):
        td_aug, cache = dev_sets[i % n_sets]
        return rb.fused_rollout(decoder, cache, env, td_aug, N_START, True, "greedy", check=False)
    ms_kernel, _ = timed(kernel_only, args.steps, 2)

    # ---- standalone env-step and gather kernels (the "env-step HBM GB/s" half of the metric) ---------------
    def env_step_probe():
        # reference layout, the C2 rollout count: R = 8192 x 101 rollouts, one RCVRPEnv._step + get_action_mask
        # through the C ABI with pre-allocated outputs (610 MB of algorithmic traffic per launch, >> L2)
        from rrnco_b200._lib import call, ptr, stream_ptr
        td_aug, _ = dev_sets[0]
        R_probe = Bp * N_START
        N = N_LOC + 1
        g = torch.Generator(device=dev).manual_seed(0)
        demand = rb.batchify(rb.batchify(td_aug["demand"], N_AUG), N_START).contiguous()  # [R, N-1] as upstream's batchify
        cap = torch.ones(R_probe, device=dev)
        used = torch.rand(R_probe, device=dev, generator=g) * 0.5
        visited = (torch.rand(R_probe, N, device=dev, generator=g) < 0.3).to(torch.uint8)
        action = torch.randint(1, N, (R_probe,), device=dev, generator=g)
        used_o, vis_o = torch.empty_like(used), torch.empty_like(visited)
        cur_o = torch.empty(R_probe, dtype=torch.int64, device=dev)
        done_o = torch.empty(R_probe, dtype=torch.bool, device=dev)
        mask_o = torch.empty(R_probe, N, dtype=torch.bool, device=dev)

        def launch():
            call("rrnco_rcvrp_step", R_probe, N, R_probe, ptr(action), ptr(demand), ptr(cap), R_probe, ptr(used),
                 ptr(visited), None, ptr(used_o), ptr(vis_o), ptr(cur_o), ptr(done_o), ptr(mask_o), stream_ptr(dev))
        for _ in range(3):
            launch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            launch()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        nbytes = R_probe * (7 * N + 30)  # SURVEY.md 8(d): RCVRP 7N+30 B per rollout-step
        return {"kernel": "rrnco::rcvrp_step_kernel (RCVRPEnv._step + get_action_mask, reference layout)",
                "rollouts": R_probe, "ms_per_launch": ms, "algorithmic_bytes_per_launch": nbytes,
                "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s"}

    def time_launch(launch, reps=10, warm=3):
        for _ in range(warm):
            launch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            launch()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def atsp_step_probe():
        # ATSPEnv._step in the reference layout at the same rollout count (bool mask rows r/w + int64 scalars)
        from rrnco_b200._lib import call, ptr, stream_ptr
        R_probe, N = Bp * N_START, N_LOC
        g = torch.Generator(device=dev).manual_seed(1)
        mask_in = torch.rand(R_probe, N, device=dev, generator=g) < 0.7
        action = torch.randint(0, N, (R_probe,), device=dev, generator=g)
        step_i = torch.full((R_probe,), 5, dtype=torch.int64, device=dev)
        first_in = torch.randint(0, N, (R_probe,), device=dev, generator=g)
        mask_o = torch.empty_like(mask_in)
        first_o, cur_o = torch.empty_like(first_in), torch.empty_like(first_in)
        done_o = torch.empty(R_probe, dtype=torch.bool, device=dev)
        ms = time_launch(lambda: call("rrnco_atsp_step", R_probe, N, ptr(action), ptr(step_i), ptr(mask_in),
                                      ptr(first_in), ptr(mask_o), ptr(first_o), ptr(cur_o), ptr(done_o),
                                      stream_ptr(dev)))
        nbytes = R_probe * (2 * N + 50)  # SURVEY.md 8(d): ATSP 2N+50 B per rollout-step
        return {"kernel": "rrnco::atsp_step_kernel (ATSPEnv._step, reference layout)", "rollouts": R_probe,
                "ms_per_launch": ms, "algorithmic_bytes_per_launch": nbytes,
                "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s"}

    def rcvrptw_step_probe():
        # RMTVRPEnv._step + get_action_mask at the C3 size: 1024 instances x 100 starts; instance data stays
        # un-replicated (data_rows = 1024, 84 MB: the matrix rows / columns are served by L2), the rollout state is
        # in the reference layout.  Bytes are SURVEY.md 8(d)'s algorithmic count (39N+100 per rollout-step), so this
        # figure is NOT bounded by the HBM peak.
        import ctypes as C
        from rrnco_b200._lib import call, ptr, stream_ptr
        from rrnco_b200.envs import RMTVRPEnv
        Bt, St, N = B, 100, N_LOC + 1
        g = torch.Generator(device=dev).manual_seed(2)
        env_tw = RMTVRPEnv(generator_params={"num_loc": N_LOC}, check_solution=False, device=dev)
        dm = torch.rand(Bt, N, N, device=dev, generator=g)
        td0 = rb.TensorDictLite({
            "locs": torch.rand(Bt, N, 2, device=dev, generator=g), "distance_matrix": dm,
            "duration_matrix": dm * (0.5 + torch.rand(Bt, N, N, device=dev, generator=g)),
            "demand_linehaul": torch.rand(Bt, N_LOC, device=dev, generator=g) * 0.2,
            "time_windows": torch.stack([torch.rand(Bt, N, device=dev, generator=g), 4 + torch.rand(Bt, N, device=dev, generator=g)], -1),
            "service_time": torch.rand(Bt, N, device=dev, generator=g) * 0.05}, batch_size=[Bt])
        td0 = env_tw.reset(td0)
        td_r = rb.batchify(td0, St)
        R_probe = Bt * St
        keep = []
        data = RMTVRPEnv.instance_data(td0, keep)
        visited = torch.rand(R_probe, N, device=dev, generator=g) < 0.3
        td_r.update({"visited": visited, "current_node": torch.randint(1, N, (R_probe,), device=dev, generator=g),
                     "current_time": torch.rand(R_probe, 1, device=dev, generator=g),
                     "used_capacity_linehaul": torch.rand(R_probe, 1, device=dev, generator=g) * 0.5})
        s_in = RMTVRPEnv._state(td_r, keep)
        out = {k: torch.empty_like(td_r[k].reshape(-1) if k != "visited" else td_r[k]) for k in
               ("current_node", "current_time", "current_route_length", "used_capacity_linehaul",
                "used_capacity_backhaul", "visited")}
        s_out = type(s_in)()
        for k, v in out.items():
            setattr(s_out, k, ptr(v))
        action = torch.randint(1, N, (R_probe,), device=dev, generator=g)
        done_o = torch.empty(R_probe, dtype=torch.bool, device=dev)
        mask_o = torch.empty(R_probe, N, dtype=torch.bool, device=dev)
        ms = time_launch(lambda: call("rrnco_rmtvrp_step", R_probe, N, C.byref(data), ptr(action), C.byref(s_in),
                                      C.byref(s_out), ptr(done_o), ptr(mask_o), stream_ptr(dev)))
        nbytes = R_probe * (39 * N + 100)  # SURVEY.md 8(d): RCVRPTW 39N+100 B per rollout-step
        return {"kernel": "rrnco::rmtvrp_step_kernel (RMTVRPEnv._step + get_action_mask; instance data un-replicated, "
                          "L2-served: algorithmic bytes, not HBM-bounded)", "rollouts": R_probe,
                "ms_per_launch": ms, "algorithmic_bytes_per_launch": nbytes,
                "achieved": nbytes / (ms * 1e-3) / 1e9, "unit": "GB/s"}

    def gather_probe():
        from rrnco_b200.sampler import CityOnDevice, gather_submatrix
        city = CityOnDevice(make_city(3), dev)
        rng = np.random.RandomState(1)
        idx = torch.from_numpy(np.array([rng.choice(1000, N_LOC + 1, replace=False) for _ in range(4096)])).to(dev)
        ms = time_launch(lambda: gather_submatrix(city.distance_f32, idx, normalize=True), reps=20)
        ms64 = time_launch(lambda: gather_submatrix(city.distance, idx, normalize=True), reps=20)
        n2 = 4096 * (N_LOC + 1) ** 2
        # time and bytes of the SAME variant: fp32 source = 4 B gathered + 4 B written per element; the fp64 source (SURVEY
        # 8(d)'s 12 n^2) is reported beside it with its own time
        return {"kernel": "rrnco::gather_submatrix_kernel<float> (+ fused reset normalisation; source = the fp32 copy of the "
                          "fp64 city matrix that Real_World_Sampler keeps: 8 n^2 B per instance)",
                "instances": 4096, "ms_per_launch": ms, "algorithmic_bytes_per_launch": 8 * n2,
                "achieved": 8 * n2 / (ms * 1e-3) / 1e9, "unit": "GB/s",
                "fp64_source": {"ms_per_launch": ms64, "algorithmic_bytes_per_launch": 12 * n2,
                                "achieved": 12 * n2 / (ms64 * 1e-3) / 1e9, "unit": "GB/s"},
                "note": "the city matrix (4 / 8 MB) is L2-resident and n of 1000 columns per row are wanted: bound by L2 "
                        "sector requests, not HBM (ncu: profiles/r1_ncu_env_kernels_v4.txt)"}

    def nab_probe():
        """Encoder hot spot (SURVEY 8(f) rank 4): one DistAngleFusion module (gating neural adaptive bias, ATSP / RCVRP
        variant) over the augmented batch of the headline config -- the encoder evaluates 12 of them per encode."""
        torch.manual_seed(1234)
        mod = rb.DistAngleFusion(128).to(dev)
        Bn = B * N_AUG
        g = torch.Generator(device=dev).manual_seed(11)
        coords = torch.rand(Bn, N_LOC + 1, 2, device=dev, generator=g)
        cost = torch.rand(Bn, N_LOC + 1, N_LOC + 1, device=dev, generator=g)
        with torch.no_grad():
            ms = time_launch(lambda: mod(coords, cost), reps=10)
            ms_t = time_launch(lambda: mod(coords, cost.transpose(1, 2)), reps=10)
            ms_brute = time_launch(lambda: mod(coords, cost, variant=1), reps=5)
        pairs = Bn * (N_LOC + 1) ** 2
        entry = {"kernel": "rrnco::nab_gating_table_kernel (DistAngleFusion.forward, attn_freenet.py:242-289, collapsed to four "
                           "piecewise-linear scalar functions per module: two segment searches + 4 FMAs per pair; nothing "
                           "materialised)",
                 "instances": Bn, "pairs": pairs, "ms_per_launch": ms, "ms_per_launch_transposed_cost": ms_t,
                 "algorithmic_bytes_per_launch": 8 * pairs, "achieved": 8 * pairs / (ms * 1e-3) / 1e9, "unit": "GB/s",
                 "brute_force_variant": {"ms_per_launch": ms_brute, "fp32_lane_ops_per_pair": 1024,
                                         "fp32_frac": 1024 * pairs / (ms_brute * 1e-3) / (148 * 128 * 1.965e9),
                                         "what": "sum over the 128 hidden units (2 x 128 relu-FMAs + 4 x 128 FMAs per pair), "
                                                 "compute-bound on the fp32 pipes: the cross-check"},
                 "reference_flops_per_pair": 4 * 128 * 128 + 8 * 128,
                 "reference_activation_bytes_per_pair": 2 * 128 * 4 * 2,
                 "note": "`frac` = 4 B read + 4 B written per pair over the measured HBM peak"}
        # the whole O(N^2) part of a block fused (bias -> row softmax -> exp -> two [N,N] x [N,E] products -> sigmoid gate)
        q, k, v = (torch.randn(Bn, N_LOC + 1, 128, device=dev, generator=g) for _ in range(3))

        def unfused():  # the same math with the bias kernel + torch ops, as AFTFull.forward writes it (attn_freenet.py:319-324)
            a = torch.exp(torch.softmax(mod(coords, cost, scale=0.9), dim=-1))
            e1 = torch.exp(torch.softmax(k, dim=1))
            return torch.sigmoid(q) * (a @ (e1 * v)) / (a @ e1)
        with torch.no_grad():
            ms_f = time_launch(lambda: rb.aft_nab(q, k, v, coords, cost, mod, scale=0.9), reps=10)
            ms_u = time_launch(unfused, reps=5)
            err = (rb.aft_nab(q[:64], k[:64], v[:64], coords[:64], cost[:64], mod, scale=0.9) -
                   (lambda a, e1: torch.sigmoid(q[:64]) * (a @ (e1 * v[:64])) / (a @ e1))(
                       torch.exp(torch.softmax(mod(coords[:64], cost[:64], scale=0.9), dim=-1)), torch.exp(torch.softmax(k[:64], dim=1)))
                   ).abs().max().item()
        aft_bytes = Bn * (4 * (N_LOC + 1) * 128 * 4 + (N_LOC + 1) ** 2 * 4)
        entry["fused_aft_block"] = {
            "kernel": "rrnco::aft_nab_kernel (neural adaptive bias + AFTFull.forward :309-327 without its Linear layers; "
                      "adapt_bias, its softmax / exp and E1 / E2 never reach HBM)",
            "ms_per_launch": ms_f, "ms_unfused_bias_kernel_plus_torch": ms_u, "max_abs_diff_vs_unfused": err,
            "algorithmic_bytes_per_launch": aft_bytes, "achieved": aft_bytes / (ms_f * 1e-3) / 1e9, "unit": "GB/s",
            "frac": aft_bytes / (ms_f * 1e-3) / 1e9 / peaks()[0],
            "fp32_fma_per_launch": Bn * 2 * (N_LOC + 1) ** 2 * 128,
            "what": "q, k, v read + y written ([B,N,128] fp32 each) + the cost matrix once = algorithmic bytes"}
        # rcvrptw variant (duration channel, three-way gate) on tcgen05, at config C3's batch (1024 instances)
        torch.manual_seed(1235)
        modd = rb.DistAngleFusion(128, use_duration_matrix=True).to(dev)
        modd.check_overflow = False
        Bd = B
        durm = torch.rand(Bd, N_LOC + 1, N_LOC + 1, device=dev, generator=g)

        def torch_materialised(nb):  # upstream's op sequence on the GPU (materialises three [B,N,N,E] embeddings), small batch
            import torch.nn.functional as F
            c, u = cost[:nb].unsqueeze(-1), durm[:nb].unsqueeze(-1)
            diff = coords[:nb].unsqueeze(2) - coords[:nb].unsqueeze(1)
            a = torch.atan2(diff[..., 1], diff[..., 0]).unsqueeze(-1)
            d, an, du = modd.dist_emb(c), modd.angle_emb(a), modd.dur_emb(u)
            gt = F.softmax(modd.gate(torch.cat([d, an, du], -1)) / modd.gate_temperature.exp(), -1)
            return modd.out_lin(gt[..., [0]] * d + gt[..., [1]] * an + gt[..., [2]] * du).squeeze(-1)
        with torch.no_grad():
            ms_d = time_launch(lambda: modd(coords[:Bd], cost[:Bd], durm), reps=10)
            nb = 64
            ms_t = time_launch(lambda: torch_materialised(nb), reps=3, warm=1)
            errd = (modd(coords[:nb], cost[:nb], durm[:nb]) - torch_materialised(nb)).abs().max().item()
        pairs_d = Bd * (N_LOC + 1) ** 2
        flops_issued = pairs_d * 3 * 2 * 384 * 128  # three split terms
        entry["duration_gate"] = {
            "kernel": "rrnco::nab_dur_kernel (DistAngleFusion.forward with the duration channel, attn_freenet.py:242-289: "
                      "[pairs x 3E] x [3E x E] on tcgen05, three-term fp16 split, A operand generated on the fly)",
            "instances": Bd, "pairs": pairs_d, "ms_per_launch": ms_d,
            "issued_tflops": flops_issued / (ms_d * 1e-3) / 1e12, "tensor_peak_tflops": peaks()[1],
            "tensor_frac_issued": flops_issued / (ms_d * 1e-3) / 1e12 / peaks()[1],
            "algorithmic_bytes_per_launch": 12 * pairs_d, "achieved": 12 * pairs_d / (ms_d * 1e-3) / 1e9, "unit": "GB/s",
            "ms_torch_materialised_same_batch_extrapolated": ms_t * Bd / nb, "torch_sample_instances": nb,
            "max_abs_diff_vs_torch_fp32": errd}
        if not args.no_cpu_baseline:
            from oracle import encoder as oenc
            torch.set_num_threads(os.cpu_count() or 1)
            k = 8
            pc = {kk: v.detach().cpu() for kk, v in mod.state_dict().items()}
            cc, cm = coords[:k].cpu(), cost[:k].cpu()
            with torch.inference_mode():
                oenc.dist_angle_fusion(pc, cc[:1], cm[:1])
                t0 = time.perf_counter()
                oenc.dist_angle_fusion(pc, cc, cm)
                dt = time.perf_counter() - t0
            entry["cpu_baseline"] = {"value": k / dt, "unit": "instances/s per module", "cores": os.cpu_count() or 1, "kind": "port",
                                     "sample": f"{k} instances, {dt:.2f} s"}
            entry["value"] = Bn / (ms * 1e-3)
            entry["value_unit"] = "instances/s per module"
        return entry

    env_probe = env_step_probe() if rank == 0 else None
    nab_entry = nab_probe() if rank == 0 else None
    gat_probe = gather_probe() if rank == 0 else None
    atsp_probe = atsp_step_probe() if rank == 0 else None
    tw_probe = rcvrptw_step_probe() if rank == 0 else None

    # ---- e2e: host inputs, H2D + reset + cache + rollout + reduction + D2H ----------------------------
    ms_e2e, best = timed(step_e2e, args.steps, 2)
    raw, row, col = host_sets[0]
    h2d = sum(v.numel() * v.element_size() for v in raw.values()) + 2 * row.numel() * row.element_size()
    d2h = B * 4

    # ---- the other BASELINE configs, one short measured line each ------------------------------------
    cfg_block = None
    if not args.no_configs:
        del dev_sets, host_sets, out, best
        torch.cuda.empty_cache()
        cfg_block = measure_configs(args, rb, dev, rank, world, dist_on, timed)

    # ---- training hand-off (SURVEY 8(f) rank 2): one REINFORCE step at the C5 per-GPU shape, rank 0 only ----------------
    train_entry = None
    if rank == 0 and not args.no_configs:
        torch.cuda.empty_cache()
        train_entry = training_probe(rb, dev)

    if rank == 0:
        hbm_peak, tf_peak, peak_src = peaks()
        stamp = profile_stamp()
        # rollout-steps the kernel actually ran: every (instance, tile) CTA stops when ITS rollouts are done
        rollout_steps = int((tile_steps.long() - 1).clamp_min(0).sum().item()) * N_START
        tile_steps_total = int((tile_steps.long() - 1).clamp_min(0).sum().item())
        alg_bytes = rollout_steps * BYTES_PER_ROLLOUT_STEP
        alg_flops = rollout_steps * FLOPS_PER_ROLLOUT_STEP
        issued_flops = tile_steps_total * issued_mma_flops_per_tile_step(N_LOC + 1, args.precision)
        sec = ms_kernel * 1e-3
        line = {
            "metric": "RCVRP n100 POMO rollout instances/s", "value": value, "unit": "instances/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (fp32-faithful: three-term fp16-split tcgen05 contractions, fp32 accumulate)" if args.precision == 3 else "f16 (single pass, fp32 accumulate)",
            "data": "synthetic (city-like asymmetric 1000-node matrices, integer demands 1-9 / 50; random-init "
                    "decoder seed 1234; encoder output = unit-variance stand-in embeddings)",
            "config": {"workload": "RCVRP n=100 POMO multi-start x8 aug greedy rollout, batch 1024 per GPU "
                                   "(BASELINE config[1])",
                       "instances_per_gpu": B, "n_aug": N_AUG, "num_starts": N_START, "decode_steps_max": T,
                       "decode_steps_mean_per_tile": tile_steps_total / max(1, tile_steps.numel()),
                       "rollouts_per_gpu": Bp * N_START,
                       "augmentation": "dihedral8 on locs; distance matrices / demands shared by the 8 copies (not replicated)",
                       "l2_policy": "two alternating input sets, 1.7 GB of key cache per set (>> 126 MB L2)"},
            "clocks": clocks,
            "gpu_launches": int(launches),
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "instances/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e,
                    "what": "RRNetPolicy.forward on pinned HOST inputs (instance td + encoder output): H2D "
                            "(every step, on the copy stream, double-buffered: the copy of batch i+1 overlaps the rollout "
                            "of batch i), x8 augmentation, env.reset normalisation, cache GEMM, fused rollout, best-of "
                            "reduction, D2H of the [B] best costs.  The ENCODER is outside both arms (it stays the "
                            "reference's PyTorch module; its output is the host input here), and policy() returns "
                            "actions [R,T] / reward [R] on the device as upstream does."},
            "roofline": {"bound": "tensor", "achieved": alg_flops / sec / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": alg_flops / sec / 1e12 / tf_peak,
                         "traffic": stamp.get("rollout_c2_dram_bytes") if B == 1024 else None,
                         "traffic_source": stamp.get("rollout_c2_source") if B == 1024 else None,
                         "peak_source": peak_src + ", sustained cuBLAS bf16",
                         "kernel": "rrnco::rollout_lean_kernel<RCVRP, 3>", "ms_per_launch": ms_kernel,
                         "algorithmic_flops_per_launch": alg_flops, "rollout_steps_per_launch": rollout_steps,
                         "what": "algorithmic = 373 kFLOP per rollout-step (SURVEY 8(d)) x rollout-steps summed over the tiles "
                                 "(each CTA stops at its own tour length)",
                         "issued": {"tflops": issued_flops / sec / 1e12, "frac": issued_flops / sec / 1e12 / tf_peak,
                                    "what": "tcgen05 FLOPs actually issued: 3 fp16 operand terms per product (fp32-faithful), "
                                            "128-row tiles for 101 starts, keys padded 101 -> 112",
                                    "tensor_pipe_active_pct_ncu": stamp.get("rollout_tensor_pipe_active_pct")},
                         "hbm_algorithmic": {"achieved": alg_bytes / sec / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                             "frac": alg_bytes / sec / 1e9 / hbm_peak,
                                             "algorithmic_bytes_per_launch": alg_bytes,
                                             "what": "north-star figure: 3.2 KB per rollout-step (SURVEY 8(d)) over the "
                                                     "measured HBM peak; the fused kernel's real DRAM traffic is `traffic`"}},
        }
        for probe, key in ((env_probe, "rcvrp_step_dram_bytes"), (gat_probe, "gather_dram_bytes"),
                           (atsp_probe, "atsp_step_dram_bytes"), (tw_probe, "rcvrptw_step_dram_bytes"),
                           (nab_entry, "nab_dram_bytes")):
            probe["peak"] = hbm_peak
            probe["frac"] = probe["achieved"] / hbm_peak
            probe["dram_bytes_measured"] = stamp.get(key)  # ncu dram__bytes_read + write of this build (None: not captured)
            if stamp.get(key):
                probe["dram_frac"] = stamp[key] / (probe["ms_per_launch"] * 1e-3) / 1e9 / hbm_peak
        line["env_step"] = env_probe
        line["env_step_atsp"] = atsp_probe
        line["env_step_rcvrptw"] = tw_probe
        line["gather"] = gat_probe
        line["encoder_nab"] = nab_entry
        if cfg_block is not None:
            line["configs"] = cfg_block
        if train_entry is not None:
            line["training_step"] = train_entry
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            rate, dt, cost, Tc = cpu_rollout_rate(args.cpu_sample, threads)
            line["cpu_baseline"] = {"value": rate, "unit": "instances/s", "cores": threads, "kind": "port",
                                    "sample": f"{args.cpu_sample} instances x {N_AUG} aug x {N_START} starts, "
                                              f"{Tc} decode steps, {dt:.1f} s on {threads} threads"}
        print(json.dumps(line), flush=True)
    if dist_on:
        dist.destroy_process_group()


def training_probe(rb, dev, n_inst=512, steps=3):
    """One training step as upstream's `shared_step` runs it (rl.py:99-130) at the per-GPU shape of config C5: sampling
    rollout on the fused kernel (no graph) -> differentiable replay of the sampled actions -> POMO shared-baseline loss ->
    backward to the decoder parameters and the encoder output.  Timed on the device (CUDA events, median of `steps` after one
    warm-up) for the hand-written replay kernels (librrnco_b200_train.so) and, once, for the plain-torch (ATen) replay."""
    from rrnco_b200 import training as tr, train_ops
    S = N_LOC + 1
    env = rb.RCVRPEnv(generator_params={"num_loc": N_LOC}, check_solution=False, device=dev)
    raw = host_instances(n_inst, seed=31337)
    td = env.reset(rb.TensorDictLite({k: v.to(dev) for k, v in raw.items()}, batch_size=[n_inst]))
    row, col = stand_in_embeddings(n_inst, seed=31338)
    row, col = row.to(dev).requires_grad_(True), col.to(dev).requires_grad_(True)
    torch.manual_seed(1234)
    decoder = rb.RRNetDecoder(env_name="rcvrp").to(dev)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col

    pol = rb.RRNetPolicy(encoder=Enc(), decoder=decoder, env_name="rcvrp").to(dev)

    def one(impl):
        tr.REPLAY_IMPL = impl
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        with torch.no_grad():
            out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S)
        ll = rb.replay_log_likelihood(pol, td, env, out["actions"], S, embeddings=(row, col))
        rb.pomo_shared_baseline_loss(out["reward"], ll, S).backward()
        e1.record()
        torch.cuda.synchronize()
        err = (ll.detach() - out["log_likelihood"]).abs().max().item()
        gn = float(sum(p.grad.double().pow(2).sum() for p in decoder.parameters() if p.grad is not None).sqrt())
        pol.zero_grad(set_to_none=True)
        row.grad = col.grad = None
        return e0.elapsed_time(e1), int(out["actions"].shape[1]), err, gn

    try:
        one("fused")
        runs = sorted(one("fused") for _ in range(steps))
        train_ops.check_status(dev)
        ms, T, err, gn = runs[len(runs) // 2]
        one("aten")
        ms_aten, T_aten, err_aten, _ = one("aten")
    finally:
        tr.REPLAY_IMPL = "fused"
    return {"workload": f"one REINFORCE step, RCVRP n={N_LOC}: {n_inst} instances x {S} starts sampled by the fused rollout kernel, "
                        "differentiable replay of the sampled actions, POMO shared-baseline loss, backward (rl.py:99-130; per-GPU "
                        "share of config C5)",
            "ms_per_step": ms, "instances_per_s": n_inst / (ms * 1e-3), "decode_steps": T,
            "replay": "hand-written kernels, forward and backward (librrnco_b200_train.so: tcgen05 FFN / pointer GEMMs in the "
                      "three-term fp16 split, CUDA-core + mma.sync 3xTF32 attention), fp32-faithful",
            "max_abs_loglik_diff_vs_sampling_kernel": err, "decoder_grad_norm": gn,
            "aten_replay": {"ms_per_step": ms_aten, "decode_steps": T_aten, "max_abs_loglik_diff_vs_sampling_kernel": err_aten,
                            "what": "the same step with the plain-torch replay (fp32 SDPA / cuBLAS SIMT GEMMs / element-wise ATen)"},
            "timing": f"CUDA events around the whole step, median of {steps} after one warm-up; ATen arm: second of two steps"}


# --------------------------------------------------------------------------------------------------
# the other BASELINE configs (C1, C3, C4, C5): value / e2e / cpu sample / roofline fractions each
# --------------------------------------------------------------------------------------------------
CONFIG_SPECS = {
    "C1": dict(env="atsp", n=100, batch=32, aug=8, starts=100, decode="greedy", scaling="weak", steps=5,
               what="ATSP n=100 greedy rollout x8 aug, batch 32 (BASELINE config[0]; the reference runs it on the CPU)"),
    "C3": dict(env="rcvrptw", n=100, batch=1024, aug=1, starts=100, decode="sampling", scaling="weak", steps=5,
               what="RCVRPTW n=100 with duration matrix and time windows, sampling decode, batch 1024 (BASELINE config[2])"),
    "C4": dict(env="atsp", n=1000, batch=64, aug=1, starts=100, decode="greedy", scaling="weak", steps=2,
               what="ATSP n=1000 generalisation rollout, batch 64, 100 starts as test.py:129-130 (BASELINE config[3])"),
    "C5": dict(env="rcvrp", n=100, batch=None, aug=1, starts=101, decode="sampling", scaling="strong", steps=5,
               what="RCVRP n=100 REINFORCE training rollouts, GLOBAL batch 4096 x 101 starts sharded over the ranks, instances "
                    "sub-sampled on the device from synthetic 1000-node city matrices (BASELINE config[4])"),
}


def cpu_config_rate(spec, n_inst, threads, seed=777):
    """CPU arm of one config: the oracle port on a bounded sample (host cores of this box)."""
    from oracle import envs as oenvs, model as omodel, synth
    from oracle.td import batchify
    torch.set_num_threads(threads)
    name, n = spec["env"], spec["n"]
    N = n if name == "atsp" else n + 1
    t0 = time.perf_counter()
    raw = synth.make_instances(name, n_inst, n, seed=seed, city=synth.make_city(0, length=max(1000, N)))  # incl. the NumPy gather
    t_gen = time.perf_counter() - t0
    env = oenvs.make_env(name, n, check_solution=False)
    p = omodel.init_decoder_params(name, seed=1234)
    row, col = synth.random_embeddings(n_inst * spec["aug"], N, seed=seed)
    with torch.inference_mode():
        t0 = time.perf_counter()
        td = env.reset(raw)
        if spec["aug"] > 1:
            td = batchify(td, spec["aug"])
        out = omodel.policy_forward(p, env, td, row, col, decode_type="multistart_" + spec["decode"], num_starts=spec["starts"],
                                    generator=torch.Generator().manual_seed(seed))
        dt = time.perf_counter() - t0
    if spec["scaling"] == "strong":
        dt += t_gen  # C5 generates its instances inside the step
    return n_inst / dt, dt, int(out["actions"].shape[1])


def measure_configs(args, rb, dev, rank, world, dist_on, timed, only=None, steps=None, warmup=3, dump_dir=None):
    from rrnco_b200.sharding import gather_costs
    hbm_peak, tf_peak, _ = peaks()
    block = {}
    # 8 synthetic cities: every per-rank batch (32 ... 4096) splits evenly over them (upstream's `target // n_cities`
    # integer division would otherwise hand back slightly fewer instances than asked, generator_lazy.py:203)
    cities = [rb.CityOnDevice(make_city(c), dev) for c in range(8)]
    cpu_samples = {"C1": 4, "C3": 16, "C4": 1, "C5": 16}
    for cname, spec in CONFIG_SPECS.items():
        if only is not None and cname not in only:
            continue
        if steps is not None:
            spec = dict(spec, steps=steps)
        name, n, A, S = spec["env"], spec["n"], spec["aug"], spec["starts"]
        N = n if name == "atsp" else n + 1
        Bc = spec["batch"] if spec["batch"] is not None else max(1, args.c5_global_batch // world)
        env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False, device=dev)
        torch.manual_seed(1234)
        decoder = rb.RRNetDecoder(env_name=name).to(dev)
        gen_cls = {"atsp": rb.LazyATSPGenerator, "rcvrp": rb.LazyRCVRPGenerator, "rcvrptw": rb.LazyRMTVRPGenerator}[name]
        big = [rb.CityOnDevice(make_city(20 + c, length=1200), dev) for c in range(2)] if n >= 1000 else cities
        gen = gen_cls(num_loc=n, cities=big, device=dev, seed=1000 * (rank + 1) + 7, chunk_size=max(1000, Bc))
        augment = rb.StateAugmentation(num_augment=A, augment_fn="dihedral8", no_aug_coords=False, share_instance_data=True) if A > 1 else None
        kind = spec["decode"]
        g = torch.Generator(device=dev).manual_seed(5 + rank)
        embeds = [(torch.randn(Bc * A, N, 128, device=dev, generator=g), torch.randn(Bc * A, N, 128, device=dev, generator=g))
                  for _ in range(2)]

        def make_td():
            td = gen(Bc)
            assert td.batch_size[0] == Bc, (td.batch_size, Bc)
            return env.reset(augment(td) if augment is not None else td)

        rollout = rb.fused_rollout if N <= 1024 else rb.stepwise_rollout
        state = {}

        if spec["scaling"] == "strong":
            # C5: generate batch i+1 (index sampling + gather + laws + reset) on a side stream under the rollout of batch i
            side = torch.cuda.Stream(device=dev)
            pending = {}

            def prefetch(i):
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    td = make_td()
                    cache = decoder._precompute_cache(embeds[i % 2])
                    ev = torch.cuda.Event()
                    ev.record(side)
                pending[i] = (td, cache, ev)

            def step(i):
                if i not in pending:
                    prefetch(i)
                prefetch(i + 1)
                td, cache, ev = pending.pop(i)
                torch.cuda.current_stream(dev).wait_event(ev)
                out = rollout(decoder, cache, env, td, S, True, kind, seed=1234 + i, check=False)
                best = out["reward"].view(S, Bc).amax(0)
                if dist_on:
                    gather_costs(best, world * Bc)
                state["out"] = out
                return best.cpu()  # D2H of the costs: the step's host-visible result
            ms_val, _ = timed(step, spec["steps"], warmup)
            ms_e2e, h2d, d2h = ms_val, 0, Bc * 4
            e2e_what = ("same pipeline (this config has no host inputs: instances are generated on the device from the "
                        "HBM-resident city matrices, the encoder output is a resident stand-in); D2H of the [B] best costs")
            n_units = Bc * world if dist_on else Bc
        else:
            sets = [(make_td(), decoder._precompute_cache(embeds[i])) for i in range(2)]
            torch.cuda.synchronize()

            def step(i):
                td, cache = sets[i % 2]
                out = rollout(decoder, cache, env, td, S, True, kind, seed=1234 + i, check=False)
                best = rb.unbatchify(out["reward"], (A, S)).amax(-1).amax(-1) if A > 1 else out["reward"].view(S, Bc).amax(0)
                if dist_on:
                    gather_costs(best, world * Bc)
                state["out"] = out
                return out
            ms_val, _ = timed(step, spec["steps"], warmup)
            # e2e through the public API: pinned host instance td + encoder output -> H2D -> (aug) -> reset -> policy -> D2H
            host_td = {k: v.cpu().pin_memory() for k, v in gen(Bc).items()}
            host_emb = (embeds[0][0].cpu().pin_memory(), embeds[0][1].cpu().pin_memory())

            class Enc(torch.nn.Module):
                row = col = None

                def forward(self, td, phase=None):
                    return self.row, self.col
            enc_cfg = Enc()
            policy = rb.RRNetPolicy(encoder=enc_cfg, decoder=decoder, env_name=name).to(dev)
            # like the headline's e2e: every step copies ITS batch from pinned host memory; the copy of step i + 1 is issued
            # on the copy stream before step i's kernels (rrnco_b200.HostPrefetcher, double-buffered)
            pf = rb.HostPrefetcher(dev)
            tk = {}
            host_batch = {**host_td, "__row_emb": host_emb[0], "__col_emb": host_emb[1]}

            def step_e2e_cfg(i):
                if i not in tk:
                    tk[i] = pf.submit(host_batch)
                tk[i + 1] = pf.submit(host_batch)
                ticket = tk.pop(i)
                d = pf.acquire(ticket)
                enc_cfg.row, enc_cfg.col = d["__row_emb"], d["__col_emb"]
                td = rb.TensorDictLite({k: v for k, v in d.items() if not k.startswith("__")}, batch_size=[Bc])
                td = env.reset(augment(td) if augment is not None else td)
                with torch.no_grad():
                    out = policy(td, env, phase="train" if kind == "sampling" else "val", decode_type="multistart_" + kind,
                                 num_starts=S, seed=99 + i)
                best = rb.unbatchify(out["reward"], (A, S)).amax(-1).amax(-1) if A > 1 else out["reward"].view(S, Bc).amax(0)
                pf.release(ticket)
                return best.cpu()
            ms_e2e, _ = timed(step_e2e_cfg, spec["steps"], 2)
            h2d = sum(v.numel() * v.element_size() for v in host_td.values()) + 2 * host_emb[0].numel() * 4
            d2h = Bc * 4
            e2e_what = ("RRNetPolicy.forward on pinned HOST inputs (instance td + encoder output): H2D every step on the copy stream "
                        "(double-buffered HostPrefetcher: the copy of batch i+1 overlaps the rollout of batch i), reset, cache "
                        "GEMM, rollout, D2H of the [B] costs")
            n_units = Bc * world
        out = state["out"]
        if dump_dir and rank == 0:  # the rollout of the last timed step
            dump_outputs(dump_dir, out)
        if "tile_steps" in out:
            ts = (out["tile_steps"].long() - 1).clamp_min(0)
            tr = rb._lib.lib().rrnco_rollout_tile_rows(rb._lib.ENV_ID[name], N, Bc * A, S)  # POMO starts per CTA tile
            n_tiles = (S + tr - 1) // tr
            rows = torch.tensor([min(tr, S - t * tr) for t in range(n_tiles)], device=ts.device).repeat(ts.numel() // n_tiles)
            rollout_steps = int((ts * rows).sum().item())
        else:
            rollout_steps = Bc * A * S * (out["actions"].shape[1] - 1)
        b_alg, f_alg = algorithmic_per_rollout_step(name, N, S)
        sec = ms_val * 1e-3
        entry = {"workload": spec["what"], "value": n_units / sec, "unit": "instances/s", "scaling": spec["scaling"],
                 "ms_per_step": ms_val, "steps": spec["steps"], "instances_per_gpu": Bc, "n_aug": A, "num_starts": S,
                 "decode": kind, "decode_steps_max": int(out["actions"].shape[1]),
                 "path": "fused persistent kernel (rrnco_rollout, lean engine)" if N <= 112 else
                         "fused persistent key-tiled kernel (rrnco_rollout, rollout_tiled.cu: 128-key tiles, CTA pairs)" if N <= 1024
                         else "per-step pipeline (rrnco_decoder_logits_large + rrnco_select_action + env step)",
                 "e2e": {"value": n_units / (ms_e2e * 1e-3), "unit": "instances/s", "h2d_bytes_per_step": int(h2d),
                         "d2h_bytes_per_step": int(d2h), "what": e2e_what},
                 "roofline": {"hbm_algorithmic": {"achieved": rollout_steps * b_alg / sec / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                  "frac": rollout_steps * b_alg / sec / 1e9 / hbm_peak,
                                                  "bytes_per_rollout_step": b_alg},
                              "tensor_algorithmic": {"achieved": rollout_steps * f_alg / sec / 1e12, "peak": tf_peak,
                                                     "unit": "TFLOP/s", "frac": rollout_steps * f_alg / sec / 1e12 / tf_peak,
                                                     "flops_per_rollout_step": f_alg},
                              "rollout_steps_per_step": rollout_steps}}
        if rank == 0 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            k = cpu_samples[cname]
            rate, dt, Tc = cpu_config_rate(spec, k, threads)
            entry["cpu_baseline"] = {"value": rate, "unit": "instances/s", "cores": threads, "kind": "port",
                                     "sample": f"{k} instance(s) x {A} aug x {S} starts, {Tc} decode steps, {dt:.1f} s on {threads} threads"}
        block[cname] = entry
        del gen, decoder, embeds, out
        state.clear()
        if spec["scaling"] != "strong":
            del sets
        torch.cuda.empty_cache()
    return block


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
