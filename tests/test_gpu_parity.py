"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Every call goes through the C-ABI library.

Bars (BASELINE.json north star):
  * forced action sequences: masks / visited / tours bit-exact, load / time / reward <= 1e-6 relative;
  * greedy rollouts from identical weights: per-instance costs within 1e-4 relative on >= 99.9 % of instances
    (the fp32-vs-fp64 oracle disagreement is measured beside it as the noise floor);
  * fp32 logits within 2e-5 absolute of the reference's (3xTF32 contractions).
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import envs as oenvs, model as omodel, sampler as osampler, synth
from oracle.td import TD, batchify as obatchify

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
dev = "cuda"


@pytest.fixture(scope="module")
def rb():
    import rrnco_b200
    rrnco_b200.set_precision(3)
    return rrnco_b200


def load(name):
    z = np.load(os.path.join(GOLDEN, name))
    return {k: torch.from_numpy(z[k]) if z[k].shape != () else z[k].item() for k in z.files}


def lite(rb, td, device=dev):
    return rb.TensorDictLite({k: v.to(device) for k, v in td.items()}, batch_size=list(td.batch_size))


def make_policy(rb, name, p, row, col):
    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col
    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(p, strict=True)
    return pol


def rel(a, b):
    return ((a - b).abs() / b.abs().clamp_min(1e-12)).max().item()


# ----------------------------------------------------------------------------------------------------
# env step / mask / reward on forced action sequences
# ----------------------------------------------------------------------------------------------------
ENV_FILES = sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, "env_*.npz")))


@pytest.mark.parametrize("fname", ENV_FILES)
def test_env_forced_sequence_vs_reference_golden(rb, fname):
    z = load(fname)
    name = fname[4:-4].split("_")[0]
    raw = TD({k[3:]: v for k, v in z.items() if k.startswith("in.")}, batch_size=[z["actions"].shape[0]])
    n = raw["distance_matrix"].shape[-1] - (0 if name == "atsp" else 1)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=(name != "rcvrptw"))
    td = env.reset(lite(rb, raw, "cpu"))  # host td: reset does the H2D
    assert td["action_mask"].is_cuda
    assert torch.equal(td["action_mask"].cpu(), z["reset.action_mask"])
    assert torch.equal(td["distance_matrix"].cpu(), z["reset.distance_matrix"])
    assert torch.equal(td["min_distance"].cpu(), z["reset.min_distance"])
    assert torch.equal(td["max_distance"].cpu(), z["reset.max_distance"])
    acts = z["actions"].to(dev)
    for t in range(acts.shape[1]):
        td.set("action", acts[:, t])
        td = env.step(td)["next"]
        for k in [k for k in z if k.startswith("step.")]:
            got, want = td[k[5:]].cpu(), z[k][t]
            assert got.shape == want.shape and got.dtype == want.dtype, (k, t)
            assert torch.equal(got, want), (k, t)  # fp32 state too: same _rn operations in the same order
    real, norm = env.get_reward(td, acts)
    assert rel(real.cpu(), z["reward.real"]) < 1e-6 and rel(norm.cpu(), z["reward.norm"]) < 1e-6
    if name == "rcvrptw":
        assert torch.equal(td["distance_matrix"].cpu(), z["after_reward.distance_matrix"])


@pytest.mark.parametrize("name,n,B", [("atsp", 100, 64), ("rcvrp", 100, 64), ("rcvrptw", 100, 64), ("rcvrp", 37, 33),
                                        ("rcvrp", 28, 40), ("rcvrp", 40, 36), ("rcvrp", 4, 32), ("atsp", 37, 33),
                                        ("atsp", 3, 32), ("rcvrptw", 30, 20)])
def test_env_random_transitions_vs_oracle(rb, name, n, B):
    """>= 1e5 random forced transitions at n=100 in total: masks / visited bit-exact, scalars <= 1e-6 rel."""
    g = torch.Generator().manual_seed(n + B)
    raw = synth.make_instances(name, B, n, seed=n, integer_demand=False)
    oenv = oenvs.make_env(name, n, check_solution=False)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    S = 8
    otd = obatchify(oenv.reset(raw), S)
    td = rb.batchify(env.reset(lite(rb, raw)), S)
    actions, t = [], 0
    while not otd["done"].all():
        a = torch.multinomial(otd["action_mask"].float(), 1, generator=g).squeeze(1)
        otd["action"] = a
        otd = oenv.step(otd)["next"]
        td.set("action", a.to(dev))
        td = env.step(td)["next"]
        actions.append(a)
        assert torch.equal(td["action_mask"].cpu(), otd["action_mask"]), t
        assert torch.equal(td["done"].cpu(), otd["done"]), t
        if name != "atsp":
            assert torch.equal(td["visited"].cpu(), otd["visited"]), t
        for k in ("used_capacity", "current_time", "current_route_length", "used_capacity_linehaul"):
            if k in otd:
                assert torch.equal(td[k].cpu(), otd[k]), (k, t)
        t += 1
    acts = torch.stack(actions, 1)
    real, norm = env.get_reward(td, acts.to(dev))
    oreal, onorm = oenv.get_reward(otd, acts)
    assert rel(real.cpu(), oreal) < 1e-6 and rel(norm.cpu(), onorm) < 1e-6
    # static get_action_mask on the final state
    assert torch.equal(type(env).get_action_mask(td).cpu(), otd["action_mask"]) if name != "atsp" else True


def test_rcvrp_env_step_persistent_pipeline_many_blocks(rb):
    """40 400 rollouts = 1262 blocks of 32 (+ a tail of 16): every warp of the persistent staged env-step kernel runs its
    double-buffered loop more than once; a few random forced transitions, everything bit-exact vs the oracle."""
    name, n, B, S = "rcvrp", 100, 404, 100
    g = torch.Generator().manual_seed(7)
    raw = synth.make_instances(name, B, n, seed=11, integer_demand=False)
    oenv = oenvs.make_env(name, n, check_solution=False)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    otd = obatchify(oenv.reset(raw), S)
    td = rb.batchify(env.reset(lite(rb, raw)), S)
    assert td["visited"].shape[0] == 40400
    for t in range(4):
        a = torch.multinomial(otd["action_mask"].float(), 1, generator=g).squeeze(1)
        otd["action"] = a
        otd = oenv.step(otd)["next"]
        td.set("action", a.to(dev))
        td = env.step(td)["next"]
        for k in ("action_mask", "done", "visited", "used_capacity", "current_node"):
            assert torch.equal(td[k].cpu(), otd[k]), (k, t)


def test_env_step_pipelines_wrap_their_stage_rings(rb):
    """Staged env-step kernels at sizes where every warp runs its cp.async ring several times around (ATSP: 4 stages x 16
    warps x 148 CTAs; RCVRP: 2 stages x 6 warps): checked against the step rule written in plain torch ops
    (atsp/env.py:79-105, rcvrp/env.py:90-122,183-195), bit-exact."""
    from rrnco_b200._lib import call, ptr, stream_ptr
    g = torch.Generator(device=dev).manual_seed(3)
    # ATSP: 12 001 blocks of 32 rollouts (> 4 x 2368) + a tail of 7
    R, N = 32 * 12001 + 7, 100
    mask_in = torch.rand(R, N, device=dev, generator=g) < 0.6
    action = torch.randint(0, N, (R,), device=dev, generator=g)
    first_in = torch.randint(0, N, (R,), device=dev, generator=g)
    for step_val in (0, 5):
        step_i = torch.full((1,), step_val, dtype=torch.int64, device=dev)
        mask_o = torch.empty_like(mask_in)
        first_o, cur_o = torch.empty_like(first_in), torch.empty_like(first_in)
        done_o = torch.empty(R, dtype=torch.bool, device=dev)
        call("rrnco_atsp_step", R, N, ptr(action), ptr(step_i), ptr(mask_in), ptr(first_in), ptr(mask_o), ptr(first_o),
             ptr(cur_o), ptr(done_o), stream_ptr(dev))
        want = mask_in.clone()
        want[torch.arange(R, device=dev), action] = False
        assert torch.equal(mask_o, want) and torch.equal(cur_o, action)
        assert torch.equal(done_o, ~want.any(1)) and torch.equal(first_o, action if step_val == 0 else first_in)
    # RCVRP: 4001 blocks (> 3 x 888) + a tail of 5, N - 1 a multiple of 20 (chunks only) and not (chunk + tail)
    for N in (101, 29):
        R = 32 * 4001 + 5
        demand = torch.rand(R, N - 1, device=dev, generator=g) * 0.3
        cap = torch.ones(R, device=dev)
        used = torch.rand(R, device=dev, generator=g) * 0.8
        visited = (torch.rand(R, N, device=dev, generator=g) < 0.4).to(torch.uint8)
        action = torch.randint(0, N, (R,), device=dev, generator=g)
        used_o, vis_o = torch.empty_like(used), torch.empty_like(visited)
        cur_o = torch.empty(R, dtype=torch.int64, device=dev)
        done_o = torch.empty(R, dtype=torch.bool, device=dev)
        mask_o = torch.empty(R, N, dtype=torch.bool, device=dev)
        call("rrnco_rcvrp_step", R, N, R, ptr(action), ptr(demand), ptr(cap), R, ptr(used), ptr(visited), None, ptr(used_o),
             ptr(vis_o), ptr(cur_o), ptr(done_o), ptr(mask_o), stream_ptr(dev))
        sel = torch.gather(demand, 1, (action - 1).clamp(0, N - 2)[:, None]).squeeze(1)
        w_used = (used + sel) * (action != 0).float()
        w_vis = visited.clone()
        w_vis[torch.arange(R, device=dev), action] = 1
        free = ~(w_vis[:, 1:].bool() | (demand + w_used[:, None] > cap[:, None]))
        w_mask = torch.cat([~((action == 0) & free.any(1))[:, None], free], 1)
        assert torch.equal(used_o, w_used) and torch.equal(vis_o, w_vis) and torch.equal(cur_o, action)
        assert torch.equal(mask_o, w_mask) and torch.equal(done_o, w_vis.sum(1) == N)


def test_host_prefetcher_round_trip(rb):
    """Double-buffered pinned-host -> HBM staging: three batches through two slots, contents intact, slot reuse ordered."""
    pf = rb.HostPrefetcher(dev)
    batches = [{"a": torch.randn(1 << 20).pin_memory(), "b": torch.randint(0, 255, (4097, 3), dtype=torch.uint8).pin_memory()}
               for _ in range(3)]
    t0 = pf.submit(batches[0])
    t1 = pf.submit(batches[1])
    d0 = pf.acquire(t0)
    s0 = d0["a"].double().sum()
    assert torch.equal(d0["b"].cpu(), batches[0]["b"])
    pf.release(t0)
    t2 = pf.submit(batches[2])  # reuses slot 0 after its release event
    assert t2 == t0
    assert torch.equal(pf.acquire(t1)["a"].cpu(), batches[1]["a"])
    pf.release(t1)
    assert torch.equal(pf.acquire(t2)["a"].cpu(), batches[2]["a"])
    assert abs(s0.item() - batches[0]["a"].double().sum().item()) < 1e-6
    with pytest.raises(RuntimeError, match="pinned"):
        pf.submit({"a": torch.zeros(4), "b": batches[0]["b"]})


def test_npz_test_set_through_prefetcher_matches_direct_path(rb, tmp_path):
    """test.py:152-212 data path: test-set .npz -> pinned host -> HostPrefetcher -> reset -> x8 aug -> policy; same tours
    and costs as feeding the tensors directly."""
    B, n, S = 6, 20, 21
    raw = synth.make_instances("rcvrp", B, n, seed=5)
    data = {k: raw[k].numpy() for k in ("depot", "locs", "distance_matrix")}
    data["demand"] = (raw["demand"] * 30).numpy()
    data["capacity"] = np.full(B, 30, np.float32)
    np.savez(tmp_path / "rcvrp20.npz", **data)
    td_host = rb.prepare_test_td(rb.load_npz_to_tensordict(str(tmp_path / "rcvrp20.npz"), pin=True), "rcvrp")
    env = rb.get_env("rcvrp", generator_params={"num_loc": n}, check_solution=False)
    row, col = synth.random_embeddings(8 * B, n + 1, seed=6)
    p = omodel.init_decoder_params("rcvrp", seed=7)
    pf = rb.HostPrefetcher(dev)
    costs, acts = [], []
    for i, batch in enumerate(rb.iter_batches(td_host, 4)):
        b = batch.batch_size[0]
        d = pf.acquire(pf.submit({k: batch[k].contiguous().pin_memory() for k in batch.keys()}))
        td = rb.batchify(env.reset(rb.TensorDictLite(dict(d), batch_size=[b])), 8)
        sel = torch.cat([torch.arange(4 * i, 4 * i + b) + a * B for a in range(8)])
        pol = make_policy(rb, "rcvrp", p, row[sel].to(dev), col[sel].to(dev))
        out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
        costs.append(rb.unbatchify(out["reward"], (8, S)).amax(-1).amax(-1).cpu())
        acts.append(out["actions"].cpu())
    raw2 = TD({**{k: raw[k] for k in ("depot", "locs", "distance_matrix")}, "demand": torch.from_numpy(data["demand"]) / 30},
              batch_size=[B])
    td = rb.batchify(env.reset(lite(rb, raw2)), 8)
    pol = make_policy(rb, "rcvrp", p, row.to(dev), col.to(dev))
    out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    want = rb.unbatchify(out["reward"], (8, S)).amax(-1).amax(-1).cpu()
    got = torch.cat(costs)
    # identical inputs -> identical costs: one thread issues every MMA in a fixed order, so the rollout is bitwise
    # reproducible whatever the batch composition (DESIGN 4.2)
    assert torch.equal(got, want)


def test_env_edge_cases(rb):
    env = rb.RCVRPEnv(generator_params={"num_loc": 3}, check_solution=True)
    # demand exactly filling the vehicle is feasible (strict >), one that overflows by an ulp is not
    raw = TD({"locs": torch.rand(2, 3, 2), "depot": torch.rand(2, 2), "distance_matrix": torch.rand(2, 4, 4),
              "demand": torch.tensor([[0.5, 0.5, 1.0], [0.5, 0.5000001, 0.25]])}, batch_size=[2])
    td = env.reset(lite(rb, raw))
    assert td["action_mask"].cpu().tolist() == [[False, True, True, True]] * 2
    td.set("action", torch.tensor([1, 1], device=dev))
    td = env.step(td)["next"]
    assert td["action_mask"].cpu().tolist() == [[True, False, True, False], [True, False, False, True]]
    assert td["current_node"].shape == (2, 1) and td["visited"].dtype == torch.uint8
    # empty batch is a no-op
    empty = TD({"locs": torch.rand(0, 3, 2), "depot": torch.rand(0, 2), "distance_matrix": torch.rand(0, 4, 4),
                "demand": torch.rand(0, 3)}, batch_size=[0])
    assert env.reset(lite(rb, empty))["action_mask"].shape == (0, 4)
    # invalid tours are rejected with the reference's message
    with pytest.raises(AssertionError, match="Invalid tour"):
        env.get_reward(td, torch.tensor([[1, 1, 2, 0], [1, 2, 3, 0]], device=dev))


# ----------------------------------------------------------------------------------------------------
# gather + reset normalisation
# ----------------------------------------------------------------------------------------------------
def test_gather_matches_reference_sampler_golden(rb):
    from rrnco_b200.sampler import CityOnDevice, gather_submatrix
    z = np.load(os.path.join(GOLDEN, "sampler.npz"))
    city = {k[5:]: z[k] for k in z.files if k.startswith("city.")}
    c = CityOnDevice(city)
    idx = torch.from_numpy(z["indices"])
    assert np.array_equal(gather_submatrix(c.distance, idx).cpu().numpy(), z["c.distance_matrix"].astype(np.float32))
    assert np.array_equal(gather_submatrix(c.duration, idx).cpu().numpy(), z["tw.duration_matrix"].astype(np.float32))
    # the fp32 copy of the city matrix (what Real_World_Sampler gathers from) gives the same bits
    assert np.array_equal(gather_submatrix(c.distance_f32, idx).cpu().numpy(), z["c.distance_matrix"].astype(np.float32))
    np.random.seed(4321)
    s = rb.Real_World_Sampler(with_duration=True).sample(c, 5, 11)
    assert np.array_equal(s["distance_matrix"].cpu().numpy(), z["tw.distance_matrix"].astype(np.float32))
    assert np.array_equal(s["points"].cpu().numpy(), z["tw.points"].astype(np.float32))
    with pytest.raises(ValueError):
        rb.Real_World_Sampler().sample(c, 0, 3)
    with pytest.raises(ValueError):
        rb.Real_World_Sampler().sample(c, 2, 61)


def test_gather_full_size_and_fused_normalise(rb):
    from rrnco_b200.sampler import CityOnDevice, gather_submatrix
    city = synth.make_city(3, 1000)
    rng = np.random.RandomState(0)
    idx = osampler.uniform_sample(256, 1000, 101, rng)
    want = torch.from_numpy(osampler.gather_submatrix(city["distance"], idx).astype(np.float32))
    c = CityOnDevice(city)
    got = gather_submatrix(c.distance, torch.from_numpy(idx))
    assert torch.equal(got.cpu(), want)
    got_n, mn, mx = gather_submatrix(c.distance, torch.from_numpy(idx), normalize=True)
    lo, hi = want.amin((1, 2), keepdim=True), want.amax((1, 2), keepdim=True)
    assert torch.equal(got_n.cpu(), (want - lo) / (hi - lo + 1e-6))
    assert torch.equal(mn.cpu(), lo.flatten()) and torch.equal(mx.cpu(), hi.flatten())
    for src in (c.distance, c.distance_f32):  # fp64 / fp32 source, shared-memory tile (n = 101) and re-read path (n = 300)
        for n in (101, 300):
            idx_n = osampler.uniform_sample(8, 1000, n, np.random.RandomState(n))
            w = torch.from_numpy(osampler.gather_submatrix(city["distance"], idx_n).astype(np.float32))
            g_n, mn_n, mx_n = gather_submatrix(src, torch.from_numpy(idx_n), normalize=True)
            lo_n, hi_n = w.amin((1, 2), keepdim=True), w.amax((1, 2), keepdim=True)
            assert torch.equal(gather_submatrix(src, torch.from_numpy(idx_n)).cpu(), w)
            assert torch.equal(g_n.cpu(), (w - lo_n) / (hi_n - lo_n + 1e-6)) and torch.equal(mn_n.cpu(), lo_n.flatten())
    # idempotence property: gathering with the identity permutation returns the (cast) matrix itself
    ident = torch.arange(1000).unsqueeze(0)
    assert torch.equal(gather_submatrix(c.distance, ident)[0].cpu(), torch.from_numpy(city["distance"].astype(np.float32)))


# ----------------------------------------------------------------------------------------------------
# decoder logits / fused rollout vs the reference's golden outputs
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["atsp", "rcvrp", "rcvrptw"])
def test_decoder_and_rollout_vs_reference_golden(rb, name):
    z = load(f"policy_{name}.npz")
    B = z["row_emb"].shape[0]
    raw = TD({k[3:]: v for k, v in z.items() if k.startswith("in.")}, batch_size=[B])
    p = {k[6:]: v for k, v in z.items() if k.startswith("param.")}
    n = raw["distance_matrix"].shape[-1] - (0 if name == "atsp" else 1)
    S = z["num_starts"]
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=(name != "rcvrptw"))
    row, col = z["row_emb"].to(dev), z["col_emb"].to(dev)
    pol = make_policy(rb, name, p, row, col)
    assert env.get_num_starts(env.reset(lite(rb, raw))) == S

    # RRNetDecoder.forward at the mid-rollout state, driven through env.step like upstream's loop
    td = rb.batchify(env.reset(lite(rb, raw)), S)
    for t in range(4):
        td.set("action", z["greedy.actions"][:, t].to(dev))
        td = env.step(td)["next"]
    _, _, cache = pol.decoder.pre_decoder_hook(td, env, (row, col), S)
    logits, mask = pol.decoder(td, cache, S)
    assert torch.equal(mask.cpu(), z["mid.mask"])
    assert logits.dtype == torch.float32 and logits.shape == z["mid.logits"].shape
    assert (logits.cpu() - z["mid.logits"]).abs().max() < 2e-5

    # RRNetPolicy.forward (fused rollout): tours identical, reward / log-likelihood within tolerance
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert torch.equal(out["actions"].cpu(), z["greedy.actions"])
    assert out["actions"].dtype == torch.int64
    assert rel(out["reward"].cpu(), z["greedy.reward"]) < 1e-6
    assert rel(out["normalized_reward"].cpu(), z["greedy.normalized_reward"]) < 1e-6
    assert (out["log_likelihood"].cpu() - z["greedy.log_likelihood"]).abs().max() < 1e-4
    # rewards are consistent with env.get_reward on the emitted tours (independent kernel)
    tdb = rb.batchify(env.reset(lite(rb, raw)), S)
    real, norm = env.get_reward(tdb, out["actions"])
    assert rel(real, out["reward"]) < 1e-6

    # non-multistart evaluate (flat td, start action scored by the policy; atsp uses the placeholder context)
    rowb, colb = rb.batchify(row, S), rb.batchify(col, S)
    pol2 = make_policy(rb, name, p, rowb, colb)
    td_flat = rb.batchify(env.reset(lite(rb, raw)), S)
    out2 = pol2(td_flat, env, phase="val", actions=z["greedy.actions"].to(dev))
    assert torch.equal(out2["actions"].cpu(), z["greedy.actions"])
    assert (out2["log_likelihood"].cpu() - z["evaluate.log_likelihood"]).abs().max() < 1e-4
    assert rel(out2["reward"].cpu(), z["evaluate.reward"]) < 1e-6


@pytest.mark.parametrize("name,n,B", [("rcvrp", 100, 16), ("atsp", 100, 8), ("rcvrptw", 100, 8), ("rcvrp", 50, 8),
                                       ("atsp", 128, 2), ("rcvrp", 7, 5),
                                       # key-tile boundaries of the tcgen05 engine: N = 16, 34, 112 (last size of the
                                       # 13-tile variant), 120 (16-tile variant with time windows)
                                       ("rcvrp", 15, 4), ("atsp", 34, 3), ("rcvrp", 111, 2), ("rcvrptw", 119, 2)])
def test_greedy_rollout_vs_oracle(rb, name, n, B):
    raw = synth.make_instances(name, B, n, seed=n + B)
    oenv = oenvs.make_env(name, n, check_solution=False)
    otd = oenv.reset(raw)
    N = otd["action_mask"].shape[-1]
    S = oenv.get_num_starts(otd)
    row, col = synth.random_embeddings(B, N, seed=n)
    p = omodel.init_decoder_params(name, seed=n)
    oout = omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_greedy", num_starts=S)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=(name != "rcvrptw"))
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    acts, want = out["actions"].cpu(), oout["actions"]
    assert acts.shape[0] == want.shape[0] and abs(acts.shape[1] - want.shape[1]) <= 2
    T = max(acts.shape[1], want.shape[1])  # a flipped decision may lengthen one tour: pad with depot visits
    acts = torch.nn.functional.pad(acts, (0, T - acts.shape[1]))
    want = torch.nn.functional.pad(want, (0, T - want.shape[1]))
    same = (acts == want).all(1)
    assert same.float().mean() >= 0.99, same.float().mean()
    # identical tours must give (near-)identical reward and log-likelihood
    assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
    ll, oll = out["log_likelihood"].cpu()[same], oout["log_likelihood"][same]
    assert ((ll - oll).abs() <= 1e-5 * oll.abs() + 5e-5).all()  # sum of ~T fp32 log-probs of magnitude ~1
    best, obest = out["reward"].cpu().view(S, B).max(0)[0], oout["reward"].view(S, B).max(0)[0]
    assert (((best - obest).abs() / obest.abs()) < 1e-4).float().mean() >= 0.999
    # every emitted tour is feasible (reference's own validity oracle)
    if name != "rcvrptw":
        env.check_solution_validity(rb.batchify(env.reset(lite(rb, raw)), S), out["actions"])


def test_fp16_operand_overflow_is_loud(rb):
    """The tcgen05 engine computes on fp16 hi | lo operand pairs (|activation| < 4094): an overflow must surface as the
    reference's "Logits contain NaNs" assertion (decoder.py:303-304), never as silently wrong tours."""
    name, n, B = "rcvrp", 20, 2
    raw = synth.make_instances(name, B, n, seed=3)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=4)
    p = omodel.init_decoder_params(name, seed=5)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    with torch.no_grad():
        pol.decoder.pointer.ffn.lins[0].weight.mul_(1.0e5)  # hidden activations ~1e5 >> fp16 range
    with pytest.raises(AssertionError, match="Logits contain NaNs"):
        pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=env.get_num_starts(td))


def test_more_starts_than_one_tile(rb):
    """num_starts > 128 spans two CTA tiles per instance (start nodes wrap around, as upstream's modulo does)."""
    name, n, B, S = "rcvrp", 40, 3, 150
    raw = synth.make_instances(name, B, n, seed=8)
    oenv = oenvs.make_env(name, n, check_solution=False)
    row, col = synth.random_embeddings(B, n + 1, seed=9)
    p = omodel.init_decoder_params(name, seed=10)
    oout = omodel.policy_forward(p, oenv, oenv.reset(raw), row, col, decode_type="multistart_greedy", num_starts=S)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert out["actions"].shape == oout["actions"].shape
    assert (out["actions"].cpu() == oout["actions"]).all(1).float().mean() >= 0.99
    assert rel(out["reward"].cpu(), oout["reward"]) < 1e-4


@pytest.mark.parametrize("engine", [0, 1])
def test_ffn_engines_agree(rb, engine):
    """Both FFN engines of the fused kernel (mma.sync / tcgen05) reproduce the oracle's tours."""
    rb.set_ffn_engine(engine)
    try:
        test_greedy_rollout_vs_oracle(rb, "rcvrp", 50, 8)
        test_greedy_rollout_vs_oracle(rb, "rcvrptw", 20, 4)
    finally:
        rb.set_ffn_engine(2)  # the default: the lean kernel for N <= 112


def test_pointer_ffn_tcgen05(rb):
    """Standalone tcgen05 FFN (decoder.py:272-277,296) vs a torch fp64 reference: fp32-level accuracy."""
    from rrnco_b200 import _lib
    from rrnco_b200._lib import call, ptr, stream_ptr
    torch.manual_seed(0)
    for M in (1, 127, 128, 300):
        g = torch.randn(M, 128, device=dev)
        lin1, lin2 = torch.nn.Linear(128, 512).to(dev), torch.nn.Linear(512, 128).to(dev)
        w1, b1, w2, b2 = [t.detach().contiguous() for t in (lin1.weight, lin1.bias, lin2.weight, lin2.bias)]
        out = torch.empty_like(g)
        ws = torch.empty(_lib.lib().rrnco_pointer_ffn_workspace_bytes(), dtype=torch.uint8, device=dev)
        call("rrnco_pointer_ffn", M, ptr(g), ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(out), ptr(ws), stream_ptr())
        g64 = g.double()
        ref = torch.relu(g64 @ w1.double().t() + b1.double()) @ w2.double().t() + b2.double() + g64
        assert (out.double() - ref).abs().max() < 2e-5


_LARGE_N_ORACLE = {}


@pytest.mark.parametrize("path", ["fused", "stepwise"])
@pytest.mark.parametrize("name,n,B,S", [("atsp", 150, 2, None), ("rcvrp", 140, 2, None), ("rcvrptw", 130, 2, 40),
                                         ("atsp", 1000, 1, 100), ("atsp", 257, 3, 130), ("rcvrp", 300, 2, 70)])
def test_large_n_rollout_vs_oracle(rb, name, n, B, S, path):
    """N > 128 (incl. BASELINE's ATSP n=1000 generalisation case, 100 starts like test.py:129-130) through both CUDA paths:
    "fused" = the key-tiled persistent tcgen05 kernel (rollout_tiled.cu: one launch per rollout), "stepwise" = decoder +
    select + env-step kernels per decode step.  Matrices are never replicated over the starts."""
    raw = synth.make_instances(name, B, n, seed=n)
    oenv = oenvs.make_env(name, n, check_solution=False)
    otd = oenv.reset(raw)
    N = otd["action_mask"].shape[-1]
    S = oenv.get_num_starts(otd) if S is None else S
    row, col = synth.random_embeddings(B, N, seed=n + 1)
    p = omodel.init_decoder_params(name, seed=n + 2)
    if (name, n, B, S) not in _LARGE_N_ORACLE:  # the CPU oracle run is shared by the two paths
        with torch.inference_mode():
            _LARGE_N_ORACLE[(name, n, B, S)] = omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_greedy",
                                                                      num_starts=S)
    oout = _LARGE_N_ORACLE[(name, n, B, S)]
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    pol.large_n_path = path
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    if path == "fused":
        assert rb.models.FALLBACKS["softmax_range"] == 0  # the fused kernel served it
    acts, want = out["actions"].cpu(), oout["actions"]
    T = max(acts.shape[1], want.shape[1])
    acts = torch.nn.functional.pad(acts, (0, T - acts.shape[1]))
    want = torch.nn.functional.pad(want, (0, T - want.shape[1]))
    same = (acts == want).all(1)
    assert same.float().mean() >= 0.97, same.float().mean()
    assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
    ll, oll = out["log_likelihood"].cpu()[same], oout["log_likelihood"][same]
    assert ((ll - oll).abs() <= 2e-5 * oll.abs() + 2e-3).all(), (ll - oll).abs().max()
    best, obest = out["reward"].cpu().view(S, B).max(0)[0], oout["reward"].view(S, B).max(0)[0]
    assert ((best - obest).abs() / obest.abs() < 1e-4).all()
    if name == "atsp":  # every tour is a permutation
        assert (out["actions"].sort(1)[0] == torch.arange(N, device=dev)).all()


def test_key_tiled_kernel_exact_softmax_shift_on_peaked_heads(rb):
    """rollout_tiled.cu picks the softmax shift per decode step: the Cauchy-Schwarz bound when every head's scores stay
    within +-4.8, else a first sweep of single-term scores for the masked row maxima.  Embeddings scaled x2 give scores of
    +-13 (peaked heads, every step in the second mode): tours / costs / log-likelihoods must still match the fp32 oracle,
    and the per-step pipeline (running maximum).  Scaled x14 the scores leave even that sweep's range: the policy must then
    serve the call through the per-step pipeline (loud status bit, counted), never return the fused kernel's numbers."""
    name, n, B, S = "atsp", 300, 2, 64
    raw = synth.make_instances(name, B, n, seed=5)
    oenv = oenvs.make_env(name, n, check_solution=False)
    row, col = synth.random_embeddings(B, n, seed=6)
    row, col = 2.0 * row, 2.0 * col
    p = omodel.init_decoder_params(name, seed=7)
    with torch.inference_mode():
        oout = omodel.policy_forward(p, oenv, oenv.reset(raw), row, col, decode_type="multistart_greedy", num_starts=S)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    before = rb.models.FALLBACKS["softmax_range"]
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert rb.models.FALLBACKS["softmax_range"] == before
    same = _same_tours(out["actions"].cpu(), oout["actions"])
    assert same.float().mean() >= 0.95, same.float().mean()  # (peaked heads amplify the 1e-6 logit noise of any fp32 path)
    assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
    ll, oll = out["log_likelihood"].cpu()[same], oout["log_likelihood"][same]
    assert ((ll - oll).abs() <= 2e-5 * oll.abs() + 2e-3).all(), (ll - oll).abs().max()
    pol.large_n_path = "stepwise"
    out2 = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert _same_tours(out["actions"], out2["actions"]).float().mean() >= 0.95
    # beyond the single-term sweep's range: fused kernel refuses loudly, the policy falls back to the per-step kernels
    pol14 = make_policy(rb, name, p, (7.0 * row).to(dev), (7.0 * col).to(dev))
    cache = pol14.decoder._precompute_cache(((7.0 * row).to(dev), (7.0 * col).to(dev)))
    td = env.reset(lite(rb, raw))
    with pytest.raises(rb.models.SoftmaxRangeError):
        rb.fused_rollout(pol14.decoder, cache, env, td, S, True, "greedy", check=False)
    out3 = pol14(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert rb.models.FALLBACKS["softmax_range"] == before + 1
    assert (out3["actions"].sort(1)[0] == torch.arange(n, device=dev)).all()


def test_key_tiled_kernel_tilings_and_single_start(rb):
    """rollout_tiled.cu: (a) one CTA per tile, CTA pairs and start-split tilings (rrnco_set_start_split 2 / 0 / 1) decode the
    same tours; (b) the non-multistart path (one rollout per instance, learned placeholder query at step 0 for ATSP,
    depot start for the VRPs) matches the per-step pipeline and the oracle."""
    L = rb._lib.lib()
    name, n, B, S = "atsp", 180, 3, 90
    raw = synth.make_instances(name, B, n, seed=41)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    row, col = synth.random_embeddings(B, n, seed=42)
    p = omodel.init_decoder_params(name, seed=43)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    td = env.reset(lite(rb, raw))
    outs = {}
    try:
        for mode in (0, 1, 2):
            assert L.rrnco_set_start_split(mode) == 0
            outs[mode] = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
        assert L.rrnco_rollout_tile_rows(0, n, B, S) == 128
        L.rrnco_set_start_split(1)
        assert L.rrnco_rollout_tile_rows(0, n, B, S) == 32  # 148 SMs / 3 instances: whole warps of 32 starts
    finally:
        L.rrnco_set_start_split(0)
    for mode in (1, 2):
        assert torch.equal(outs[mode]["actions"], outs[0]["actions"]), mode
        assert torch.equal(outs[mode]["reward"], outs[0]["reward"])
        assert (outs[mode]["log_likelihood"] - outs[0]["log_likelihood"]).abs().max() < 1e-3
    for name, n, B in (("atsp", 150, 5), ("rcvrp", 139, 4)):
        raw = synth.make_instances(name, B, n, seed=n)
        oenv = oenvs.make_env(name, n, check_solution=False)
        otd = oenv.reset(raw)
        N = otd["action_mask"].shape[-1]
        row, col = synth.random_embeddings(B, N, seed=n + 1)
        p = omodel.init_decoder_params(name, seed=n + 2)
        with torch.inference_mode():
            oout = omodel.policy_forward(p, oenv, otd, row, col, decode_type="greedy")
        env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
        pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
        out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="greedy")
        same = _same_tours(out["actions"].cpu(), oout["actions"])
        assert same.float().mean() >= 0.75, (name, same)  # B rollouts only: at most one may differ
        assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
        pol.large_n_path = "stepwise"
        out2 = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="greedy")
        assert _same_tours(out["actions"], out2["actions"]).float().mean() >= 0.75


def test_key_tiled_kernel_sampling_evaluate_and_determinism(rb):
    """rollout_tiled.cu, the other decode modes at N > 128: sampling draws arg-max(v + Gumbel) with the same Philox
    counters as rrnco_select_action (so the per-step pipeline with the same seed samples the same tours), evaluate mode
    reproduces the per-step log-probs of those tours, and two runs are bitwise identical."""
    name, n, B, S = "rcvrp", 200, 3, 64
    raw = synth.make_instances(name, B, n, seed=21)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    row, col = synth.random_embeddings(B, n + 1, seed=22)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=23), row.to(dev), col.to(dev))
    td = env.reset(lite(rb, raw))
    kw = dict(phase="val", decode_type="multistart_sampling", num_starts=S, seed=99, return_sum_log_likelihood=False)
    out = pol(td, env, **kw)
    again = pol(td, env, **kw)
    assert torch.equal(out["actions"], again["actions"]) and torch.equal(out["log_likelihood"], again["log_likelihood"])
    assert torch.equal(out["reward"], again["reward"])
    srt = out["actions"].sort(1)[0]
    assert (srt[:, -n:] == torch.arange(1, n + 1, device=dev)).all() and (srt[:, :-n] == 0).all()
    pol.large_n_path = "stepwise"
    ref = pol(td, env, **kw)
    pol.large_n_path = "fused"
    same = _same_tours(out["actions"], ref["actions"])
    assert same.float().mean() >= 0.97, same.float().mean()
    T = min(out["log_likelihood"].shape[1], ref["log_likelihood"].shape[1])
    assert (out["log_likelihood"][same][:, :T] - ref["log_likelihood"][same][:, :T]).abs().max() < 1e-4
    assert rel(out["reward"][same], ref["reward"][same]) < 1e-6
    # evaluate: the sampled decisions forced back in give the same per-step log-probs
    ev = pol(td, env, phase="train", num_starts=S, actions=out["actions"][:, 1:], return_sum_log_likelihood=False)
    assert torch.equal(ev["actions"], out["actions"])
    assert (ev["log_likelihood"] - out["log_likelihood"]).abs().max() < 1e-5
    assert rel(ev["reward"], out["reward"]) < 1e-6
    # not a multiple of four nodes (bias rows not 16-byte aligned: 4-byte cp.async pieces) and more starts than one tile
    name, n, S = "atsp", 203, 203
    raw = synth.make_instances(name, 2, n, seed=31)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    row, col = synth.random_embeddings(2, n, seed=32)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=33), row.to(dev), col.to(dev))
    td = env.reset(lite(rb, raw))
    a = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    pol.large_n_path = "stepwise"
    b = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    same = _same_tours(a["actions"], b["actions"])
    assert same.float().mean() >= 0.97 and rel(a["reward"][same], b["reward"][same]) < 1e-6


@pytest.mark.parametrize("name,n,S", [("atsp", 200, 37), ("rcvrptw", 150, 20), ("rcvrp", 133, 5)])
def test_large_n_tiled_decoder_matches_the_streaming_one(rb, name, n, S):
    """rrnco_decoder_logits_large: shared-memory key tiles per (instance, start group) vs one warp streaming per rollout,
    on a mid-rollout state with ragged groups.  Both use the same accumulation order; the tcgen05 FFN between the two
    stages is reproducible to the last ulp only (several MMA-issuing threads), hence a 2e-6 bar instead of bit equality."""
    B = 3
    raw = synth.make_instances(name, B, n, seed=n)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=n + 1)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=n + 2), row.to(dev), col.to(dev))
    cache = pol.decoder._precompute_cache((row.to(dev), col.to(dev)))
    from rrnco_b200.models import _ROLLOUT_STATE_KEYS
    roll = rb.TensorDictLite({k: (rb.batchify(td[k], S) if k in _ROLLOUT_STATE_KEYS[name] else td[k])
                              for k in td.keys() if k != "done"}, batch_size=[B * S])
    g = torch.Generator().manual_seed(n)
    for _ in range(7):  # a few random feasible transitions so that masks / current nodes differ between the starts
        a = torch.multinomial(roll["action_mask"].float().cpu(), 1, generator=g).squeeze(1).to(dev)
        roll.set("action", a)
        roll = env.step(roll)["next"]
    try:
        rb.set_step_tiling(1)
        tiled_mma, _ = pol.decoder(roll, cache, S)
        rb.set_step_tiling(2)
        tiled, _ = pol.decoder(roll, cache, S)
        rb.set_step_tiling(0)
        streamed, _ = pol.decoder(roll, cache, S)
    finally:
        rb.set_step_tiling(1)
    assert torch.isfinite(tiled).all() and (tiled - streamed).abs().max().item() < 2e-6
    # 3xTF32 tensor-core logits: fp32-faithful, not the same rounding (bar of the logits elsewhere in this file: 2e-5)
    assert torch.isfinite(tiled_mma).all() and (tiled_mma - streamed).abs().max().item() < 1e-5


@pytest.mark.parametrize("name,n,B", [("rcvrp", 50, 6), ("rcvrptw", 30, 4), ("atsp", 40, 3)])
def test_training_handoff_replay_matches_fused_kernel_loglik(rb, name, n, B):
    """rl.py:99-130 hand-off: actions sampled by the fused kernel; the differentiable batched replay (env replayed on the
    CUDA step kernels, all decode steps as dense torch ops) reproduces the kernel's log-likelihoods and yields finite,
    non-zero gradients for the decoder parameters and the encoder output."""
    raw = synth.make_instances(name, B, n, seed=n)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    N = td["action_mask"].shape[-1]
    S = env.get_num_starts(td)
    row, col = synth.random_embeddings(B, N, seed=n + 1)
    row, col = row.to(dev).requires_grad_(True), col.to(dev).requires_grad_(True)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=n + 2), row, col)
    with torch.no_grad():
        out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S)
    ll = rb.replay_log_likelihood(pol, td, env, out["actions"], S, embeddings=(row, col))
    assert ll.shape == out["log_likelihood"].shape and ll.requires_grad
    assert (ll - out["log_likelihood"]).abs().max().item() < 2e-3, (ll - out["log_likelihood"]).abs().max()
    # the drop-in form: phase "train" with grad enabled returns the differentiable log-likelihood itself (rl.py:119-128)
    out_t = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=77)
    with torch.no_grad():
        out_k = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=77)
    assert out_t["log_likelihood"].requires_grad and torch.equal(out_t["actions"], out_k["actions"])
    assert (out_t["log_likelihood"] - out_k["log_likelihood"]).abs().max().item() < 2e-3
    loss = rb.pomo_shared_baseline_loss(out["reward"], ll, S) + rb.pomo_shared_baseline_loss(out_t["reward"], out_t["log_likelihood"], S)
    loss.backward()
    for gname, gten in (("W1", pol.decoder.pointer.ffn.lins[0].weight.grad), ("Wnode", pol.decoder.project_node_embeddings.weight.grad),
                        ("alpha", pol.decoder.alpha.grad), ("row", row.grad), ("col", col.grad)):
        assert gten is not None and torch.isfinite(gten).all() and gten.abs().max() > 0, gname


def test_per_step_decoder_entry_points_agree_below_128_nodes(rb):
    """RRNetDecoder.forward at N <= 128: `rrnco_decoder_logits` (the N <= 128 per-step kernel) and the any-N tile kernels
    (`rrnco_decoder_logits_large`, the default from 8 starts per instance) give the same logits (bar 2e-5)."""
    from rrnco_b200 import _lib
    from rrnco_b200.models import _ROLLOUT_STATE_KEYS
    name, n, B, S = "rcvrptw", 50, 5, 19
    raw = synth.make_instances(name, B, n, seed=3)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=4)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=5), row.to(dev), col.to(dev))
    cache = pol.decoder._precompute_cache((row.to(dev), col.to(dev)))
    roll = rb.TensorDictLite({k: (rb.batchify(td[k], S) if k in _ROLLOUT_STATE_KEYS[name] else td[k])
                              for k in td.keys() if k != "done"}, batch_size=[B * S])
    g = torch.Generator().manual_seed(1)
    for _ in range(5):
        a = torch.multinomial(roll["action_mask"].float().cpu(), 1, generator=g).squeeze(1).to(dev)
        roll.set("action", a)
        roll = env.step(roll)["next"]
    keep = _lib.MIN_STARTS_TILED
    try:
        tiled, _ = pol.decoder(roll, cache, S)
        _lib.MIN_STARTS_TILED = 1 << 30
        small, _ = pol.decoder(roll, cache, S)
    finally:
        _lib.MIN_STARTS_TILED = keep
    assert torch.isfinite(tiled).all() and (tiled - small).abs().max().item() < 2e-5


def test_select_action_matches_process_logits(rb):
    """rrnco_select_action == decoding.py process_logits + greedy / evaluate on random logits and masks."""
    g = torch.Generator().manual_seed(3)
    R, N = 257, 333
    logits = torch.randn(R, N, generator=g) * 3
    mask = torch.rand(R, N, generator=g) < 0.4
    mask[:, 0] = True
    logp = omodel.process_logits(logits.clone(), mask)
    a, lp, _ = rb.select_action(logits.to(dev), mask.to(dev), "greedy")
    assert torch.equal(a.cpu(), logp.argmax(-1))
    assert (lp.cpu() - logp.gather(1, a.cpu()[:, None]).squeeze(1)).abs().max() < 1e-5
    forced = torch.multinomial(mask.float(), 1, generator=g).squeeze(1)
    a2, lp2, _ = rb.select_action(logits.to(dev), mask.to(dev), "evaluate", forced_action=forced.to(dev))
    assert torch.equal(a2.cpu(), forced)
    assert (lp2.cpu() - logp.gather(1, forced[:, None]).squeeze(1)).abs().max() < 1e-5


def test_evaluate_multistart_vs_oracle(rb):
    name, n, B = "rcvrptw", 30, 6
    raw = synth.make_instances(name, B, n, seed=9)
    oenv = oenvs.make_env(name, n)
    otd = oenv.reset(raw)
    S = oenv.get_num_starts(otd)
    row, col = synth.random_embeddings(B, n + 1, seed=2)
    p = omodel.init_decoder_params(name, seed=4)
    g = torch.Generator().manual_seed(0)
    osamp = omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_sampling", num_starts=S, generator=g)
    forced = osamp["actions"][:, 1:]
    oev = omodel.policy_forward(p, oenv, oenv.reset(raw), row, col, num_starts=S, actions=forced)
    env = rb.get_env(name, generator_params={"num_loc": n})
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    out = pol(env.reset(lite(rb, raw)), env, phase="train", num_starts=S, actions=forced.to(dev),
              return_sum_log_likelihood=False)
    assert torch.equal(out["actions"].cpu(), osamp["actions"])
    assert (out["log_likelihood"].cpu() - oev["logprobs"]).abs().max() < 1e-4
    assert rel(out["reward"].cpu(), oev["reward"]) < 1e-6
    # an infeasible forced action is reported with the reference's message
    bad = forced.clone()
    bad[:, 0] = osamp["actions"][:, 0]  # revisit the start node
    with pytest.raises(AssertionError, match="infeasible action selected"):
        pol(env.reset(lite(rb, raw)), env, phase="train", num_starts=S, actions=bad.to(dev))


# ----------------------------------------------------------------------------------------------------
# sampling: Gumbel-max with a counter RNG -- exact twin in numpy, plus a distribution test
# ----------------------------------------------------------------------------------------------------
def philox4x32(c0, c1, c2, c3, k0, k1):
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c = [np.asarray(x, dtype=np.uint64) for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [(hi1 ^ c[1] ^ k0) & mask, lo1, (hi0 ^ c[3] ^ k1) & mask, lo0]
        k0, k1 = (k0 + np.uint64(W0)) & mask, (k1 + np.uint64(W1)) & mask
    return c


def gumbel_twin(seed, n_inst, S, N):
    """noise(step, [R,N]): Gumbel noise of (rollout r, step, column c) = Philox(seed; (r, step, c >> 2))[c & 3],
    r = s * n_inst + b the reference-layout rollout id -- the kernels' documented mapping."""
    def noise(step_idx, shape):
        step = step_idx - 1  # the strategy has already stored the forced start
        R = S * n_inst
        r = np.repeat(np.arange(R), N)
        c = np.tile(np.arange(N), R)
        x = philox4x32(r & 0xFFFFFFFF, r >> 32, np.full(R * N, step), c >> 2, seed & 0xFFFFFFFF, seed >> 32)
        x = np.stack(x, 0)[c & 3, np.arange(R * N)]
        u = ((x >> np.uint64(9)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 8388608.0)  # rrnco_u01
        return torch.from_numpy((-np.log(-np.log(u))).astype(np.float32).reshape(R, N))
    return noise


def test_sampling_matches_gumbel_twin_and_is_valid(rb):
    name, n, B, seed = "rcvrp", 20, 3, 77
    raw = synth.make_instances(name, B, n, seed=5)
    oenv = oenvs.make_env(name, n)
    otd = oenv.reset(raw)
    S = oenv.get_num_starts(otd)
    row, col = synth.random_embeddings(B, n + 1, seed=3)
    p = omodel.init_decoder_params(name, seed=6)
    oout = omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_sampling", num_starts=S,
                                 gumbel_noise=gumbel_twin(seed, B, S, n + 1))
    env = rb.get_env(name, generator_params={"num_loc": n})
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    with torch.no_grad():  # the kernel's own log-likelihood (with grad enabled phase "train" returns the replayed one)
        out = pol(env.reset(lite(rb, raw)), env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=seed)
    T = min(out["actions"].shape[1], oout["actions"].shape[1])
    same = (out["actions"].cpu()[:, :T] == oout["actions"][:, :T]).all(1)
    assert same.float().mean() >= 0.97, same.float().mean()  # identical noise => identical sampled tours
    ll, oll = out["log_likelihood"].cpu()[same], oout["log_likelihood"][same]
    assert ((ll - oll).abs() <= 1e-5 * oll.abs() + 5e-5).all()
    env.check_solution_validity(rb.batchify(env.reset(lite(rb, raw)), S), out["actions"])
    with torch.no_grad():
        out_b = pol(env.reset(lite(rb, raw)), env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=seed + 1)
    assert not torch.equal(out_b["actions"][:, : T], out["actions"][:, : T])  # different seed, different tours


def test_sampling_distribution_chi_square(rb):
    """First sampled decision over many seeds follows softmax(logits) (chi-square, 5 sigma)."""
    name, n, B = "atsp", 12, 1
    raw = synth.make_instances(name, B, n, seed=1)
    oenv = oenvs.make_env(name, n)
    otd = oenv.reset(raw)
    S = n
    row, col = synth.random_embeddings(B, n, seed=8)
    p = omodel.init_decoder_params(name, seed=8)
    trace = []
    omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_greedy", num_starts=S, trace=trace)
    probs = omodel.process_logits(trace[0]["logits"].clone(), trace[0]["mask"]).exp()[0]  # rollout s=0, b=0
    env = rb.get_env(name, generator_params={"num_loc": n})
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    td0 = env.reset(lite(rb, raw))
    counts = torch.zeros(n)
    trials = 600
    with torch.no_grad():
        for sd in range(trials):
            out = pol(td0, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=1000 + sd)
            counts[out["actions"][0, 1].item()] += 1
    exp = probs * trials
    keep = exp > 5
    chi2 = (((counts - exp) ** 2) / exp.clamp_min(1e-9))[keep].sum().item()
    dof = int(keep.sum()) - 1
    assert chi2 < dof + 5 * (2 * dof) ** 0.5 + 5, (chi2, dof)


# ----------------------------------------------------------------------------------------------------
# the 99.9 % bar at a size where it means something: 1024 instances per env at n = 100 (configs C1-C3 sizes)
# ----------------------------------------------------------------------------------------------------
def _chunked_oracle(p, oenv, raw, row, col, S, chunk, dtype=torch.float32):
    """Greedy multistart oracle rollout in chunks (upstream's batchify replicates every [N,N] matrix S times:
    128 instances x 100 starts x 101^2 fp32 = 0.5 GB per matrix and chunk)."""
    best, acts = [], []
    B = raw.batch_size[0]
    pp = omodel.cast_params(p, dtype) if dtype != torch.float32 else p
    with torch.inference_mode():
        for i in range(0, B, chunk):
            b = min(chunk, B - i)
            sub = TD({k: v[i:i + chunk] for k, v in raw.items()}, batch_size=[b])
            o = omodel.policy_forward(pp, oenv, oenv.reset(sub), row[i:i + chunk].to(dtype), col[i:i + chunk].to(dtype),
                                      decode_type="multistart_greedy", num_starts=S)
            best.append(o["reward"].float().view(S, b).max(0)[0].clone())
            acts.append(o["actions"].view(S, b, -1).clone())
    return torch.cat(best), acts


def _same_tours(a, b):
    T = max(a.shape[-1], b.shape[-1])
    return (torch.nn.functional.pad(a, (0, T - a.shape[-1])) == torch.nn.functional.pad(b, (0, T - b.shape[-1]))).all(-1)


@pytest.mark.parametrize("name", ["rcvrp", "atsp", "rcvrptw"])
def test_greedy_cost_parity_on_1024_instances(rb, name, capsys):
    """North-star bar: greedy rollouts from identical random-init weights give per-instance costs within 1e-4 relative
    on >= 99.9 % of instances -- asserted on 1024 instances (at most ONE may miss), n = 100, POMO multistart
    (decoding.py:272-298, test.py:210-212 reduction).  The fp32-oracle-vs-fp64-oracle disagreement on the first 128
    instances is the noise floor of the discontinuous argmax and is printed beside it; the same inputs are run twice
    and must give bitwise identical outputs (fixed MMA issue order)."""
    B, n, chunk, B64 = 1024, 100, 128, 128
    raw = synth.make_instances(name, B, n, seed=2025)
    oenv = oenvs.make_env(name, n, check_solution=False)
    S = oenv.get_num_starts(oenv.reset(TD({k: v[:2] for k, v in raw.items()}, batch_size=[2])))
    N = n if name == "atsp" else n + 1
    row, col = synth.random_embeddings(B, N, seed=77)
    p = omodel.init_decoder_params(name, seed=1234)
    obest, oacts = _chunked_oracle(p, oenv, raw, row, col, S, chunk)
    raw64 = TD({k: v[:B64] for k, v in raw.items()}, batch_size=[B64])
    o64best, o64acts = _chunked_oracle(p, oenv, raw64, row[:B64], col[:B64], S, chunk, torch.float64)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    outs = []
    for _ in range(2):
        out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
        outs.append({k: out[k].cpu() for k in ("actions", "reward", "log_likelihood")})
    # run-to-run determinism: bitwise
    for k in ("actions", "reward", "log_likelihood"):
        assert torch.equal(outs[0][k], outs[1][k]), k
    best = outs[0]["reward"].view(S, B).max(0)[0]
    relc = (best - obest).abs() / obest.abs()
    frac = (relc < 1e-4).float().mean().item()
    ga = outs[0]["actions"].view(S, B, -1)
    same = torch.cat([_same_tours(ga[:, i * chunk:(i + 1) * chunk], oa) for i, oa in enumerate(oacts)], 1)
    floor_c = ((obest[:B64] - o64best).abs() / o64best.abs() < 1e-4).float().mean().item()
    floor_t = _same_tours(oacts[0], o64acts[0]).float().mean().item()
    with capsys.disabled():
        print(f"\n[parity-1024] {name}: instances within 1e-4: {frac:.5f} (max rel {relc.max():.2e}); rollouts with "
              f"identical tours {same.float().mean():.5f}; noise floor (fp32 vs fp64 oracle, {B64} instances): "
              f"instances {floor_c:.5f}, tours {floor_t:.5f}; run-to-run bitwise identical")
    assert frac >= 0.999, frac
    assert same.float().mean() >= 0.999, same.float().mean()


def test_sampling_twin_rcvrptw_n100(rb):
    """Config C3's decode mode at C3's shape: RCVRPTW n=100, multistart sampling (decoding.py:284-298), against the oracle
    driven by the NumPy twin of the kernel's Philox / Gumbel stream; also bitwise run-to-run."""
    name, n, B, seed = "rcvrptw", 100, 8, 4242
    raw = synth.make_instances(name, B, n, seed=31)
    oenv = oenvs.make_env(name, n, check_solution=False)
    otd = oenv.reset(raw)
    S = oenv.get_num_starts(otd)
    assert S == 100
    row, col = synth.random_embeddings(B, n + 1, seed=32)
    p = omodel.init_decoder_params(name, seed=33)
    with torch.inference_mode():
        oout = omodel.policy_forward(p, oenv, otd, row, col, decode_type="multistart_sampling", num_starts=S,
                                     gumbel_noise=gumbel_twin(seed, B, S, n + 1))
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=seed)
        out_b = pol(env.reset(lite(rb, raw)), env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=seed)
    assert torch.equal(out["actions"], out_b["actions"]) and torch.equal(out["log_likelihood"], out_b["log_likelihood"])
    same = _same_tours(out["actions"].cpu(), oout["actions"])
    assert same.float().mean() >= 0.97, same.float().mean()  # identical noise => identical sampled tours
    ll, oll = out["log_likelihood"].cpu()[same], oout["log_likelihood"][same]
    assert ((ll - oll).abs() <= 1e-5 * oll.abs() + 1e-4).all()
    assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
    # every customer exactly once
    srt = out["actions"].sort(1)[0]
    assert (srt[:, -n:] == torch.arange(1, n + 1, device=dev)).all() and (srt[:, :-n] == 0).all()


def test_c4_shape_atsp_n1000_batch4_vs_oracle(rb):
    """Config C4's shape with more than one instance: ATSP n=1000, 4 instances x 100 starts (test.py:129-130), through the
    key-tiled fused kernel (8 key tiles)."""
    name, n, B, S = "atsp", 1000, 4, 100
    raw = synth.make_instances(name, B, n, seed=1000)
    oenv = oenvs.make_env(name, n, check_solution=False)
    row, col = synth.random_embeddings(B, n, seed=1001)
    p = omodel.init_decoder_params(name, seed=1002)
    with torch.inference_mode():
        oout = omodel.policy_forward(p, oenv, oenv.reset(raw), row, col, decode_type="multistart_greedy", num_starts=S)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    same = _same_tours(out["actions"].cpu(), oout["actions"])
    assert same.float().mean() >= 0.97, same.float().mean()
    assert rel(out["reward"].cpu()[same], oout["reward"][same]) < 1e-6
    best, obest = out["reward"].cpu().view(S, B).max(0)[0], oout["reward"].view(S, B).max(0)[0]
    assert ((best - obest).abs() / obest.abs() < 1e-4).all()
    assert (out["actions"].sort(1)[0] == torch.arange(n, device=dev)).all()


def test_truncated_rollout_is_reported_and_open_route_reward_does_not_mutate(rb, caplog):
    """A rollout cut at t_cap with unfinished tours sets RRNCO_DEV_TRUNCATED and is logged like policy.py:222-226;
    RMTVRPEnv.get_reward leaves the reset td's matrix alone for open routes (upstream mutates a throw-away copy)."""
    import logging
    name, n, B = "rcvrptw", 20, 3
    raw = synth.make_instances(name, B, n, seed=9)
    raw["open_route"] = torch.tensor([[True], [False], [True]])
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    S = env.get_num_starts(td)
    row, col = synth.random_embeddings(B, n + 1, seed=10)
    p = omodel.init_decoder_params(name, seed=11)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    cache = pol.decoder._precompute_cache((row.to(dev), col.to(dev)))
    with caplog.at_level(logging.ERROR, logger="rrnco_b200"):
        out = rb.fused_rollout(pol.decoder, cache, env, td, S, True, "greedy", t_cap=6)
    assert out["actions"].shape[1] == 6
    assert any("Exceeded maximum number of steps" in r.message for r in caplog.records)
    caplog.clear()
    before = td["distance_matrix"].clone()
    with caplog.at_level(logging.ERROR, logger="rrnco_b200"):
        full = rb.fused_rollout(pol.decoder, cache, env, td, S, True, "greedy")
    assert not caplog.records
    real, norm = env.get_reward(td, full["actions"])  # un-replicated td: rollout r reads row r % B
    assert torch.equal(td["distance_matrix"], before)
    assert rel(real, full["reward"]) < 1e-6
    real_b, _ = env.get_reward(rb.batchify(td, S), full["actions"])  # upstream's layout (its own copy is zeroed)
    assert torch.equal(td["distance_matrix"], before) and torch.equal(real_b, real)
    # oracle (= upstream's in-place zeroing on its own copy) agrees
    oenv = oenvs.make_env(name, n, check_solution=False)
    otd = obatchify(oenv.reset(raw), S)
    oreal, _ = oenv.get_reward(otd, full["actions"].cpu())
    assert rel(real.cpu(), oreal) < 1e-6


# ----------------------------------------------------------------------------------------------------
# on-device instance generation, un-materialised x8 augmentation
# ----------------------------------------------------------------------------------------------------
def test_gather_duration_law_and_outlier_city(rb):
    """rrnco_gather_submatrix normalize == 2 = the generators' duration law (rmtvrp/generator_lazy.py:365-369), incl. a
    constant matrix; a city with > 1e5 entries is cleaned at upload like sampler.py:41-60 (reference golden)."""
    from rrnco_b200.sampler import CityOnDevice, gather_submatrix
    city = synth.make_city(5, length=300)
    city["duration"][:40, :40] = 3.25  # instances drawn from here have a zero range
    dev_city = CityOnDevice(city, dev)
    rng = np.random.RandomState(3)
    idx = np.array([rng.choice(300, 31, replace=False) for _ in range(64)])
    idx[7] = np.arange(31)  # constant sub-matrix
    got, mn, mx = gather_submatrix(dev_city.duration_f32, torch.from_numpy(idx), normalize=2)
    raw = torch.from_numpy(city["duration"][idx[:, :, None], idx[:, None, :]].astype(np.float32))
    lo, hi = raw.amin(dim=(1, 2), keepdim=True), raw.amax(dim=(1, 2), keepdim=True)
    want = (raw - lo) / torch.where(hi - lo == 0, torch.ones_like(hi), hi - lo)
    assert torch.equal(got.cpu(), want) and (got[7] == 0).all()
    assert torch.equal(mn.cpu(), lo.reshape(-1)) and torch.equal(mx.cpu(), hi.reshape(-1))
    z = np.load(os.path.join(GOLDEN, "sampler_outliers.npz"))
    bad_city = {k[5:]: z[k] for k in z.files if k.startswith("city.")}
    np.random.seed(99)
    s = rb.Real_World_Sampler(with_duration=True).sample(bad_city, 4, 9)
    assert torch.equal(s["distance_matrix"].cpu(), torch.from_numpy(z["distance_matrix"].astype(np.float32)))
    assert torch.equal(s["duration_matrix"].cpu(), torch.from_numpy(z["duration_matrix"].astype(np.float32)))
    assert torch.equal(s["points"].cpu(), torch.from_numpy(z["points"].astype(np.float32)))


@pytest.mark.parametrize("name", ["rcvrp", "rcvrptw", "atsp"])
def test_on_device_generator_feeds_the_rollout(rb, name):
    """Lazy*Generator on the device (10 synthetic cities -> gather -> laws) -> env.reset -> fused rollout: the instances
    obey the reference's laws and every tour is feasible; the generator's own arithmetic is pinned bit-exactly to the
    reference in tests/test_generator.py."""
    n, B = 50, 200
    cities = [synth.make_city(c, length=400) for c in range(12)]
    cls = {"rcvrp": rb.LazyRCVRPGenerator, "rcvrptw": rb.LazyRMTVRPGenerator, "atsp": rb.LazyATSPGenerator}[name]
    gen = cls(num_loc=n, cities=cities, device=dev, seed=11, chunk_size=100)
    td = gen(B)
    assert td.batch_size[0] == B and td["distance_matrix"].shape == (B, n + (name != "atsp"), n + (name != "atsp"))
    if name == "rcvrp":
        d = td["demand"] * 40.0  # CAPACITIES[50]
        assert (d >= 1).all() and (d < 10).all()
    if name == "rcvrptw":
        assert td["duration_matrix"].amin() == 0 and td["duration_matrix"].amax() == 1
        assert (td["time_windows"][:, 0, 1] == 4.6).all() and not td["open_route"].any()
        d = td["demand_linehaul"] * 40  # get_vehicle_capacity(50) = 40
        assert torch.equal(d.round(), d.round().clamp(1, 9)) and (td["demand_backhaul"] == 0).all()
    gen2 = cls(num_loc=n, cities=cities, device=dev, seed=11, chunk_size=100)
    assert torch.equal(gen2(B)["distance_matrix"], td["distance_matrix"])  # seeded: reproducible
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    tdr = env.reset(td)
    S = env.get_num_starts(tdr)
    N = n if name == "atsp" else n + 1
    row, col = synth.random_embeddings(B, N, seed=1)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=2), row.to(dev), col.to(dev))
    out = pol(tdr, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    srt = out["actions"].sort(1)[0]
    if name == "atsp":
        assert (srt == torch.arange(n, device=dev)).all()
    else:
        assert (srt[:, -n:] == torch.arange(1, n + 1, device=dev)).all() and (srt[:, :-n] == 0).all()
    if name == "rcvrp":
        env.check_solution_validity(rb.batchify(tdr, S), out["actions"])


def test_shared_instance_augmentation_equals_materialised(rb):
    """StateAugmentation(dihedral8, share_instance_data=True) -> reset -> RRNetPolicy.forward gives the same tours and
    rewards as upstream's materialised batchify x8 (transforms.py:142-154, test.py:188-212)."""
    for n, B, A, S in ((30, 5, 8, 31), (135, 2, 8, 20)):  # the lean kernel; the key-tiled kernel (136 nodes, CTA pairs)
        raw = synth.make_instances("rcvrp", B, n, seed=21)
        env = rb.get_env("rcvrp", generator_params={"num_loc": n}, check_solution=False)
        row, col = synth.random_embeddings(A * B, n + 1, seed=22)
        pol = make_policy(rb, "rcvrp", omodel.init_decoder_params("rcvrp", seed=23), row.to(dev), col.to(dev))
        outs = []
        for share in (False, True):
            aug = rb.StateAugmentation(num_augment=A, augment_fn="dihedral8", no_aug_coords=False, share_instance_data=share)
            td = env.reset(aug(lite(rb, raw)))
            assert td.batch_size[0] == A * B and td["distance_matrix"].shape[0] == (B if share else A * B)
            out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
            outs.append((out["actions"].cpu(), out["reward"].cpu(), td["locs"].cpu()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])


# ----------------------------------------------------------------------------------------------------
# bindings: TORCH_LIBRARY ops vs ctypes over the same C ABI; real-TensorDict duck typing
# ----------------------------------------------------------------------------------------------------
def test_torch_ops_and_ctypes_bindings_agree(rb):
    """Every hot call goes through `torch.ops.rrnco_b200.*` by default; the ctypes fallback must give bitwise the same."""
    from rrnco_b200 import torch_ops
    assert torch_ops.enabled(), "librrnco_b200_torch.so missing: the torch-op binding is the default"
    res = {}
    for binding in (True, False):
        assert rb.use_torch_ops(binding) == binding
        for name, n, B in (("rcvrp", 20, 3), ("atsp", 12, 2), ("rcvrptw", 15, 2)):
            raw = synth.make_instances(name, B, n, seed=3)
            env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
            td = env.reset(lite(rb, raw))
            S = env.get_num_starts(td)
            N = td["action_mask"].shape[-1]
            row, col = synth.random_embeddings(B, N, seed=4)
            pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=5), row.to(dev), col.to(dev))
            out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
            with torch.no_grad():
                smp = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=7)
            # per-step API: one env.step + get_reward on the batchified td
            tdb = rb.batchify(td, S)
            tdb.set("action", env.select_start_nodes(td, S))
            tdb = env.step(tdb)["next"]
            real, norm = env.get_reward(rb.batchify(td, S), out["actions"])
            res.setdefault(name, []).append([out["actions"], out["reward"], out["log_likelihood"], smp["actions"],
                                             smp["log_likelihood"], tdb["action_mask"], tdb["current_node"], real, norm])
        city = rb.CityOnDevice(synth.make_city(2, length=120), dev)
        idx = torch.from_numpy(np.array([np.random.RandomState(1).choice(120, 21, replace=False) for _ in range(9)]))
        from rrnco_b200.sampler import gather_submatrix
        res.setdefault("gather", []).append(list(gather_submatrix(city.distance_f32, idx, normalize=1)) +
                                            [gather_submatrix(city.distance, idx)])
    rb.use_torch_ops(True)
    for name, (a, b) in res.items():
        for x, y in zip(a, b):
            assert x.shape == y.shape and torch.equal(x, y), name


def test_reference_tensordict_duck_typing(rb):
    """The envs / policy accept a TensorDict-like container that is NOT rrnco_b200's own (here the stand-in that the golden
    generator runs the unmodified reference on): td[...], td.set, td.update, td.keys, td.batch_size, td.device."""
    import sys
    shims = os.path.join(os.path.dirname(os.path.dirname(__file__)), "oracle", "shims")
    sys.path.insert(0, shims)
    try:
        from tensordict import TensorDict
    finally:
        sys.path.remove(shims)
    name, n, B = "rcvrp", 20, 3
    raw = synth.make_instances(name, B, n, seed=8)
    td_ref = TensorDict({k: v.to(dev) for k, v in raw.items()}, batch_size=[B])
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=True)
    td = env.reset(td_ref)
    assert type(td).__name__ == "TensorDict" and td["action_mask"].shape == (B, n + 1)
    row, col = synth.random_embeddings(B, n + 1, seed=9)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=10), row.to(dev), col.to(dev))
    out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=n + 1)
    want = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_greedy", num_starts=n + 1)
    assert torch.equal(out["actions"], want["actions"]) and torch.equal(out["reward"], want["reward"])


# ----------------------------------------------------------------------------------------------------
# full BASELINE sizes: size-independent properties
# ----------------------------------------------------------------------------------------------------
def test_full_size_rcvrp_rollout_properties(rb):
    """RCVRP n=100, 128 instances x 8 aug x 101 starts: all tours valid, in-kernel reward == independent
    tour-reward kernel, evaluate replay reproduces the log-likelihood, best-of-aug reduction."""
    n, B, A = 100, 128, 8
    raw = synth.make_instances("rcvrp", B, n, seed=11)
    env = rb.RCVRPEnv(generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    td_aug = rb.batchify(td, A)
    S = env.get_num_starts(td_aug)
    assert S == 101
    row, col = synth.random_embeddings(A * B, n + 1, seed=12)
    p = omodel.init_decoder_params("rcvrp", seed=13)
    pol = make_policy(rb, "rcvrp", p, row.to(dev), col.to(dev))
    out = pol(td_aug, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    acts = out["actions"]
    R = A * B * S
    assert acts.shape[0] == R and out["reward"].shape == (R,)
    # permutation property: every customer exactly once, zeros elsewhere
    srt = acts.sort(1)[0]
    assert (srt[:, -n:] == torch.arange(1, n + 1, device=dev)).all() and (srt[:, :-n] == 0).all()
    # capacity property via the reference's running-load check on a slice (the loop is O(T) launches)
    sl = slice(0, 20000)
    tdb = rb.TensorDictLite({"demand": td_aug["demand"][torch.arange(R, device=dev)[sl] % (A * B)],
                             "vehicle_capacity": torch.ones(20000, 1, device=dev)}, batch_size=[20000])
    env.check_solution_validity(tdb, acts[sl])
    # reward == independent tour-length kernel over un-replicated matrices (data_rows = A*B)
    from rrnco_b200.envs import tour_reward
    real, norm = tour_reward(acts, td_aug["distance_matrix"], True, None, td_aug["min_distance"], td_aug["max_distance"])
    assert rel(norm, out["normalized_reward"]) < 1e-6 and rel(real, out["reward"]) < 1e-6
    # evaluate replay of the greedy tours reproduces the log-likelihood
    out2 = pol(td_aug, env, phase="val", num_starts=S, actions=acts[:, 1:])
    # (same MMAs in the same order on both calls; only the select epilogue differs: forced column vs argmax)
    assert (out2["log_likelihood"] - out["log_likelihood"]).abs().max() < 1e-5
    assert torch.equal(out2["actions"], acts)
    # augmentation copies share matrices and (here) differ only by embeddings: best-of reduction shape
    best = rb.unbatchify(out["reward"], (A, S)).max(-1)[0].max(-1)[0]
    assert best.shape == (B,)


def test_full_size_c4_rollout_properties(rb):
    """BASELINE config C4 at its full size (ATSP n = 1000, 64 instances x 100 starts, 999 decode steps) through the
    key-tiled fused kernel with CTA pairs: every tour a permutation, in-kernel reward == the independent tour-reward kernel,
    log-likelihoods finite and negative, the evaluate replay of the greedy tours reproduces them, two runs are bitwise
    identical, and a sample of rollouts is re-decoded by the per-step pipeline."""
    name, n, B, S = "atsp", 1000, 64, 100
    raw = synth.make_instances(name, B, n, seed=31)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(lite(rb, raw))
    row, col = synth.random_embeddings(B, n, seed=32)
    pol = make_policy(rb, name, omodel.init_decoder_params(name, seed=33), row.to(dev), col.to(dev))
    before = rb.models.FALLBACKS["softmax_range"]
    out = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert rb.models.FALLBACKS["softmax_range"] == before  # served by the fused kernel (some CTAs in exact-shift mode)
    acts = out["actions"]
    assert acts.shape == (B * S, n)
    assert (acts.sort(1)[0] == torch.arange(n, device=dev)).all()
    assert (acts[:, 0].view(S, B) == (torch.arange(S, device=dev) % n)[:, None]).all()  # select_start_nodes
    from rrnco_b200.envs import tour_reward
    real, norm = tour_reward(acts, td["distance_matrix"], False, None, td["min_distance"], td["max_distance"])
    assert rel(norm, out["normalized_reward"]) < 1e-6 and rel(real, out["reward"]) < 1e-6
    ll = out["log_likelihood"]
    assert torch.isfinite(ll).all() and (ll < 0).all()
    again = pol(td, env, phase="val", decode_type="multistart_greedy", num_starts=S)
    assert torch.equal(again["actions"], acts) and torch.equal(again["log_likelihood"], ll)
    ev = pol(td, env, phase="val", num_starts=S, actions=acts[:, 1:])
    assert torch.equal(ev["actions"], acts)
    assert (ev["log_likelihood"] - ll).abs().max() < 1e-4
    # two instances again through the per-step kernels (running-maximum softmax, three-pass select)
    sub = rb.TensorDictLite({k: v[:2] for k, v in raw.items()}, batch_size=[2])
    pol2 = make_policy(rb, name, omodel.init_decoder_params(name, seed=33), row[:2].to(dev), col[:2].to(dev))
    pol2.large_n_path = "stepwise"
    ref = pol2(env.reset(lite(rb, sub)), env, phase="val", decode_type="multistart_greedy", num_starts=S)
    mine = acts.view(S, B, n)[:, :2].reshape(2 * S, n)
    same = (mine == ref["actions"]).all(1)
    assert same.float().mean() >= 0.97, same.float().mean()
