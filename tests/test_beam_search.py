"""Beam search (rl4co 0.6.0 BeamSearch, decoding.py:402-542) and select_best.

The reference is the oracle's decoder / envs with rl4co's BeamSearch restated here as a subclass of
oracle.model.Strategy (`BeamSearch`, `beam_step`, `backtrack`, `beam_forward`): the oracle has no beam search.  The rules
are the ones include/rrnco_b200.h states for rrnco_beam_select (ranking by value descending, then flat index ascending;
ranks from #finite upward copy rank 0).
CPU: the restated step against a brute-force sorted(), the restated search against the oracle's evaluate replay, argument
checks, and select_best.  GPU: rrnco_beam_select against the restated step, beam rollouts against the restated search.
Beam sets are compared per instance on the instances whose restated search never had two candidates within EPS of each
other at the beam cut (there fp32 rounding may legitimately change the kept set); the other instances are counted.
"""
import math

import pytest
import torch

from oracle import envs as oenvs, model as omodel, synth
from oracle.td import batchify

dev = "cuda"
EPS = 1e-4


# ---------------------------------------------------------------------------------------------------
# the restatement
# ---------------------------------------------------------------------------------------------------
def beam_step(lp, score, W):
    """One BeamSearch._make_beam_step on [W * B, N] log-probs in (w b) order -> (parent row, action, lp of the action in
    the parent's row, new score, cut margin [B]); the margin is the gap between the W-th and (W+1)-th candidate."""
    R, N = lp.shape
    B = R // W
    cand = (score[:, None] + lp).view(W, B, N).permute(1, 0, 2).reshape(B, W * N)
    vals, idx = torch.sort(cand, dim=1, descending=True, stable=True)  # equal values: lower flat index first
    margin = vals[:, W - 1] - vals[:, W]
    margin = torch.where(torch.isfinite(vals[:, W]), margin, torch.full_like(margin, math.inf))
    vals, idx = vals[:, :W], idx[:, :W]
    fill = torch.arange(W)[None, :] >= torch.isfinite(vals).sum(1, keepdim=True)  # _fill_up_beams
    vals = torch.where(fill, vals[:, :1], vals)
    idx = torch.where(fill, idx[:, :1], idx)
    parent = ((idx // N) * B + torch.arange(B)[:, None]).t().reshape(-1)
    action = (idx % N).t().reshape(-1)
    return parent, action, lp[parent, action], vals.t().reshape(-1), margin


def log_probs(logits, mask, temperature=1.0, clip=10.0):
    """oracle process_logits, with the masked entries of a fully masked row at -inf rather than NaN."""
    return omodel.process_logits(logits.clone(), mask, temperature, clip).masked_fill(~mask, -math.inf)


def brute_force_step(lp, score, W):
    """The same step with Python's sorted() over (-value, flat index), instance by instance."""
    R, N = lp.shape
    B = R // W
    parent, action, new = [0] * R, [0] * R, [0.0] * R
    for b in range(B):
        items = []
        for w in range(W):
            for n in range(N):
                v = (score[w * B + b] + lp[w * B + b, n]).item()  # fp32 add, as the kernel
                items.append((-v, w * N + n, v))
        top = sorted(items)[:W]
        fin = sum(1 for t in top if math.isfinite(t[2]))
        for rk in range(W):
            _, f, v = top[rk if rk < fin else 0]
            parent[rk * B + b], action[rk * B + b], new[rk * B + b] = (f // N) * B + b, f % N, v
    return torch.tensor(parent), torch.tensor(action), torch.tensor(new, dtype=torch.float32)


def backtrack(actions, parents, logprobs):
    """BeamSearch._backtrack on step-major [T, R] tensors -> [R, T] aligned actions and log-probs."""
    T, R = actions.shape
    cur = torch.arange(R)
    a, lp = torch.empty(R, T, dtype=actions.dtype), torch.empty(R, T, dtype=logprobs.dtype)
    for t in reversed(range(T)):
        a[:, t], lp[:, t] = actions[t, cur], logprobs[t, cur]
        cur = parents[t, cur]
    return a, lp


class BeamSearch(omodel.Strategy):
    """rl4co 0.6.0 BeamSearch restated on the oracle's Strategy surface (pre_decoder_hook / step / post_decoder_hook)."""

    def __init__(self, beam_width=None, temperature=1.0, tanh_clipping=10.0):
        super().__init__("greedy", multistart=False, temperature=temperature, tanh_clipping=tanh_clipping)
        self.beam_width, self.parents, self.score = beam_width, [], None
        self.margin = None

    def pre_decoder_hook(self, td, env):
        W = env.get_num_starts(td) if self.beam_width is None else self.beam_width
        if W < 2:
            raise ValueError("beam width must be >= 2")
        self.beam_width = W
        action = env.select_start_nodes(td, num_starts=W)
        td = batchify(td, W)
        td["action"] = action
        td = env.step(td)["next"]
        R = action.shape[0]
        self.actions.append(action)
        self.logprobs.append(torch.zeros(R, dtype=torch.float32))
        self.parents.append(torch.zeros(R, dtype=torch.int64))
        self.score = torch.zeros(R, dtype=torch.float32)
        self.margin = torch.full((R // W,), math.inf)
        return td, env, W

    def step(self, logits, mask, td, action=None):
        lp = omodel.process_logits(logits, mask, self.temperature, self.tanh_clipping, self.mask_logits)
        parent, sel, lp_sel, self.score, margin = beam_step(lp, self.score, self.beam_width)
        self.margin = torch.minimum(self.margin, margin)
        td = td[parent]  # each new beam continues from its parent's state
        td["action"] = sel
        self.actions.append(sel)
        self.logprobs.append(lp_sel)
        self.parents.append(parent)
        return td

    def post_decoder_hook(self, td, env):
        acts, lps = backtrack(torch.stack(self.actions), torch.stack(self.parents), torch.stack(self.logprobs))
        return lps, acts, td, env


def beam_forward(p, oenv, td, row, col, beam_width=None):
    """policy.py:175-255 with the restated BeamSearch; all W * B beams (select_best is applied by the caller)."""
    strat = BeamSearch(beam_width)
    td, env, W = strat.pre_decoder_hook(td, oenv)
    cache = omodel.precompute_cache(p, row, col)
    while not td["done"].all():
        logits, mask = omodel.decoder_forward(p, oenv.name, td, cache, W)
        td = strat.step(logits, mask, td)
        td = oenv.step(td)["next"]
    lps, acts, td, env = strat.post_decoder_hook(td, oenv)
    reward = oenv.get_reward(td, acts)
    reward = reward[0] if isinstance(reward, tuple) else reward
    return {"actions": acts, "logprobs": lps, "log_likelihood": lps.sum(1), "reward": reward, "W": W,
            "margin": strat.margin, "score": strat.score}


class StartsFrom:
    """An env whose select_start_nodes returns given start nodes (evaluate replays of beams that start anywhere)."""

    def __init__(self, env, starts):
        self._env, self._starts = env, starts

    def select_start_nodes(self, td, num_starts):
        return self._starts

    def __getattr__(self, k):
        return getattr(self._env, k)


def oracle_replay(p, oenv, raw, row, col, actions, W):
    """The oracle's multistart evaluate of [W * B, T] actions (column 0 = the start): per-step log-probs [W * B, T]."""
    out = omodel.policy_forward(p, StartsFrom(oenv, actions[:, 0]), oenv.reset(raw), row, col, num_starts=W,
                                actions=actions[:, 1:])
    return out["logprobs"]


def pick_best(reward, W):
    B = reward.shape[0] // W
    return reward.view(W, B).argmax(0) * B + torch.arange(B, device=reward.device)


def random_rows(seed, W=6, B=5, N=9):
    """[W * B, N] logits / masks / scores with masked entries, exact ties and a row group with < W finite candidates."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(W * B, N, generator=g) * 3
    mask = torch.rand(W * B, N, generator=g) < 0.6
    mask[:, 0] = True
    score = -torch.rand(W * B, generator=g) * 4
    # instance 1: two identical beams (duplicate starts) -> exact ties between their candidates
    logits[B + 1], mask[B + 1], score[B + 1] = logits[1], mask[1], score[1]
    # instance 2: saturated tanh -> ties at +-clip inside a row
    logits[2, :4] = 50.0
    # instance 3: fewer than W finite candidates (fill-up)
    for w in range(W):
        mask[w * B + 3] = False
    mask[3, :2] = True
    mask[B + 3, 1] = True
    return logits, mask, score


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_beam_step_matches_brute_force(seed):
    W, B, N = 6, 5, 9
    logits, mask, score = random_rows(seed, W, B, N)
    lp = log_probs(logits, mask)
    parent, action, lp_sel, new, _ = beam_step(lp, score, W)
    bp, ba, bn = brute_force_step(lp, score, W)
    assert torch.equal(parent, bp) and torch.equal(action, ba) and torch.equal(new, bn)
    assert torch.equal(lp_sel, lp[bp, ba])
    # fill-up: instance 3 has 3 finite candidates; ranks 3.. copy rank 0
    b3 = torch.arange(W) * B + 3
    assert torch.isfinite(new[b3]).sum() == W and len(set(action[b3[3:]].tolist())) == 1
    assert action[b3[3]] == action[b3[0]] and parent[b3[3]] == parent[b3[0]]
    # scores non-increasing by rank (except where fill-up copied rank 0)
    sc = new.view(W, B)[:, [0, 1, 2, 4]]
    assert (sc[1:] <= sc[:-1]).all()


@pytest.mark.parametrize("name,n,W", [("rcvrp", 8, 4), ("atsp", 7, 3), ("rcvrptw", 8, None)])
def test_restated_beam_search_is_consistent(name, n, W):
    B = 3
    raw = synth.make_instances(name, B, n, seed=5)
    oenv = oenvs.make_env(name, n, check_solution=False)
    N = n if name == "atsp" else n + 1
    row, col = synth.random_embeddings(B, N, seed=6)
    p = omodel.init_decoder_params(name, seed=7)
    out = beam_forward(p, oenv, oenv.reset(raw), row, col, W)
    W = out["W"]
    # the final score is the running fp32 sum of the aligned log-probs, non-increasing by rank
    assert torch.allclose(out["log_likelihood"], out["score"], atol=1e-5)
    sc = out["score"].view(W, B)
    assert (sc[1:] <= sc[:-1]).all()
    # each beam's log-likelihood is the oracle's evaluate replay of its actions
    lps = oracle_replay(p, oenv, raw, row, col, out["actions"], W)
    assert (lps.sum(1) - out["log_likelihood"]).abs().max() < 1e-5
    assert torch.isfinite(out["log_likelihood"]).all()


@pytest.mark.parametrize("bad", [1, 0, -3, 2.5])
def test_bad_beam_width_raises_before_launch(bad):
    from rrnco_b200.models import beam_args
    import rrnco_b200
    with pytest.raises(ValueError):
        beam_args(bad)
    with pytest.raises(ValueError):  # CPU tensors: nothing could be launched, the check comes first
        rrnco_b200.beam_select(torch.zeros(4, 3), torch.ones(4, 3, dtype=torch.bool), torch.zeros(4), bad)


def test_unsupported_beam_calls_raise():
    import rrnco_b200

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            raise AssertionError("not reached")

    class Td:
        device = torch.device("cpu")

    pol = rrnco_b200.RRNetPolicy(encoder=Enc(), env_name="rcvrp")
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="top_k"):
            pol(Td(), object(), phase="test", decode_type="beam_search", top_k=5)
        with pytest.raises(NotImplementedError, match="actions"):
            pol(Td(), object(), phase="test", decode_type="beam_search", actions=torch.zeros(2, 3, dtype=torch.long))
        with pytest.raises(ValueError):
            pol(Td(), object(), phase="test", decode_type="beam_search", beam_width=1)
    with torch.enable_grad():
        with pytest.raises(NotImplementedError, match="does not beam"):
            pol(Td(), object(), phase="train", decode_type="beam_search")


def test_c_abi_rejects_bad_beam_width_before_any_cuda_call():
    from rrnco_b200 import _lib
    from rrnco_b200.build import build_library
    build_library()
    h = _lib.lib()
    sel = lambda W: h.rrnco_beam_select(0, W, 10, None, None, None, 10.0, 1.0, None, None, None, None, None, None)
    assert sel(2) == 0  # zero instances: nothing to do
    for W in (1, 0, -5):
        assert sel(W) == -1, W
    assert sel(_lib.MAX_BEAM_WIDTH + 1) == -2
    assert h.rrnco_beam_backtrack(0, 3, None, None, None, None, None, None, None, None) == 0
    assert h.rrnco_beam_backtrack(4, 3, None, None, None, None, None, None, None, None) == -1


def test_select_best_rows_first_maximum():
    from rrnco_b200.models import select_best_rows
    S, B = 4, 3
    reward = torch.tensor([[-5.0, -2.0, -7.0], [-1.0, -2.0, -7.0], [-1.0, -3.0, -7.0], [-4.0, -2.0, -7.0]]).reshape(-1)
    acts = torch.arange(S * B * 5).view(S * B, 5)
    ll = torch.arange(S * B, dtype=torch.float32)
    out = select_best_rows({"reward": reward, "actions": acts, "log_likelihood": ll, "hidden": "cache"}, S)
    rows = torch.tensor([1 * B + 0, 0 * B + 1, 0 * B + 2])  # first maximum = lowest start index among equal rewards
    assert torch.equal(out["reward"], reward[rows]) and torch.equal(out["actions"], acts[rows])
    assert torch.equal(out["log_likelihood"], ll[rows]) and out["hidden"] == "cache"
    assert out["actions"].shape == (B, 5)


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rb():
    import rrnco_b200
    rrnco_b200.set_precision(3)
    return rrnco_b200


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("temperature,clip", [(1.0, 10.0), (0.7, 0.0)])
def test_beam_select_vs_restatement(rb, seed, temperature, clip):
    W, B, N = 6, 5, 9
    logits, mask, score = random_rows(seed, W, B, N)
    lp = log_probs(logits, mask, temperature, clip)
    parent, action, lp_sel, new, margin = beam_step(lp, score, W)
    a, par, l, s, st = rb.beam_select(logits.to(dev), mask.to(dev), score.to(dev), W, clip, temperature)
    assert int(st.item()) == 0
    clear = (margin > 1e-5).repeat(W)
    assert torch.equal(par.cpu()[clear], parent[clear]) and torch.equal(a.cpu()[clear], action[clear])
    assert ((s.cpu() - new).abs() <= 1e-6 * new.abs().clamp_min(1.0))[clear].all()
    assert ((l.cpu() - lp_sel).abs() <= 1e-5)[clear].all()
    # a larger case: 300 nodes, 40 beams
    g = torch.Generator().manual_seed(seed)
    W, B, N = 40, 7, 300
    logits = torch.randn(W * B, N, generator=g) * 3
    mask = torch.rand(W * B, N, generator=g) < 0.5
    mask[:, 0] = True
    score = -torch.rand(W * B, generator=g) * 10
    lp = log_probs(logits, mask, temperature, clip)
    parent, action, lp_sel, new, margin = beam_step(lp, score, W)
    a, par, l, s, st = rb.beam_select(logits.to(dev), mask.to(dev), score.to(dev), W, clip, temperature)
    clear = (margin > 1e-5).repeat(W)
    assert clear.any()
    # within a clear instance the kept set is the same; the ranks may swap only between near-equal scores
    for b in range(B):
        if clear[b]:
            rows = torch.arange(W) * B + b
            got = sorted(zip(par.cpu()[rows].tolist(), a.cpu()[rows].tolist()))
            want = sorted(zip(parent[rows].tolist(), action[rows].tolist()))
            assert got == want
    assert (s.cpu() - new).abs().max() <= 1e-5 * new.abs().max()


@pytest.mark.gpu
def test_beam_select_bindings_agree_and_fill_up(rb):
    from rrnco_b200 import torch_ops
    W, B, N = 6, 5, 9
    logits, mask, score = random_rows(3, W, B, N)
    args = (logits.to(dev), mask.to(dev), score.to(dev), W)
    g = torch.Generator().manual_seed(1)
    acts = torch.randint(0, N, (5, W * B), generator=g).to(dev)
    pars = torch.randint(0, W * B, (5, W * B), generator=g).to(dev)
    lps = torch.randn(5, W * B, generator=g).to(dev)
    outs = []
    for flag in (True, False):
        torch_ops.use_torch_ops(flag)
        try:
            outs.append(rb.beam_select(*args)[:4])
            outs.append(rb.beam_backtrack(acts, pars, lps)[:3])
        finally:
            torch_ops.use_torch_ops(True)
    for x, y in zip(outs[0] + outs[1], outs[2] + outs[3]):
        assert torch.equal(x, y)
    # the backtrack kernel against the restatement
    a, lp, ll = outs[1]
    wa, wl = backtrack(acts.cpu(), pars.cpu(), lps.cpu())
    assert torch.equal(a.cpu(), wa) and torch.equal(lp.cpu(), wl)
    assert (ll.cpu() - wl.double().sum(1).float()).abs().max() < 1e-6
    # fill-up on the device: instance 3 has 3 finite candidates
    act, par = outs[0][0].cpu(), outs[0][1].cpu()
    b3 = torch.arange(W) * B + 3
    assert (act[b3[3:]] == act[b3[0]]).all() and (par[b3[3:]] == par[b3[0]]).all()
    # parents of step 0 are never read; a parent row outside [0, R) later on is reported, and that row comes out NaN
    for flag in (True, False):
        torch_ops.use_torch_ops(flag)
        try:
            p2 = pars.clone()
            p2[0] = -7
            *_, st = rb.beam_backtrack(acts, p2, lps)
            assert int(st.item()) == 0
            p2[3, 4] = W * B
            a2, l2, ll2, st = rb.beam_backtrack(acts, p2, lps)
        finally:
            torch_ops.use_torch_ops(True)
        assert int(st.item()) & rb._lib.DEV_BAD_PARENT
        bad = torch.isnan(ll2.cpu())
        assert bad.any() and not bad.all()
        assert torch.isnan(l2.cpu()[bad][:, 0]).all() and (a2.cpu()[bad][:, 0] == 0).all()
        assert torch.equal(ll2.cpu()[~bad], ll.cpu()[~bad])


def lite(rb, td):
    return rb.TensorDictLite({k: v.to(dev) for k, v in td.items()}, batch_size=list(td.batch_size))


def setup_case(rb, name, N, B, seed, variant=""):
    n = N if name == "atsp" else N - 1
    raw = synth.make_instances(name, B, n, seed=seed)
    if variant:
        g = torch.Generator().manual_seed(seed)
        if "O" in variant:
            raw["open_route"] = torch.ones(B, 1, dtype=torch.bool)
        if "L" in variant:
            raw["distance_limit"] = torch.full((B, 1), 2.8)
        if "B" in variant:
            is_b = torch.rand(B, n, generator=g) < 0.3
            dl = raw["demand_linehaul"]
            raw["demand_backhaul"], raw["demand_linehaul"] = dl * is_b, dl * ~is_b
            raw["backhaul_class"] = torch.full((B, 1), 1.0)
    oenv = oenvs.make_env(name, n, check_solution=False)
    row, col = synth.random_embeddings(B, N, seed=seed + 1)
    p = omodel.init_decoder_params(name, seed=seed + 2)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row.to(dev), col.to(dev)

    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(p, strict=True)
    return raw, oenv, row, col, p, env, pol


def kernel_replay(rb, pol, env, raw, actions, W):
    """The kernels' own multistart evaluate of [W * B, T] actions whose column 0 is the start: log-likelihood [W * B]."""
    td = env.reset(lite(rb, raw))
    row, col = pol.encoder(td)
    cache = pol.decoder._precompute_cache((row, col), num_starts=W)
    out = rb.stepwise_rollout(pol.decoder, cache, StartsFrom(env, actions[:, 0]), td, W, True, "evaluate",
                              forced_actions=actions[:, 1:], calc_reward=False)
    return out["log_likelihood"]


def match_beam_sets(acts, reward, want, W, tag):
    """Per-instance beam sets (order-free: ranks may swap between near-equal scores) against the restated search, and the
    rewards of the same sequences.  Instances whose restated search had a cut margin <= EPS may differ (trajectories
    diverge after an fp32 flip); every other instance must match.  -> (matching instances, instances clear of near-ties)"""
    B = want["reward"].shape[0] // W
    acts, reward, oacts = acts.cpu(), reward.cpu(), want["actions"]
    same, n_clear = 0, 0
    for b in range(B):
        rows = torch.arange(W) * B + b
        clear = bool(want["margin"][b] > EPS)
        n_clear += clear
        got = sorted(tuple(x) for x in acts[rows].tolist())
        exp = sorted(tuple(x) for x in oacts[rows].tolist())
        if got == exp:
            same += 1
            gk = {tuple(x): float(r) for x, r in zip(acts[rows].tolist(), reward[rows])}
            for x, r in zip(oacts[rows].tolist(), want["reward"][rows]):
                assert abs(gk[tuple(x)] - float(r)) <= 1e-4 * max(1.0, abs(float(r))), (tag, b)
        else:
            assert not clear, (tag, b)
    print(f"{tag}: identical beam sets on {same} / {B} instances, {n_clear} clear of near-ties")
    assert same >= 0.999 * n_clear
    return same, n_clear


def compare_beams(rb, pol, env, raw, out, want, W, tag):
    match_beam_sets(out["actions"], out["reward"], want, W, tag)
    ll = kernel_replay(rb, pol, env, raw, out["actions"], W)
    assert (ll - out["log_likelihood"]).abs().max() < 1e-4, tag


def record_beam_steps(monkeypatch):
    """Records the inputs and outputs of every rrnco_beam_select call a beam rollout makes."""
    from rrnco_b200 import models
    real, rec = models.beam_select, []

    def spy(logits, mask, score, beam_width, *a, **k):
        res = real(logits, mask, score, beam_width, *a, **k)
        rec.append((logits.cpu(), mask.cpu(), score.cpu(), [x.cpu() for x in res[:4]]))
        return res
    monkeypatch.setattr(models, "beam_select", spy)
    return rec


def check_beam_steps(rec, W, tag, temperature=1.0, clip=10.0, near=1e-5, min_share=0.8):
    """Every recorded step against the restated step on the kernel's own logits, mask and scores: parents, actions and
    rank order bit-exact on each (step, instance) whose W + 1 best candidates hold no two values within `near` of each
    other, except exact ties (two candidates with bitwise-identical inputs: parent rows with the same logits, mask and
    score, and the same logit), which the tie rule decides and which are compared.  A zero gap between candidates whose
    inputs differ is a near-tie that fp32 rounding made equal in one of the two computations: not compared.  Scores within
    1e-6 relative.  -> compared selections that held exact ties."""
    n_all = n_cmp = n_tie = 0
    for logits, mask, score, (a, par, lp, new) in rec:
        lpr = log_probs(logits, mask, temperature, clip)
        parent, action, lp_sel, want, _ = beam_step(lpr, score, W)
        R, N = logits.shape
        B = R // W
        cand = (score[:, None] + lpr).view(W, B, N).permute(1, 0, 2).reshape(B, W * N)
        top, idx = cand.sort(dim=1, descending=True, stable=True)
        top, idx = top[:, : W + 1], idx[:, : W + 1]
        gaps = top[:, :-1] - top[:, 1:]
        fin = torch.isfinite(top[:, :-1]) & torch.isfinite(top[:, 1:])
        lbits, sbits = logits.view(torch.int32), score.view(torch.int32)
        for b in range(B):
            n_all += 1
            rows_of = (idx[b] // N) * B + b
            cols = idx[b] % N

            def same_inputs(i, j):
                r1, r2 = int(rows_of[i]), int(rows_of[j])
                return (lbits[r1, cols[i]] == lbits[r2, cols[j]] and sbits[r1] == sbits[r2]
                        and torch.equal(lbits[r1], lbits[r2]) and torch.equal(mask[r1], mask[r2]))
            tie, skip = False, False
            for i in torch.nonzero(fin[b] & (gaps[b] <= near)).flatten().tolist():
                if gaps[b, i] == 0 and same_inputs(i, i + 1):
                    tie = True
                else:
                    skip = True
                    break
            if skip:
                continue
            n_cmp += 1
            n_tie += tie
            rows = torch.arange(W) * B + b
            assert torch.equal(par[rows], parent[rows]) and torch.equal(a[rows], action[rows]), (tag, b)
            assert ((new[rows] - want[rows]).abs() <= 1e-5 + 1e-6 * want[rows].abs()).all(), (tag, b)
            assert ((lp[rows] - lp_sel[rows]).abs() <= 1e-5).all(), (tag, b)
    print(f"{tag}: {n_cmp} / {n_all} (step, instance) selections compared bit-exact, {n_tie} of them with exact ties")
    assert n_cmp >= min_share * n_all, (tag, n_cmp, n_all)
    return n_tie


BEAM_CASES = [(name, N, W) for name in ("atsp", "rcvrp", "rcvrptw") for N in (20, 50, 100) for W in (2, 8, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,W", BEAM_CASES)
def test_beam_search_vs_restatement(rb, name, N, W, monkeypatch):
    B = 3
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, 17 + N)
    want = beam_forward(p, oenv, oenv.reset(raw), row, col, W)
    W = want["W"]
    rec = record_beam_steps(monkeypatch)
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="test", decode_type="beam_search", beam_width=W, select_best=False)
    check_beam_steps(rec, W, f"{name} N={N} W={W}")
    with torch.no_grad():
        best = pol(env.reset(lite(rb, raw)), env, phase="test", decode_type="beam_search", beam_width=W)
    assert out["actions"].shape[0] == W * B and best["actions"].shape[0] == B
    compare_beams(rb, pol, env, raw, out, want, W, f"{name} N={N} W={W}")
    # select_best: first maximum of the reward over the beams, on the kernel's own beams
    rows = pick_best(out["reward"], W)
    for k in ("actions", "reward"):
        assert torch.equal(best[k], out[k][rows]), k
    # (two calls: from 8 beams on, the per-step decoder's tcgen05 FFN may round the last bit differently run to run)
    assert (best["log_likelihood"] - out["log_likelihood"][rows]).abs().max() < 1e-5
    # scores are non-increasing by rank (the final ranks hold the running sums)
    ll = out["log_likelihood"].view(W, B)
    assert (ll[1:] <= ll[:-1] + 1e-4).all()


@pytest.mark.gpu
def test_beam_search_rcvrptw_olb_and_augmentation(rb, monkeypatch):
    name, N, B = "rcvrptw", 50, 2
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, 3, variant="OLB")
    want = beam_forward(p, oenv, oenv.reset(raw), row, col, 8)
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="test", decode_type="beam_search", beam_width=8, select_best=False)
    compare_beams(rb, pol, env, raw, out, want, 8, "rcvrptw OLB N=50 W=8")
    # x8 augmentation: the beam runs on the 8 * B augmented instances
    raw8 = synth.make_instances("rcvrp", 2, 19, seed=4)
    oenv8 = oenvs.make_env("rcvrp", 19, check_solution=False)
    env8 = rb.get_env("rcvrp", generator_params={"num_loc": 19}, check_solution=False)
    td = rb.StateAugmentation(num_augment=8)(env8.reset(lite(rb, raw8)))
    Ba = td["action_mask"].shape[0]
    assert Ba == 16
    row8, col8 = synth.random_embeddings(Ba, 20, seed=9)
    p8 = omodel.init_decoder_params("rcvrp", seed=10)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row8.to(dev), col8.to(dev)

    pol8 = rb.RRNetPolicy(encoder=Enc(), env_name="rcvrp").to(dev)
    pol8.decoder.load_state_dict(p8, strict=True)
    rec = record_beam_steps(monkeypatch)
    with torch.no_grad():
        out8 = pol8(td, env8, phase="test", decode_type="beam_search", beam_width=5, select_best=False)
    check_beam_steps(rec, 5, "rcvrp x8 augmented N=20 W=5")
    want8 = beam_forward(p8, oenv8, batchify(oenv8.reset(raw8), 8), row8, col8, 5)
    match_beam_sets(out8["actions"], out8["reward"], want8, 5, "rcvrp x8 augmented N=20 W=5")


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,W", [("atsp", 130, 6), ("rcvrp", 200, 4), ("rcvrp", 100, 150)])
def test_beam_search_large_n_and_wide(rb, name, N, W, monkeypatch):
    B = 2
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, 5 + N)
    want = beam_forward(p, oenv, oenv.reset(raw), row, col, W)
    rec = record_beam_steps(monkeypatch)
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="test", decode_type="beam_search", beam_width=W, select_best=False)
    # more beams than start nodes: duplicate beams.  Their logits from the >= 8-beam decoder may differ in the last bit
    # (its FFN sums in no fixed order), and those near-ties are not compared; the bitwise-identical ones are exact ties
    # that the tie rule decides, and they must occur
    dup = W > N - 1
    n_tie = check_beam_steps(rec, W, f"{name} N={N} W={W}", min_share=0.5 if dup else 0.8)
    if dup:
        assert n_tie > 0
    compare_beams(rb, pol, env, raw, out, want, W, f"{name} N={N} W={W}")


@pytest.mark.gpu
@pytest.mark.parametrize("W", [4, 16])
def test_beam_search_is_reproducible_and_bindings_agree(rb, W):
    """Bitwise run to run and across bindings with fewer than 8 beams (N <= 128: the per-step decoder is the one-kernel
    rrnco_decoder_logits).  From 8 beams on, rrnco_decoder_logits_large's tcgen05 FFN accumulates its three split terms
    in no fixed order, so the log-probs may differ in the last bit: equal actions and rewards, log-probs within 1e-5."""
    from rrnco_b200 import torch_ops
    raw, oenv, row, col, p, env, pol = setup_case(rb, "rcvrp", 50, 4, 11)
    runs = []
    for flag in (True, True, False):
        torch_ops.use_torch_ops(flag)
        try:
            with torch.no_grad():
                runs.append(pol(env.reset(lite(rb, raw)), env, phase="test", decode_type="beam_search", beam_width=W,
                                select_best=False, return_sum_log_likelihood=False))
        finally:
            torch_ops.use_torch_ops(True)
    for other in runs[1:]:
        for k in ("actions", "reward"):
            assert torch.equal(runs[0][k], other[k]), k
        if W < 8:
            assert torch.equal(runs[0]["log_likelihood"], other["log_likelihood"])
        else:
            assert (runs[0]["log_likelihood"] - other["log_likelihood"]).abs().max() < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["multistart_greedy", "multistart_sampling"])
def test_multistart_select_best(rb, kind):
    raw, oenv, row, col, p, env, pol = setup_case(rb, "rcvrp", 30, 3, 23)
    S = 29
    with torch.no_grad():
        full = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type=kind, num_starts=S, seed=3)
        best = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type=kind, num_starts=S, seed=3, select_best=True)
        nocalc = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type=kind, num_starts=S, seed=3, select_best=True,
                     calc_reward=False)
    rows = pick_best(full["reward"], S)
    assert best["actions"].shape[0] == 3
    for k in ("actions", "reward", "log_likelihood"):
        assert torch.equal(best[k], full[k][rows]), k
        assert torch.equal(nocalc[k], full[k][rows]), k
