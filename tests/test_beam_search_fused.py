"""Fused beam search: rrnco_beam_rollout, the lean rollout kernel's beam instantiation (N <= 112, up to 128 beams).

Main bar: every step of the kernel's own walk against the oracle decoder in fp64.  The oracle env is replayed along the
kernel's step records (each step: its state gathered by the kernel's parent rows, then stepped with the kernel's
actions), and the fp64 decoder (tests/test_rollout_logprobs_fp64.py: Ref64, post_process, kappa) gives every candidate's
lp64 and score64 = score64[parent] + lp64.  Per (step, instance):
  * parents, actions and rank order equal the top W of score + lp64 wherever an adjacent gap of the W + 1 best
    candidates exceeds the sum of the two candidates' error bounds (C_BAR 2^-24 kappa of the lp and the fp32 rounding of
    the sum): a (step, instance) is compared when its W-th / (W+1)-th cut is clear, and then every rank is exact except
    within a run of near-tied candidates, whose ranks must hold the same candidates in some order.  `score` is the kernel's own fp32 running score, which its records give
    bit for bit (score[parent] + lp in fp32), so the ranking is held to the error of one step; an exact tie between
    candidates of bitwise-identical inputs (duplicate beams) is compared too, and the tie rule (lower flat index first)
    decides it;
  * each selected lp is within C_BAR 2^-24 kappa of lp64; each score is within the summed bounds plus fp32 rounding of
    score64, and scores are non-increasing by rank;
  * at least 80 % of the (step, instance) selections are compared.
The same cases also run the per-step pipeline (beam_search_rollout) and are cross-checked with it: rewards and
log-likelihoods of the tours both return agree.  On the shapes of test_beam_search_vs_restatement (N <= 100, W in
{2, 8, default}, T = 1, clip 10), which RRNetPolicy.forward now sends to the fused kernel, its steps are also checked
against the restated rule (check_beam_steps), which keeps the per-step pipeline's step-level coverage there.
"""
import pytest
import torch

from oracle import envs as oenvs, model as omodel, synth
from oracle.td import batchify as obatchify
from test_beam_search import check_beam_steps, lite, pick_best, record_beam_steps, setup_case
from test_rollout_logprobs_fp64 import C_BAR, U32, Ref64, post_process, ratios

dev = "cuda"
ENVS = ["atsp", "rcvrp", "rcvrptw"]


# ----------------------------------------------------------------------------------------------------
# CPU: C ABI argument checks and the routing rule
# ----------------------------------------------------------------------------------------------------
def test_c_abi_rejects_unsupported_calls_before_any_cuda_call():
    from rrnco_b200 import _lib
    from rrnco_b200.build import build_library
    build_library()
    h = _lib.lib()
    run = lambda N, W: h.rrnco_beam_rollout(1, N, 1, W, None, None, None, 2 * N + 3, None, None, None, None, None,  # noqa: E731
                                            None, None)
    for W in (1, 0, -4):
        assert run(50, W) == -1, W  # RRNCO_ERR_BAD_ARG
    assert run(50, 129) == -2 and run(113, 8) == -2 and run(200, 8) == -2  # RRNCO_ERR_UNSUPPORTED
    assert run(50, 8) == -1  # served shape, NULL arguments
    ws = lambda N, W: h.rrnco_beam_rollout_workspace_bytes(1, N, 4, W)  # noqa: E731
    assert ws(112, 128) > 0 and ws(2, 2) > 0
    assert ws(113, 8) == 0 and ws(50, 129) == 0 and ws(50, 1) == 0
    try:
        for engine in (0, 1):
            _lib.check(h.rrnco_set_ffn_engine(engine))
            assert run(50, 8) == -2 and ws(50, 8) == 0
        _lib.check(h.rrnco_set_ffn_engine(2))
        _lib.check(h.rrnco_set_precision(1))
        assert run(50, 8) == -2 and ws(50, 8) == 0
    finally:
        _lib.check(h.rrnco_set_ffn_engine(2))
        _lib.check(h.rrnco_set_precision(3))
    assert run(50, 8) == -1


def test_policy_routes_beam_calls(monkeypatch):
    """N <= 112 and W <= 128 under the default engine and precision: the fused kernel; anything else: the per-step
    pipeline.  The rollouts are replaced by recorders: no device is needed."""
    import types
    import rrnco_b200
    from rrnco_b200 import _lib, models
    from rrnco_b200.build import build_library
    build_library()
    calls = []

    def fake(tag):
        def run(decoder, cache, env, td, W, **kw):
            calls.append((tag, cache.glimpse_key.shape[1], W))
            z = torch.zeros(W * cache.glimpse_key.shape[0])
            return {"reward": z, "log_likelihood": z, "actions": torch.zeros(z.shape[0], 3, dtype=torch.long)}
        return run
    monkeypatch.setattr(models, "fused_beam_rollout", fake("fused"))
    monkeypatch.setattr(models, "beam_search_rollout", fake("per-step"))

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return None, None

    class Td:
        device = torch.device("cuda")

    pol = rrnco_b200.RRNetPolicy(encoder=Enc(), env_name="rcvrp")
    env = types.SimpleNamespace(get_num_starts=lambda td: 99)
    for N, W in [(20, 2), (112, 128), (112, None), (113, 8), (50, 129), (200, 4)]:
        monkeypatch.setattr(pol.decoder, "_precompute_cache",
                            lambda emb, num_starts=0, N=N: types.SimpleNamespace(glimpse_key=torch.empty(2, N, 1)))
        with torch.no_grad():
            pol(Td(), env, phase="test", decode_type="beam_search", beam_width=W, select_best=False)
    assert calls == [("fused", 20, 2), ("fused", 112, 128), ("fused", 112, 99), ("per-step", 113, 8),
                     ("per-step", 50, 129), ("per-step", 200, 4)]
    h = _lib.lib()
    try:
        _lib.check(h.rrnco_set_precision(1))
        assert not models.fused_beam_serves("rcvrp", 50, 8)
        _lib.check(h.rrnco_set_precision(3))
        _lib.check(h.rrnco_set_ffn_engine(1))
        assert not models.fused_beam_serves("rcvrp", 50, 8)
    finally:
        _lib.check(h.rrnco_set_ffn_engine(2))
        _lib.check(h.rrnco_set_precision(3))
    assert models.fused_beam_serves("rcvrp", 50, 8)


# ----------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rb():
    import rrnco_b200
    rrnco_b200.set_precision(3)
    return rrnco_b200


def run_fused(rb, pol, env, td, W, T=1.0, clip=10.0, per_step_logprobs=False, **kw):
    """One beam search through RRNetPolicy.forward on the fused route; also returns the kernel's step records
    (step-major actions, parent rows, log-probs: what rrnco_beam_backtrack reads)."""
    from rrnco_b200 import models
    assert models.fused_beam_serves(pol.env_name, td["action_mask"].shape[-1], W or env.get_num_starts(td))
    real, rec = models.beam_backtrack, []

    def spy(actions, parents, logprobs, *a, **k):
        rec.append((actions.cpu(), parents.cpu(), logprobs.cpu()))
        return real(actions, parents, logprobs, *a, **k)
    models.beam_backtrack = spy
    try:
        with torch.no_grad():
            out = pol(td, env, phase="test", decode_type="beam_search", beam_width=W, temperature=T, tanh_clipping=clip,
                      return_sum_log_likelihood=not per_step_logprobs, **kw)
    finally:
        models.beam_backtrack = real
    assert len(rec) == 1
    return out, rec[0]


def check_fp64_walk(name, n, p, row, col, raw, W, steps, T, clip, tag, min_share=0.8):
    """The kernel's step records against the fp64 decoder on the oracle env replayed along them (module docstring)."""
    acts, pars, lps = steps
    n_steps, R = acts.shape
    B = R // W
    ref = Ref64(name, p, row, col, dev)
    oenv = oenvs.make_env(name, n, check_solution=False)
    td = oenv.reset(raw)
    ref.set_instances(td)
    td = obatchify(td, W)
    assert torch.equal(acts[0], oenv.select_start_nodes(oenv.reset(raw), num_starts=W))
    td["action"] = acts[0]
    td = oenv.step(td)["next"]
    score64 = torch.zeros(R, dtype=torch.float64, device=dev)
    serr = torch.zeros(R, dtype=torch.float64, device=dev)
    score32 = torch.zeros(R, dtype=torch.float32)
    n_all = n_cmp = n_tie = n_exact = n_ranks = 0
    worst = 0.0
    for t in range(1, n_steps):
        x, kx, mask = ref.step(td)
        N = x.shape[1]
        lp64, klp = post_process(x, kx, mask, T, clip)
        s32 = score32.to(dev).double()
        cand = s32[:, None] + lp64  # the kernel's candidate fl(score + lp) is within the bound of it
        cbnd = C_BAR * U32 * klp + 2 * U32 * cand.abs()
        per = lambda v: v.view(W, B, N).permute(1, 0, 2).reshape(B, W * N)  # noqa: E731
        cb, bb = per(cand), per(cbnd)
        top, idx = cb.sort(dim=1, descending=True, stable=True)
        k = min(W + 1, W * N)
        top, idx = top[:, :k].cpu(), idx[:, :k].cpu()
        tb = bb.gather(1, idx.to(dev)).cpu()
        n_finite = torch.isfinite(cb).sum(1).cpu()
        xc, mc, sc = x.cpu(), mask.cpu(), score32
        par, a, l = pars[t], acts[t], lps[t]
        pw = par // B
        for b in range(B):
            n_all += 1
            rows_of = lambda f: int(f // N) * B + b  # noqa: E731
            # near[i]: sorted positions i, i + 1 are within their bounds of each other (their order is not decided by the
            # values); twin[i]: an exact tie of bitwise-identical inputs, which the tie rule orders by flat index.  Runs
            # joined by near pairs form groups; a group of twins only has an exact order, any other group only a set
            near, twin = [], []
            for i in range(k - 1):
                fin = bool(torch.isfinite(top[b, i]) and torch.isfinite(top[b, i + 1]))
                gap = float(top[b, i] - top[b, i + 1]) if fin else float("inf")
                f1, f2 = int(idx[b, i]), int(idx[b, i + 1])
                r1, r2 = rows_of(f1), rows_of(f2)
                twin.append(gap == 0 and f1 % N == f2 % N and sc[r1] == sc[r2] and torch.equal(xc[r1], xc[r2])
                            and torch.equal(mc[r1], mc[r2]))
                near.append(fin and gap <= float(tb[b, i] + tb[b, i + 1]))
            groups, lo = [], 0
            for i in range(k):
                if i == k - 1 or not near[i]:
                    groups.append((lo, i, all(twin[lo:i])))
                    lo = i + 1
            cut = [g for g in groups if g[0] < W <= g[1]]  # a group across the W-th / (W+1)-th cut
            if cut and not cut[0][2]:
                continue  # near-tied candidates of different inputs at the cut: the beam set is not decided
            n_cmp += 1
            rows = torch.arange(W) * B + b
            assert torch.equal(par[rows] % B, torch.full((W,), b)), (tag, t, b)
            got = pw[rows] * N + a[rows]
            nf = min(int(n_finite[b]), W)
            tie = False
            for g0, g1, exact in groups:  # ranks in a group of near-ties hold the same candidates
                if g0 >= nf:
                    break
                g1 = min(g1, nf - 1)
                if exact:
                    assert torch.equal(got[g0:g1 + 1], idx[b, g0:g1 + 1]), (tag, t, b, g0, g1)
                    tie |= g1 > g0
                    n_exact += 1
                else:
                    assert sorted(got[g0:g1 + 1].tolist()) == sorted(idx[b, g0:g1 + 1].tolist()), (tag, t, b, g0, g1)
                n_ranks += 1
            n_tie += tie
            assert (got[nf:] == got[0]).all(), (tag, t, b)  # fill-up: ranks from #finite upward copy rank 0
        # selected lp and scores, on every row
        pd, ad = par.to(dev), a.to(dev)
        sel64, selk = lp64[pd, ad], klp[pd, ad]
        r = ratios(l.to(dev), sel64, selk)
        worst = max(worst, float(r.max()))
        assert float(r.max()) <= C_BAR, (tag, t, float(r.max()))
        score32 = score32[par] + l
        score64 = score64[pd] + sel64
        serr = serr[pd] + C_BAR * U32 * selk + U32 * score64.abs()
        assert ((score32.to(dev).double() - score64).abs() <= serr).all(), (tag, t)
        s = score32.view(W, B)
        assert (s[1:] <= s[:-1]).all(), (tag, t)  # non-increasing by rank
        td = td[par]
        td["action"] = a
        td = oenv.step(td)["next"]
    assert bool(td["done"].all()), tag
    print(f"{tag}: {n_cmp} / {n_all} (step, instance) selections compared, {n_tie} with exact ties, "
          f"{n_exact} / {n_ranks} rank groups in exact order; worst lp ratio {worst:.3g}")
    assert n_cmp >= min_share * n_all, (tag, n_cmp, n_all)
    return n_tie


def check_tours(name, n, raw, acts, W):
    """Backtracked tours are feasible: every action allowed by the oracle env's mask along the tour, every tour done."""
    oenv = oenvs.make_env(name, n, check_solution=False)
    td = obatchify(oenv.reset(raw), W)
    acts = acts.cpu()
    for t in range(acts.shape[1]):
        a = acts[:, t]
        if t > 0:
            assert td["action_mask"].gather(1, a[:, None]).all(), t
        td["action"] = a
        td = oenv.step(td)["next"]
    assert bool(td["done"].all())
    if name != "rcvrptw":
        oenv.check_solution_validity(obatchify(oenv.reset(raw), W), acts)


def compare_with_per_step(rb, pol, env, raw, out, W, T, clip, tag, step_check=False, dup=False):
    """The per-step pipeline on the same inputs, step by step against the restated rule, then tour by tour against the
    fused result: equal tours have rewards within 1e-6 relative and log-likelihoods within 1e-4."""
    from rrnco_b200 import models
    td = env.reset(lite(rb, raw))
    cache = pol.decoder._precompute_cache(pol.encoder(td), num_starts=W)
    mp = pytest.MonkeyPatch()
    try:
        rec = record_beam_steps(mp)
        with torch.no_grad():
            ps = models.beam_search_rollout(pol.decoder, cache, env, td, W, temperature=T, tanh_clipping=clip)
    finally:
        mp.undo()
    if step_check:
        check_beam_steps(rec, W, f"{tag} per-step", temperature=T, clip=clip, min_share=0.5 if dup else 0.8)
    B = out["reward"].shape[0] // W
    fa, fr, fl = out["actions"].cpu(), out["reward"].cpu(), out["log_likelihood"].cpu()
    pa, pr, pl = ps["actions"].cpu(), ps["reward"].cpu(), ps["log_likelihood"].cpu()
    same_sets = matched = 0
    for b in range(B):
        rows = torch.arange(W) * B + b
        ptours = {tuple(pa[r].tolist()): r for r in rows.tolist()}
        ftours = [tuple(fa[r].tolist()) for r in rows.tolist()]
        same_sets += sorted(ftours) == sorted(ptours)
        for r, tour in zip(rows.tolist(), ftours):
            q = ptours.get(tour)
            if q is None:
                continue
            matched += 1
            assert abs(float(fr[r] - pr[q])) <= 1e-6 * max(1.0, abs(float(pr[q]))), (tag, b)
            assert abs(float(fl[r] - pl[q])) <= 1e-4, (tag, b)
    print(f"{tag}: identical beam sets with the per-step pipeline on {same_sets} / {B} instances, {matched} tours in both")


def beam_case(rb, name, N, W, T, clip, B=2, variant=""):
    seed = 31 + N + (W or 0)
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, seed, variant=variant)
    n = N if name == "atsp" else N - 1
    default = W is None
    if default:
        W = env.get_num_starts(env.reset(lite(rb, raw)))
    tag = f"{name}{' ' + variant if variant else ''} N={N} W={W}{' (default)' if default else ''} T={T} clip={clip}"
    out, steps = run_fused(rb, pol, env, env.reset(lite(rb, raw)), None if default else W, T, clip, select_best=False)
    assert out["actions"].shape[0] == W * B
    n_tie = check_fp64_walk(name, n, p, row, col, raw, W, steps, T, clip, tag)
    if W > n:  # duplicate beams: exact ties between bitwise-identical inputs must occur (and were compared)
        assert n_tie > 0, tag
    check_tours(name, n, raw, out["actions"], W)
    # the per-step pipeline's own step check on the shapes of test_beam_search_vs_restatement, which RRNetPolicy.forward
    # now sends to the fused kernel (check_beam_steps holds lp to 1e-5 absolute: the scale of T = 1, clip 10)
    step_check = (T, clip) == (1.0, 10.0) and N <= 100 and (default or W in (2, 8)) and not variant
    compare_with_per_step(rb, pol, env, raw, out, W, T, clip, tag, step_check=step_check, dup=W > n)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ENVS)
@pytest.mark.parametrize("N", [20, 50, 100, 112])
@pytest.mark.parametrize("W", [2, 8, 33, None, 128])
def test_fused_beam_against_fp64(rb, name, N, W):
    beam_case(rb, name, N, W, 1.0, 10.0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ENVS)
@pytest.mark.parametrize("T,clip", [(0.1, 10.0), (1.0, 0.0)])
@pytest.mark.parametrize("N,W", [(50, None), (112, 8)])
def test_fused_beam_temperature_and_clipping(rb, name, T, clip, N, W):
    beam_case(rb, name, N, W, T, clip)


@pytest.mark.gpu
@pytest.mark.parametrize("N,W", [(50, None), (100, 33)])
def test_fused_beam_rcvrptw_open_limits_backhauls(rb, N, W):
    beam_case(rb, "rcvrptw", N, W, 1.0, 10.0, variant="OLB")


@pytest.mark.gpu
def test_fused_beam_augmented_shared_instance_data(rb):
    """x8 augmentation with share_instance_data: 8 B instances over B rows of instance data (data_rows < R / W)."""
    name, n, B, W, aug = "rcvrp", 49, 2, 12, 8
    raw = synth.make_instances(name, B, n, seed=41)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = rb.StateAugmentation(num_augment=aug, share_instance_data=True)(env.reset(lite(rb, raw)))
    assert td["distance_matrix"].shape[0] == B and td["locs"].shape[0] == aug * B
    row, col = synth.random_embeddings(aug * B, n + 1, seed=42)
    p = omodel.init_decoder_params(name, seed=43)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row.to(dev), col.to(dev)

    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(p, strict=True)
    out, steps = run_fused(rb, pol, env, td, W, select_best=False)
    raw8 = obatchify(raw, aug)
    check_fp64_walk(name, n, p, row, col, raw8, W, steps, 1.0, 10.0, "rcvrp x8 shared N=50 W=12")
    check_tours(name, n, raw8, out["actions"], W)


@pytest.mark.gpu
def test_fused_beam_select_best_reproducible_and_bindings_agree(rb):
    from rrnco_b200 import torch_ops
    name, N, B, W = "rcvrp", 60, 3, 16
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, 7)
    runs = []
    for flag in (True, True, False):
        torch_ops.use_torch_ops(flag)
        try:
            runs.append(run_fused(rb, pol, env, env.reset(lite(rb, raw)), W, per_step_logprobs=True,
                                  select_best=False)[0])
        finally:
            torch_ops.use_torch_ops(True)
    for other in runs[1:]:  # run to run and torch op vs ctypes: bitwise
        for k in ("actions", "reward", "log_likelihood"):
            assert torch.equal(runs[0][k], other[k]), k
    full = run_fused(rb, pol, env, env.reset(lite(rb, raw)), W, select_best=False)[0]
    best = run_fused(rb, pol, env, env.reset(lite(rb, raw)), W)[0]
    rows = pick_best(full["reward"], W)  # first maximum of the reward over the beams
    assert best["actions"].shape[0] == B
    for k in ("actions", "reward", "log_likelihood"):
        assert torch.equal(best[k], full[k][rows]), k
    assert torch.equal(full["actions"], runs[0]["actions"]) and torch.equal(full["reward"], runs[0]["reward"])


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["nan_weight", "operand_overflow"])
def test_fused_beam_raises_like_the_rollout(rb, how):
    name, N, B, W = "rcvrp", 30, 2, 6
    raw, oenv, row, col, p, env, pol = setup_case(rb, name, N, B, 9)
    with torch.no_grad():
        if how == "nan_weight":
            pol.decoder.pointer.ffn.lins[1].weight[3, 5] = float("nan")
        else:
            pol.decoder.pointer.ffn.lins[0].weight.mul_(1.0e5)  # hidden activations ~1e5 >> the fp16 operand range
    with pytest.raises(AssertionError, match="Logits contain NaNs"):
        run_fused(rb, pol, env, env.reset(lite(rb, raw)), W)
