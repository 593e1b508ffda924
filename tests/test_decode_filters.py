"""Top-k / top-p (nucleus) logit filters in the decode kernels (rl4co process_logits, decoding.py:311-361).

The reference is the oracle's decoding (oracle.model) with the filters of rl4co's process_logits restated here
(`process_logits`, `oracle_filters`): the oracle itself has no filters.
CPU: that restatement against an independent sort-based restatement of rl4co's two helpers, the tie rule, argument checks
and the training guard.  GPU: select_action and the fused / per-step rollouts against the oracle.
Kept sets are compared on every row whose decision margin (k-th vs next value, nucleus mass vs top_p) exceeds 1e-4; the
other rows are counted and printed: there fp32 rounding may legitimately move the cut.
"""
import contextlib
import math

import numpy as np
import pytest
import torch

from oracle import envs as oenvs, model as omodel, synth

dev = "cuda"
EPS = 1e-4
FILTERS = [(10, 0.0), (0, 0.9), (20, 0.5), (3, 0.95), (400, 0.3)]


# ---------------------------------------------------------------------------------------------------
# fixtures / helpers
# ---------------------------------------------------------------------------------------------------
def rl4co_top_k(logits, top_k):
    """[rl4co-recalled] modify_logits_for_top_k_filtering (sort form), restated independently of process_logits below."""
    kth = logits.sort(dim=-1, descending=True)[0][..., top_k - 1: top_k]
    return torch.where(logits < kth, torch.full_like(logits, -math.inf), logits)


def rl4co_top_p(logits, top_p):
    """[rl4co-recalled] modify_logits_for_top_p_filtering: ascending sort, cumulative softmax, drop cum <= 1 - top_p."""
    s, idx = torch.sort(logits, descending=False)
    cum = s.softmax(dim=-1).cumsum(dim=-1)
    drop_sorted = cum <= (1 - top_p)
    drop = drop_sorted.scatter(1, idx, drop_sorted)
    return logits.masked_fill(drop, -math.inf)


def rl4co_process_logits(logits, mask, temperature, clip, top_k, top_p):
    v = torch.tanh(logits) * clip
    v = v.masked_fill(~mask, -math.inf) / temperature
    if top_k > 0:
        v = rl4co_top_k(v, min(top_k, v.size(-1)))
    if 0 < top_p < 1:
        v = rl4co_top_p(v, top_p)
    return torch.log_softmax(v, -1)


def top_p_groups(logits, top_p):
    """Top-p as the kernels define it: keep j iff the softmax mass of the entries strictly greater than v_j is < top_p.
    Without ties this is rl4co's rule (test_filters_match_rl4co_sort_form); a tie group is kept or dropped as a whole,
    where rl4co's result would depend on torch.sort's order among equal values (DESIGN.md §4.3b)."""
    s, idx = torch.sort(logits, dim=-1, descending=True)
    ps = s.softmax(dim=-1)
    before = ps.cumsum(dim=-1) - ps  # mass of the entries ahead of each one in the sorted row
    first = torch.searchsorted(-s.contiguous(), -s.contiguous(), side="left")  # first position of each tie group
    keep_sorted = before.gather(-1, first) < top_p
    keep = torch.empty_like(keep_sorted).scatter_(-1, idx, keep_sorted)
    return logits.masked_fill(~keep, -math.inf)


def process_logits(logits, mask, temperature=1.0, tanh_clipping=10.0, mask_logits=True, top_k=0, top_p=0.0):
    """oracle.model.process_logits (decoding.py:311-361) with the filters between the temperature and the log-softmax."""
    if tanh_clipping > 0:
        logits = torch.tanh(logits) * tanh_clipping
    if mask_logits:
        logits = logits.masked_fill(~mask, -math.inf)
    logits = logits / temperature
    if top_k > 0:  # rl4co modify_logits_for_top_k_filtering (topk form: ties with the k-th value are kept)
        kth = torch.topk(logits, min(top_k, logits.size(-1)), dim=-1)[0][..., -1, None]
        logits = logits.masked_fill(logits < kth, -math.inf)
    if 0 < top_p < 1:
        logits = top_p_groups(logits, top_p)
    return torch.log_softmax(logits, dim=-1)


@contextlib.contextmanager
def oracle_filters(top_k, top_p):
    """The oracle's decoding strategies (oracle.model.Strategy.step) with this file's filtered process_logits."""
    base = omodel.process_logits
    omodel.process_logits = lambda logits, mask, temperature=1.0, tanh_clipping=10.0, mask_logits=True: process_logits(
        logits, mask, temperature, tanh_clipping, mask_logits, top_k, top_p)
    try:
        yield
    finally:
        omodel.process_logits = base


def policy_forward(p, oenv, td, row, col, top_k=0, top_p=0.0, **kw):
    with oracle_filters(top_k, top_p):
        return omodel.policy_forward(p, oenv, td, row, col, **kw)


def processed(logits, mask, temperature=1.0, clip=10.0):
    v = torch.tanh(logits.double()) * clip if clip > 0 else logits.double()
    return v.masked_fill(~mask, -math.inf) / temperature


def kept_and_clear(v, top_k, top_p, eps=EPS):
    """fp64 kept set [R,N] of the filters on processed values v, and the rows whose decision margin exceeds eps."""
    R, N = v.shape
    clear = torch.ones(R, dtype=torch.bool)
    if 0 < top_k < N:
        s = v.sort(-1, descending=True)[0]
        kth, nxt = s[:, top_k - 1], s[:, top_k]
        gap = kth - nxt
        clear &= torch.isinf(kth) | ~(gap <= eps)
        v = v.masked_fill(v < kth[:, None], -math.inf)
    if 0 < top_p < 1:
        s, idx = torch.sort(v, -1, descending=True)
        ps = s.softmax(-1)
        before = ps.cumsum(-1) - ps
        first = torch.searchsorted(-s.contiguous(), -s.contiguous(), side="left")
        mass_gt = before.gather(-1, first)
        d = (mass_gt - top_p).abs().masked_fill(torch.isinf(s), math.inf)
        clear &= d.min(-1)[0] > eps
        keep_sorted = mass_gt < top_p  # a prefix of the sorted row
        # values within eps of each other at the cut may tie in fp32 (a tie group is kept whole) but not in fp64
        nk = keep_sorted.sum(-1, keepdim=True)
        last, nxt = s.gather(-1, nk - 1)[:, 0], s.gather(-1, nk.clamp(max=N - 1))[:, 0]
        clear &= (nk[:, 0] == N) | torch.isinf(nxt) | (last - nxt > eps)
        v = v.masked_fill(~torch.empty_like(keep_sorted).scatter_(-1, idx, keep_sorted), -math.inf)
    return torch.isfinite(v), clear


def random_rows(seed, R=257, N=333, p_feas=0.4):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(R, N, generator=g) * 3
    mask = torch.rand(R, N, generator=g) < p_feas
    mask[:, 0] = True
    return logits, mask, g


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("top_k,top_p,temperature", [(5, 0.0, 1.0), (0, 0.8, 1.0), (7, 0.6, 0.7), (50, 0.9, 2.0),
                                                     (1000, 0.0, 1.0), (0, 1.0, 1.0), (3, 0.3, 1.0), (1, 0.5, 1.0),
                                                     (12, 0.99, 0.5)])
def test_filters_match_rl4co_sort_form(top_k, top_p, temperature):
    g = torch.Generator().manual_seed(top_k * 31 + int(top_p * 100))
    R, N = 64, 57
    logits = torch.randn(R, N, generator=g, dtype=torch.float64) * 2  # fp64: no ties, no cumulative rounding at the cut
    mask = torch.rand(R, N, generator=g) < 0.6
    mask[:, 0] = True
    mask[:8] = False
    mask[:8, :3] = True  # rows with fewer feasible nodes than top_k
    want = rl4co_process_logits(logits, mask, temperature, 10.0, top_k, top_p)
    got = process_logits(logits.clone(), mask, temperature, 10.0, top_k=top_k, top_p=top_p)
    assert torch.equal(torch.isfinite(got), torch.isfinite(want))
    fin = torch.isfinite(want)
    assert (got[fin] - want[fin]).abs().max() < 1e-12
    # without a filter the restatement is exactly the oracle's process_logits
    assert torch.equal(process_logits(logits.clone(), mask, temperature, 10.0),
                       omodel.process_logits(logits.clone(), mask, temperature, 10.0))


def test_tie_groups_are_kept_or_dropped_whole():
    """Saturated tanh clipping ties entries at +-clip: a tie group is kept or dropped as a whole."""
    big = 50.0  # tanh(50) == 1 in fp32 and fp64: clip exactly
    row = torch.tensor([[big, big, big, 0.0, -1.0, -big]])
    mask = torch.ones_like(row, dtype=torch.bool)
    # top-k = 2 cuts inside the tie group of three: ties with the k-th value are kept
    lp = process_logits(row.clone(), mask, top_k=2)
    assert torch.isfinite(lp[0, :3]).all() and torch.isinf(lp[0, 3:]).all()
    # top-p: the group of three holds ~all the mass; p = 0.5 < its mass keeps all three (mass strictly above each is 0)
    lp = process_logits(row.clone(), mask, top_p=0.5)
    assert torch.isfinite(lp[0, :3]).all() and torch.isinf(lp[0, 3:]).all()
    assert torch.allclose(lp[0, :3].exp(), torch.full((3,), 1 / 3, dtype=lp.dtype))
    # two equal entries below the top: the pair goes together
    row2 = torch.tensor([[2.0, 1.0, 1.0, 0.5]])
    v = torch.tanh(row2) * 10
    pr = v.softmax(-1)[0]
    m2 = torch.ones_like(row2, dtype=torch.bool)
    for p, n_keep in ((float(pr[0]) * 0.999, 1), (float(pr[0]) * 1.001, 3), (float(pr[0] + 2 * pr[1]) * 1.001, 4)):
        lp = process_logits(row2.clone(), m2, top_p=p)
        assert int(torch.isfinite(lp).sum()) == n_keep, (p, lp)
    # the fp64 helper of the GPU tests agrees with the same rule
    kept, _ = kept_and_clear(processed(row2, m2), 0, float(pr[0]) * 1.001)
    assert kept.sum() == 3


@pytest.mark.parametrize("bad", [dict(top_k=-1), dict(top_p=-0.1), dict(top_p=1.5), dict(top_p=float("nan")),
                                 dict(top_k=2.5)])
def test_bad_filter_values_raise_before_launch(bad):
    import rrnco_b200
    from rrnco_b200.models import filter_args
    with pytest.raises(ValueError):
        filter_args(bad.get("top_k"), bad.get("top_p"))
    # CPU tensors: nothing could be launched, and the check comes first
    with pytest.raises(ValueError):
        rrnco_b200.select_action(torch.zeros(2, 3), torch.ones(2, 3, dtype=torch.bool), "greedy", **bad)


def test_c_abi_rejects_bad_filters_before_any_cuda_call():
    import ctypes
    from rrnco_b200 import _lib
    from rrnco_b200.build import build_library
    build_library()
    h = _lib.lib()
    sel = lambda k, p: h.rrnco_select_action_filtered(0, 4, None, None, 0, 10.0, 1.0, 0, 0, None, None, None, None, k, p,
                                                       None)
    assert sel(0, 0.0) == 0 and sel(5, 0.9) == 0  # zero rollouts: valid filters do nothing
    for k, p in ((-1, 0.0), (0, -0.5), (0, 1.01), (0, float("nan")), (3, float("inf"))):
        assert sel(k, p) == -1, (k, p)
    w, c, d = _lib.DecoderWeights(), _lib.DecoderCache(), _lib.InstanceData()
    args = lambda k, p: (1, 20, 1, 1, 0, 0, 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(d), None, 0, 1, None, None,
                         None, None, None, None, None, None, k, p, None)
    assert h.rrnco_rollout_filtered(*args(-2, 0.0)) == -1
    assert h.rrnco_rollout_filtered(*args(0, float("nan"))) == -1


def test_filtered_training_call_raises():
    import rrnco_b200

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            raise AssertionError("not reached")
    pol = rrnco_b200.RRNetPolicy(encoder=Enc(), env_name="rcvrp")
    with torch.enable_grad():
        for kw in (dict(top_k=5), dict(top_p=0.9)):
            with pytest.raises(NotImplementedError, match="replay"):
                pol(None, object(), phase="train", **kw)


# ---------------------------------------------------------------------------------------------------
# GPU: select_action
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rb():
    import rrnco_b200
    rrnco_b200.set_precision(3)
    return rrnco_b200


@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p", FILTERS)
@pytest.mark.parametrize("temperature", [1.0, 0.6])
def test_select_action_filters_vs_oracle(rb, top_k, top_p, temperature):
    logits, mask, g = random_rows(3)
    R, N = logits.shape
    kept, clear = kept_and_clear(processed(logits, mask, temperature), top_k, top_p)
    print(f"rows within {EPS} of the cut: {int((~clear).sum())} / {R}")
    logp = process_logits(logits.clone(), mask, temperature, top_k=top_k, top_p=top_p)
    L, M = logits.to(dev), mask.to(dev)
    kw = dict(temperature=temperature, top_k=top_k, top_p=top_p)
    # greedy: same action as unfiltered; log-prob renormalised over the kept set
    a0, _, _ = rb.select_action(L, M, "greedy", temperature=temperature)
    a, lp, st = rb.select_action(L, M, "greedy", **kw)
    assert torch.equal(a, a0) and int(st.item()) == 0
    want = logp.gather(1, a.cpu()[:, None]).squeeze(1)
    assert (lp.cpu() - want)[clear].abs().max() < 1e-5
    # evaluate: a feasible forced action that is filtered out gets -inf and is not reported as infeasible
    forced = torch.multinomial(mask.float(), 1, generator=g).squeeze(1)
    a2, lp2, st2 = rb.select_action(L, M, "evaluate", forced_action=forced.to(dev), **kw)
    assert torch.equal(a2.cpu(), forced) and int(st2.item()) == 0
    fk = kept.gather(1, forced[:, None]).squeeze(1)
    lp2, want2 = lp2.cpu(), logp.gather(1, forced[:, None]).squeeze(1)
    assert torch.equal(torch.isfinite(lp2)[clear], fk[clear])
    both = clear & fk
    assert (lp2 - want2)[both].abs().max() < 1e-5
    if top_k > 0 and top_k < int(mask.sum(1).min()):
        assert (~fk).any()  # the case is exercised
    # sampling: the filtered draw equals the unfiltered one whenever that one is kept, and is always in the kept set
    n_changed = 0
    for seed in range(4):
        for step in (0, 7):
            s0, _, _ = rb.select_action(L, M, "sampling", seed=seed, step=step, temperature=temperature)
            s1, _, st3 = rb.select_action(L, M, "sampling", seed=seed, step=step, **kw)
            s0, s1 = s0.cpu(), s1.cpu()
            assert int(st3.item()) == 0
            k0 = kept.gather(1, s0[:, None]).squeeze(1)
            assert torch.equal(s1[clear & k0], s0[clear & k0])
            assert kept.gather(1, s1[:, None]).squeeze(1)[clear].all()
            n_changed += int((s1 != s0).sum())
    if top_k > 0 or top_p < 0.95:
        assert n_changed > 0


@pytest.mark.gpu
def test_select_action_keep_everything_is_bitwise_unfiltered(rb):
    logits, mask, g = random_rows(5)
    L, M = logits.to(dev), mask.to(dev)
    forced = torch.multinomial(mask.float(), 1, generator=g).squeeze(1).to(dev)
    for kind in ("greedy", "sampling", "evaluate"):
        f = forced if kind == "evaluate" else None
        a0, l0, _ = rb.select_action(L, M, kind, seed=9, step=3, forced_action=f)
        for kw in (dict(top_k=logits.shape[1]), dict(top_k=10**6), dict(top_p=1.0)):
            a1, l1, _ = rb.select_action(L, M, kind, seed=9, step=3, forced_action=f, **kw)
            assert torch.equal(a0, a1) and torch.equal(l0, l1), (kind, kw)


@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p", [(4, 0.0), (0, 0.7), (6, 0.8)])
def test_select_action_filtered_distribution_chi_square(rb, top_k, top_p):
    """One row's filtered draw over many rollout ids and seeds follows the oracle's filtered softmax (5 sigma)."""
    g = torch.Generator().manual_seed(11)
    N, R = 40, 4000
    row = torch.randn(1, N, generator=g) * 0.03  # clipped values within about +-1: many entries carry mass
    mask = torch.rand(1, N, generator=g) < 0.8
    mask[0, 0] = True
    probs = process_logits(row.double().clone(), mask, top_k=top_k, top_p=top_p).exp()[0]
    counts = torch.zeros(N, dtype=torch.float64)
    L, M = row.expand(R, N).contiguous().to(dev), mask.expand(R, N).contiguous().to(dev)
    for seed in range(3):
        a, _, _ = rb.select_action(L, M, "sampling", seed=100 + seed, step=seed, top_k=top_k, top_p=top_p)
        counts += torch.bincount(a.cpu(), minlength=N).double()
    assert (counts[probs == 0] == 0).all()
    exp = probs * 3 * R
    keep = exp > 5
    chi2 = (((counts - exp) ** 2) / exp.clamp_min(1e-9))[keep].sum().item()
    dof = int(keep.sum()) - 1
    assert dof >= 2 and chi2 < dof + 5 * (2 * dof) ** 0.5 + 5, (chi2, dof)


# ---------------------------------------------------------------------------------------------------
# GPU: rollouts
# ---------------------------------------------------------------------------------------------------
def lite(rb, td):
    return rb.TensorDictLite({k: v.to(dev) for k, v in td.items()}, batch_size=list(td.batch_size))


def make_policy(rb, name, p, row, col):
    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col
    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(p, strict=True)
    return pol


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
    """The kernels' Gumbel noise of (rollout r, step, column c) = Philox(seed; (r, step, c >> 2))[c & 3]."""
    def noise(step_idx, shape):
        step = step_idx - 1  # the strategy has already stored the forced start
        R = S * n_inst
        r = np.repeat(np.arange(R), N)
        c = np.tile(np.arange(N), R)
        x = philox4x32(r & 0xFFFFFFFF, r >> 32, np.full(R * N, step), c >> 2, seed & 0xFFFFFFFF, seed >> 32)
        x = np.stack(x, 0)[c & 3, np.arange(R * N)]
        u = ((x >> np.uint64(9)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 8388608.0)
        return torch.from_numpy((-np.log(-np.log(u))).astype(np.float32).reshape(R, N))
    return noise


def step_clear(trace, top_k, top_p):
    """[R, T] decisions of the oracle's trace whose filter margin exceeds EPS (forced start column: clear)."""
    cols = [torch.ones(trace[0]["mask"].shape[0], dtype=torch.bool)]
    for t in trace:
        cols.append(kept_and_clear(processed(t["logits"], t["mask"]), top_k, top_p)[1])
    return torch.stack(cols, 1)


def setup(rb, name, N, B, seed):
    n = N if name == "atsp" else N - 1
    raw = synth.make_instances(name, B, n, seed=seed)
    oenv = oenvs.make_env(name, n, check_solution=False)
    S = oenv.get_num_starts(oenv.reset(raw))
    row, col = synth.random_embeddings(B, N, seed=seed + 1)
    p = omodel.init_decoder_params(name, seed=seed + 2)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    pol = make_policy(rb, name, p, row.to(dev), col.to(dev))
    return raw, oenv, S, row, col, p, env, pol


ROLLOUT_CASES = [(name, N) for N in (20, 101, 112, 128) for name in ("atsp", "rcvrp", "rcvrptw")]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N", ROLLOUT_CASES)
@pytest.mark.parametrize("top_k,top_p", [(5, 0.0), (0, 0.85), (8, 0.7)])
def test_fused_rollout_filters_vs_oracle(rb, name, N, top_k, top_p):
    B, seed = 2, 31
    raw, oenv, S, row, col, p, env, pol = setup(rb, name, N, B, N + B)
    fk = dict(top_k=top_k, top_p=top_p)
    # multistart sampling against the oracle's Gumbel twin with the same filters
    trace = []
    oout = policy_forward(p, oenv, oenv.reset(raw), row, col, decode_type="multistart_sampling", num_starts=S,
                                 gumbel_noise=gumbel_twin(seed, B, S, N), trace=trace, **fk)
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_sampling", num_starts=S, seed=seed,
                  return_sum_log_likelihood=False, **fk)
    T = min(out["actions"].shape[1], oout["actions"].shape[1])
    same = (out["actions"].cpu()[:, :T] == oout["actions"][:, :T]).all(1)
    clear = step_clear(trace, top_k, top_p)
    print(f"{name} N={N} {fk}: identical tours {same.float().mean():.4f}, decisions within {EPS} of the cut "
          f"{int((~clear).sum())} / {clear.numel()}")
    assert same.float().mean() >= 0.97, same.float().mean()
    env.check_solution_validity(rb.batchify(env.reset(lite(rb, raw)), S), out["actions"]) if name != "rcvrptw" else None
    # evaluate mode on the oracle's filtered tours: per-step log-probs (renormalised over the kept set)
    forced = oout["actions"][:, 1:]
    trace_e = []
    oev = policy_forward(p, oenv, oenv.reset(raw), row, col, num_starts=S, actions=forced, trace=trace_e, **fk)
    with torch.no_grad():
        ev = pol(env.reset(lite(rb, raw)), env, phase="train", num_starts=S, actions=forced.to(dev),
                 return_sum_log_likelihood=False, **fk)
    assert torch.equal(ev["actions"].cpu(), oout["actions"])
    lp, olp = ev["log_likelihood"].cpu(), oev["logprobs"]
    ce = step_clear(trace_e, top_k, top_p)[:, : lp.shape[1]]
    assert torch.equal(torch.isfinite(lp)[ce], torch.isfinite(olp)[ce])
    fin = ce & torch.isfinite(olp)
    assert (lp - olp)[fin].abs().max() < 1e-4
    # a filter that keeps everything runs the filtered kernel and gives the unfiltered results bit for bit
    for kind in ("multistart_greedy", "multistart_sampling"):
        with torch.no_grad():
            a = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type=kind, num_starts=S, seed=seed,
                    return_sum_log_likelihood=False)
            b = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type=kind, num_starts=S, seed=seed,
                    return_sum_log_likelihood=False, top_k=N)
        for k in ("actions", "log_likelihood", "reward"):
            assert torch.equal(a[k], b[k]), (kind, k)


@pytest.mark.gpu
def test_filters_on_the_one_cta_engine_match_the_lean_engine(rb):
    """N <= 112 under rrnco_set_ffn_engine(1): the one-CTA tcgen05 engine's filtered select gives the lean engine's tours."""
    from rrnco_b200 import _lib
    name, N, B, seed = "rcvrp", 60, 3, 5
    raw, oenv, S, row, col, p, env, pol = setup(rb, name, N, B, 77)
    outs = []
    try:
        for engine in (2, 1):
            _lib.check(_lib.lib().rrnco_set_ffn_engine(engine))
            with torch.no_grad():
                outs.append(pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_sampling",
                                num_starts=S, seed=seed, top_k=6, top_p=0.8))
    finally:
        _lib.check(_lib.lib().rrnco_set_ffn_engine(2))
    T = min(outs[0]["actions"].shape[1], outs[1]["actions"].shape[1])
    same = (outs[0]["actions"][:, :T] == outs[1]["actions"][:, :T]).all(1)
    assert same.float().mean() >= 0.97


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["atsp", "rcvrp"])
def test_filtered_large_n_runs_stepwise_and_matches_oracle(rb, name, monkeypatch):
    """N = 200 with a filter decodes through the per-step pipeline, never the key-tiled fused kernel."""
    from rrnco_b200 import models

    def no_fused(*a, **k):
        raise AssertionError("the key-tiled fused kernel was launched for a filtered call")
    monkeypatch.setattr(models, "fused_rollout", no_fused)
    N, B, seed = 200, 2, 13
    raw, oenv, S, row, col, p, env, pol = setup(rb, name, N, B, 41)
    S = 16
    fk = dict(top_k=7, top_p=0.8)
    trace = []
    oout = policy_forward(p, oenv, oenv.reset(raw), row, col, decode_type="multistart_sampling", num_starts=S,
                                 gumbel_noise=gumbel_twin(seed, B, S, N), trace=trace, **fk)
    with torch.no_grad():
        out = pol(env.reset(lite(rb, raw)), env, phase="val", decode_type="multistart_sampling", num_starts=S, seed=seed,
                  **fk)
    T = min(out["actions"].shape[1], oout["actions"].shape[1])
    same = (out["actions"].cpu()[:, :T] == oout["actions"][:, :T]).all(1)
    clear = step_clear(trace, *fk.values())
    print(f"{name} N=200: identical tours {same.float().mean():.4f}, decisions within {EPS} of the cut "
          f"{int((~clear).sum())} / {clear.numel()}")
    assert same.float().mean() >= 0.97
    forced = oout["actions"][:, 1:]
    trace_e = []
    oev = policy_forward(p, oenv, oenv.reset(raw), row, col, num_starts=S, actions=forced, trace=trace_e, **fk)
    with torch.no_grad():
        ev = pol(env.reset(lite(rb, raw)), env, phase="train", num_starts=S, actions=forced.to(dev),
                 return_sum_log_likelihood=False, **fk)
    lp, olp = ev["log_likelihood"].cpu(), oev["logprobs"]
    ce = step_clear(trace_e, *fk.values())[:, : lp.shape[1]]
    assert torch.equal(torch.isfinite(lp)[ce], torch.isfinite(olp)[ce])
    fin = ce & torch.isfinite(olp)
    assert (lp - olp)[fin].abs().max() < 1e-4
