"""Training replay of instances of more than 102 nodes, up to 1024: the key-tiled attention kernels (rrnco_train_attention_tiled_*),
the key-tiled pointer-score kernels (rrnco_train_inst_tiled_*) and the wide logits tail, each against fp64 torch; the fused replay
against its plain-torch form and the sampling kernel on sampled rollouts; RRNetPolicy training end to end at n = 200 and n = 1000.
Relative errors are taken against the largest magnitude of each tensor, at the bars of tests/test_train_ops.py."""
import types

import pytest
import torch
import torch.nn.functional as F


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300)).item()


def test_replay_form_choice():
    """Kernels for CUDA fp32 replays with N <= 1024; the plain-torch form for CPU tensors, REPLAY_IMPL = "aten" and N > 1024."""
    from rrnco_b200 import training, train_ops
    assert train_ops.MAX_NODES_REPLAY == 1024
    cuda_like = types.SimpleNamespace(is_cuda=True, dtype=torch.float32)
    assert training.uses_replay_kernels(cuda_like, 101)
    assert training.uses_replay_kernels(cuda_like, 1000)
    assert training.uses_replay_kernels(cuda_like, 1024)
    assert not training.uses_replay_kernels(cuda_like, 1025)
    assert not training.uses_replay_kernels(torch.zeros(1, 200, 128), 200)
    assert not training.uses_replay_kernels(types.SimpleNamespace(is_cuda=True, dtype=torch.float64), 200)
    training.REPLAY_IMPL = "aten"
    try:
        assert not training.uses_replay_kernels(cuda_like, 200)
    finally:
        training.REPLAY_IMPL = "fused"


def _attention_ref(q, k, v, mask):
    qh, kh, vh = (t.unflatten(-1, (8, 16)).transpose(1, 2) for t in (q, k, v))
    sc = torch.matmul(qh, kh.transpose(-1, -2)) / 4.0
    sc = sc.masked_fill(~mask.unsqueeze(1), float("-inf"))
    return torch.matmul(torch.softmax(sc, -1), vh).transpose(1, 2).flatten(-2) + q


def _attention_case(n_inst, L, N, qscale, dev):
    g = torch.Generator().manual_seed(L + N)
    q = torch.randn(n_inst, L, 128, generator=g) * qscale
    k = torch.randn(n_inst, N, 128, generator=g)
    v = torch.randn(n_inst, N, 128, generator=g)
    mask = torch.rand(n_inst, L, N, generator=g) < 0.4
    mask[..., 0] |= ~mask.any(-1)
    mask[0, 0] = False
    mask[0, 0, N - 1] = True                      # the only feasible key is in the last (ragged) tile
    mask[0, 1, :64] = False                       # two whole key tiles masked
    mask[0, 1, N - 1] = True
    # instance 0: scores grow along the keys, so the running maximum moves from tile to tile
    k[0] += 0.5 * (torch.arange(N, dtype=torch.float32) / N)[:, None] * q[0, 2][None, :] / qscale ** 2   # up to ~16 nats
    mask[0, 2] = True
    r = torch.randn(n_inst, L, 128, generator=g) * 1e-6
    return [t.to(dev) for t in (q, k, v, mask, r)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_inst,L,N,qscale", [(2, 300, 103, 1.0), (3, 257, 129, 1.0), (1, 600, 200, 8.0), (2, 128, 513, 1.0),
                                               (1, 200, 1000, 3.0)])
def test_tiled_attention_forward_backward(n_inst, L, N, qscale):
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    q, k, v, mask, r = _attention_case(n_inst, L, N, qscale, dev)
    q, k, v = (t.requires_grad_(True) for t in (q, k, v))
    out = train_ops.fused_attention(q, k, v, mask)
    (out * r).sum().backward()
    got = [out.detach(), q.grad, k.grad, v.grad]
    qd, kd, vd = (t.detach().double().requires_grad_(True) for t in (q, k, v))
    od = _attention_ref(qd, kd, vd, mask)
    (od * r.double()).sum().backward()
    want = [od.detach(), qd.grad, kd.grad, vd.grad]
    for name, a, b in zip(("out", "dq", "dk", "dv"), got, want):
        assert _rel(a, b) < 5e-6, (name, _rel(a, b))
    # no float atomics: a second backward gives the same bits
    q2, k2, v2 = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
    (train_ops.fused_attention(q2, k2, v2, mask) * r).sum().backward()
    assert torch.equal(q2.grad, q.grad) and torch.equal(k2.grad, k.grad) and torch.equal(v2.grad, v.grad)


@pytest.mark.gpu
def test_tiled_kernels_agree_with_single_tile_kernels_at_101(monkeypatch):
    """At N = 101 both forms accept the input: the key-tiled kernels agree with the single-tile ones at the fp64 bars."""
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    n_inst, L, N = 3, 333, 101
    q, k, v, mask, r = _attention_case(n_inst, L, N, 1.0, dev)
    gen = torch.Generator().manual_seed(5)
    lk = torch.randn(n_inst, N, 128, generator=gen).to(dev)
    dist = torch.rand(n_inst, N, N, generator=gen).to(dev)
    cur = torch.randint(0, N, (n_inst, L), generator=gen).to(dev)
    act = torch.randint(0, N, (n_inst, L), generator=gen).to(dev)
    pmask = mask.clone()
    pmask.scatter_(-1, act.unsqueeze(-1), True)
    rl = (torch.randn(n_inst, L, generator=gen) * 1e-5).to(dev)
    res = {}
    for form in ("single", "tiled"):
        if form == "tiled":
            monkeypatch.setattr(train_ops, "MAX_NODES_ATTENTION", 0)
            monkeypatch.setattr(train_ops, "MAX_NODES_POINTER", 0)
        qq, kk, vv, ll = (t.detach().clone().requires_grad_(True) for t in (q, k, v, lk))
        alpha = torch.tensor([0.9], device=dev, requires_grad=True)
        out = train_ops.fused_attention(qq, kk, vv, mask)
        logp = train_ops.pointer_logprob(out, ll, alpha, None, dist, None, cur, pmask, act, 10.0, 1.0)
        ((out * r).sum() + (logp * rl).sum()).backward()
        res[form] = [out.detach(), logp.detach(), qq.grad, kk.grad, vv.grad, ll.grad, alpha.grad]
    train_ops.check_status(dev)
    for name, a, b in zip(("out", "logp", "dq", "dk", "dv", "dlk", "dalpha"), res["tiled"], res["single"]):
        assert _rel(a, b) < 5e-6, (name, _rel(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("n_inst,L,N,gscale", [(3, 300, 129, 1.0), (2, 1000, 256, 1e-7), (2, 257, 1000, 1.0)])
def test_tiled_pointer_scores_forward_backward(n_inst, L, N, gscale):
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(L + N)
    g = (torch.randn(n_inst, L, 128, generator=gen) * 3).to(dev).requires_grad_(True)
    lk = torch.randn(n_inst, N, 128, generator=gen).to(dev).requires_grad_(True)
    r = (torch.randn(n_inst, L, N, generator=gen) * gscale).to(dev)
    r = r * torch.logspace(0, -3, L, device=dev)[None, :, None]
    z = train_ops.pointer_scores(g, lk)
    ldz = 128 * ((N + 127) // 128)
    assert z.shape == (n_inst, L, ldz) and (z[..., N:] == 0).all()
    (z[..., :N] * r).sum().backward()
    gd, ld = g.detach().double().requires_grad_(True), lk.detach().double().requires_grad_(True)
    zd = torch.bmm(gd, ld.transpose(1, 2))
    (zd * r.double()).sum().backward()
    train_ops.check_status(dev)
    assert _rel(z[..., :N].detach(), zd.detach()) < 2e-6
    assert _rel(g.grad, gd.grad) < 5e-6
    assert _rel(lk.grad, ld.grad) < 5e-6


def _tail_ref(z, alpha, beta, dist, dur, cur, mask, act, clip, temp):
    inst = torch.arange(z.shape[0], device=z.device)
    logits = z / 128 ** 0.5
    bias = alpha * dist[inst[:, None], cur]
    if dur is not None:
        bias = bias + beta * dur[inst[:, None], cur]
    logits = torch.log(torch.exp(logits - bias) + 1e-6)
    if clip > 0:
        logits = torch.tanh(logits) * clip
    logits = logits.masked_fill(~mask, float("-inf")) / temp
    return F.log_softmax(logits, -1).gather(-1, act.unsqueeze(-1)).squeeze(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("with_dur,clip,temp,N", [(False, 10.0, 1.0, 129), (True, 10.0, 0.7, 129), (False, 0.0, 0.7, 1000),
                                                  (True, 10.0, 1.0, 1000), (True, 0.0, 1.0, 1000)])
def test_wide_logits_tail_forward_backward(with_dur, clip, temp, N):
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    n_inst, L = 3, 257
    g = torch.Generator().manual_seed(N)
    z = (torch.randn(n_inst, L, N, generator=g) * 30).to(dev).requires_grad_(True)
    dist = torch.rand(n_inst, N, N, generator=g).to(dev)
    dur = torch.rand(n_inst, N, N, generator=g).to(dev) if with_dur else None
    alpha = torch.tensor([1.3], device=dev, requires_grad=True)
    beta = torch.tensor([0.6], device=dev, requires_grad=True) if with_dur else None
    cur = torch.randint(0, N, (n_inst, L), generator=g).to(dev)
    mask = (torch.rand(n_inst, L, N, generator=g) < 0.5).to(dev)
    act = torch.randint(0, N, (n_inst, L), generator=g).to(dev)
    mask.scatter_(-1, act.unsqueeze(-1), True)
    r = torch.randn(n_inst, L, generator=g).to(dev)
    zd = z.detach().double().requires_grad_(True)
    ad = alpha.detach().double().requires_grad_(True)
    bd = beta.detach().double().requires_grad_(True) if with_dur else None
    want = _tail_ref(zd, ad, bd, dist.double(), dur.double() if with_dur else None, cur, mask, act, clip, temp)
    (want * r.double()).sum().backward()
    logp = train_ops.fused_logits_tail(z * 1.0, alpha, beta, dist, dur, cur, mask, act, clip, temp)  # z * 1.0: consumed in place
    (logp * r).sum().backward()
    assert (logp.detach().double() - want.detach()).abs().max().item() < 2e-5
    assert _rel(z.grad, zd.grad) < 2e-5
    assert abs(alpha.grad.item() - ad.grad.item()) < 2e-4 * max(1.0, abs(ad.grad.item()))
    if with_dur:
        assert abs(beta.grad.item() - bd.grad.item()) < 2e-4 * max(1.0, abs(bd.grad.item()))


@pytest.mark.gpu
@pytest.mark.parametrize("with_dur,N", [(True, 200), (False, 1000)])
def test_tiled_pointer_logprob_forward_backward(with_dur, N):
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    n_inst, L = 3, 391
    gen = torch.Generator().manual_seed(N)
    g = (torch.randn(n_inst, L, 128, generator=gen) * 2).to(dev).requires_grad_(True)
    lk = (torch.randn(n_inst, N, 128, generator=gen) * 1.5).to(dev).requires_grad_(True)
    dist = torch.rand(n_inst, N, N, generator=gen).to(dev)
    dur = torch.rand(n_inst, N, N, generator=gen).to(dev) if with_dur else None
    alpha = torch.tensor([0.9], device=dev, requires_grad=True)
    beta = torch.tensor([1.2], device=dev, requires_grad=True) if with_dur else None
    cur = torch.randint(0, N, (n_inst, L), generator=gen).to(dev)
    mask = (torch.rand(n_inst, L, N, generator=gen) < 0.5).to(dev)
    act = torch.randint(0, N, (n_inst, L), generator=gen).to(dev)
    mask.scatter_(-1, act.unsqueeze(-1), True)
    r = (torch.randn(n_inst, L, generator=gen) * 1e-5).to(dev) * torch.logspace(0, -3, L, device=dev)[None]
    logp = train_ops.pointer_logprob(g, lk, alpha, beta, dist, dur, cur, mask, act, 10.0, 1.0)
    (logp * r).sum().backward()
    gd, ld = g.detach().double().requires_grad_(True), lk.detach().double().requires_grad_(True)
    ad = alpha.detach().double().requires_grad_(True)
    bd = beta.detach().double().requires_grad_(True) if with_dur else None
    want = _tail_ref(torch.bmm(gd, ld.transpose(1, 2)), ad, bd, dist.double(), dur.double() if with_dur else None, cur, mask, act,
                     10.0, 1.0)
    (want * r.double()).sum().backward()
    train_ops.check_status(dev)
    assert (logp.detach().double() - want.detach()).abs().max().item() < 5e-5
    assert _rel(g.grad, gd.grad) < 2e-5 and _rel(lk.grad, ld.grad) < 2e-5
    assert abs(alpha.grad.item() - ad.grad.item()) < 2e-4 * max(1e-6, abs(ad.grad.item())) + 1e-12
    if with_dur:
        assert abs(beta.grad.item() - bd.grad.item()) < 2e-4 * max(1e-6, abs(bd.grad.item())) + 1e-12


@pytest.mark.gpu
def test_tiled_pointer_operand_overflow_sets_status():
    """A logit key past the fp16 operand range sets the sticky status word (no device fault): check_status raises."""
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    train_ops.status_word(dev).zero_()
    gen = torch.Generator().manual_seed(3)
    g = torch.randn(2, 100, 128, generator=gen).to(dev)
    lk = torch.randn(2, 300, 128, generator=gen).to(dev)
    lk[1, 250, 7] = 1e6
    z = train_ops.pointer_scores(g, lk)
    torch.cuda.synchronize()
    assert z.shape == (2, 100, 384)
    with pytest.raises(FloatingPointError):
        train_ops.check_status(dev)
    train_ops.check_status(dev)   # the word was cleared


def _policy(name, B, n, dev, seed):
    import rrnco_b200 as rb
    from oracle import synth, model as omodel
    raw = synth.make_instances(name, B, n, seed=seed)
    env = rb.get_env(name, generator_params={"num_loc": n}, check_solution=False)
    td = env.reset(rb.TensorDictLite({k: v.to(dev) for k, v in raw.items()}, batch_size=[B]))
    N = td["action_mask"].shape[-1]
    row, col = synth.random_embeddings(B, N, seed=seed + 1)
    row, col = row.to(dev).requires_grad_(True), col.to(dev).requires_grad_(True)

    class Enc(torch.nn.Module):
        def forward(self, td, phase=None):
            return row, col

    pol = rb.RRNetPolicy(encoder=Enc(), env_name=name).to(dev)
    pol.decoder.load_state_dict(omodel.init_decoder_params(name, seed=seed + 2))
    return env, td, pol, row, col


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,B,S", [("rcvrp", 150, 3, 8), ("atsp", 200, 2, 8), ("rcvrptw", 130, 3, 8)])
def test_tiled_replay_matches_aten_replay(name, n, B, S):
    """training.batched_logprobs above 102 nodes on sampled rollouts: the kernels vs the plain-torch form (per-step log-probs), the
    summed log-likelihood vs the sampling kernel's own, and the gradients of the REINFORCE loss against an fp64 plain-torch replay:
    within 1e-4 of the tensor's maximum of the fp64 value, or no further from it than twice the fp32 plain-torch replay is.  Not for
    the tensors behind relu' of the FFN: a hidden unit within rounding of zero takes relu' from each form's own forward (see
    test_fused_replay_matches_aten_replay; at rcvrptw n = 130 unit 445 of one row does so, and carries all but 3e-7 of the squared
    error of dW1), so there the bound is 5e-2, and db1 may differ from fp64 in at most that one unit."""
    import copy
    import rrnco_b200 as rb
    from rrnco_b200 import training, train_ops
    dev = torch.device("cuda", 0)
    env, td, pol, row, col = _policy(name, B, n, dev, seed=11)
    with torch.no_grad():
        out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=7)
        inputs = rb.collect_decode_inputs(pol.decoder, env, td, out["actions"], S)
    res = {}
    for impl in ("aten", "fused", "fp64"):
        dec = copy.deepcopy(pol.decoder).double() if impl == "fp64" else pol.decoder
        dt = torch.float64 if impl == "fp64" else torch.float32
        dur = td["duration_matrix"].to(dt) if name == "rcvrptw" else None
        training.REPLAY_IMPL = "aten" if impl == "aten" else "fused"    # fp64 tensors take the plain-torch form
        try:
            r_, c_ = (t.detach().to(dt).requires_grad_(True) for t in (row, col))
            dec.zero_grad(set_to_none=True)
            logp = rb.batched_logprobs(dec, r_, c_, td["distance_matrix"].to(dt), dur, inputs, out["actions"], S, step_chunk=7)
            rb.pomo_shared_baseline_loss(out["reward"].to(dt), logp.sum(1), S).backward()
        finally:
            training.REPLAY_IMPL = "fused"
        res[impl] = (logp.detach(), {"row": r_.grad, "col": c_.grad,
                                     **{k: p.grad.clone() for k, p in dec.named_parameters() if p.grad is not None}})
    train_ops.check_status(dev)
    assert (res["fused"][0] - res["aten"][0]).abs().max().item() < 5e-5
    assert (res["fused"][0].sum(1) - out["log_likelihood"]).abs().max().item() < 2e-3
    assert set(res["fused"][1]) == set(res["aten"][1]) == set(res["fp64"][1])
    errs = {k: (_rel(res["fused"][1][k], ref), _rel(res["aten"][1][k], ref)) for k, ref in res["fp64"][1].items()}
    behind_relu = {"row", "col", "context_embedding.project_context.weight", "project_node_embeddings.weight", "pointer.ffn.lins.0.weight",
                   "pointer.ffn.lins.0.bias"}
    assert all(e_fused <= max(1e-4, 2 * e_aten) for k, (e_fused, e_aten) in errs.items() if k not in behind_relu), errs
    assert all(errs[k][0] < 5e-2 for k in behind_relu), errs
    db1, db1_ref = res["fused"][1]["pointer.ffn.lins.0.bias"].double(), res["fp64"][1]["pointer.ffn.lins.0.bias"]
    d = (db1 - db1_ref).abs()
    d[d.argmax()] = 0                                    # one hidden unit may take the other side of the relu
    assert float(d.max() / db1_ref.abs().max()) <= max(1e-4, 2 * errs["pointer.ffn.lins.0.bias"][1]), errs


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,B,S", [("atsp", 1000, 2, 16), ("rcvrp", 200, 4, 201)])
def test_policy_trains_at_large_n(name, n, B, S):
    """RRNetPolicy.forward(phase="train") under grad at n = 1000 and n = 200: the actions of the no-grad call with the same seed, its
    log-likelihood, and finite, non-zero gradients of the POMO loss for the decoder and both encoder outputs."""
    import rrnco_b200 as rb
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    env, td, pol, row, col = _policy(name, B, n, dev, seed=21)
    with torch.no_grad():
        ref = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=1234)
    out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S, seed=1234)
    assert torch.equal(out["actions"], ref["actions"])
    assert out["log_likelihood"].requires_grad
    assert (out["log_likelihood"].detach() - ref["log_likelihood"]).abs().max().item() < 2e-3
    rb.pomo_shared_baseline_loss(out["reward"], out["log_likelihood"], S).backward()
    train_ops.check_status(dev)
    grads = {"W1": pol.decoder.pointer.ffn.lins[0].weight.grad, "project_node_embeddings": pol.decoder.project_node_embeddings.weight.grad,
             "alpha": pol.decoder.alpha.grad, "row": row.grad, "col": col.grad}
    for k, gr in grads.items():
        assert gr is not None and bool(torch.isfinite(gr).all()) and float(gr.abs().max()) > 0, k


@pytest.mark.gpu
def test_tiled_replay_memory():
    """At RCVRP n = 200 the peak memory rise of batched_logprobs forward + backward stays within 1.25x of what the graph keeps,
    counted from its saved tensors per replay row (rows = R (T - 1)):
      attention  q, out [128 fp32 each], lse [8 fp32], action mask [N bytes]
      FFN        relu bit mask [16 int32], hidden activations [512 fp32, rows padded to 128 per chunk]
      pointer    g [128 fp32], tail Jacobian [ldz fp32], d logp / d alpha [1 fp32]
      context    current node [int64], state scalars [k fp32]
    plus the [R, T - 1] log-probs."""
    import rrnco_b200 as rb
    from rrnco_b200 import train_ops
    dev = torch.device("cuda", 0)
    name, n, B, S, chunk = "rcvrp", 200, 8, 201, 32
    env, td, pol, row, col = _policy(name, B, n, dev, seed=31)
    with torch.no_grad():
        out = pol(td, env, phase="train", decode_type="multistart_sampling", num_starts=S)
        inputs = rb.collect_decode_inputs(pol.decoder, env, td, out["actions"], S)
    N = td["action_mask"].shape[-1]
    Tm = out["actions"].shape[1] - 1
    R = S * B
    k_state = inputs["ctx_state"].shape[-1]
    ldz = 128 * ((N + 127) // 128)
    rows_per_chunk = [min(chunk, Tm - t0) * S for t0 in range(0, Tm, chunk)]
    kept = 0
    for L in rows_per_chunk:
        rows = B * L
        kept += rows * (4 * (128 + 128 + 8) + N + 4 * 16 + 4 * 128 + 4 * ldz + 4 + 8 + 4 * k_state)
        kept += ((rows + 127) // 128) * 128 * 512 * 4
    kept += R * Tm * 4
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    r_, c_ = row.detach().clone().requires_grad_(True), col.detach().clone().requires_grad_(True)
    logp = rb.batched_logprobs(pol.decoder, r_, c_, td["distance_matrix"].float(), None, inputs, out["actions"], S, step_chunk=chunk)
    rb.pomo_shared_baseline_loss(out["reward"], logp.sum(1), S).backward()
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated(dev) - base
    train_ops.check_status(dev)
    assert rise <= 1.25 * kept, (rise, kept, rise / kept)
