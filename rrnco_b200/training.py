"""Training hand-off (SURVEY.md 8(f) rank 2): gradients for REINFORCE from rollouts sampled by the fused kernel.

The fused rollout kernel is forward-only.  Upstream's training step (`rrnco/models/rl.py:99-130`) needs
`log_likelihood` with a graph to the decoder parameters and the encoder output.  Here the two are separated:

  1. actions are sampled by `RRNetPolicy.forward(..., phase="train")` on the fused kernel (no graph);
  2. `replay_log_likelihood` re-evaluates log pi(a_t | s_t) for those actions with autograd:
     a) the env is replayed on the CUDA step kernels (no graph) to collect the decoder inputs of every step - current /
        first node, state scalars, action mask (`iter_decode_inputs`, a generator consumed chunk by chunk);
     b) because the actions are known, ALL decode steps are evaluated at once, one row per (rollout, step)
        (`batched_logprobs`: context projection, 8-head masked attention, FFN + residual, pointer logits, scale-adaptive
        bias, tanh clip, mask, log-softmax; decoder.py:151-206,281-326, decoding.py:311-361) instead of upstream's T
        sequential small-kernel steps.  On CUDA tensors those rows go through the hand-written kernels of
        librrnco_b200_train.so, forward AND backward (`train_ops.py`: context query as a table gather, attention on the CUDA
        cores with mma.sync row sums, tcgen05 FFN with a relu bit mask and an X^T Y weight-gradient kernel, tcgen05 pointer
        scores + a one-pass tail that leaves the Jacobian; instances of more than 102 / 128 nodes, up to 1024, on the key-tiled
        attention and pointer kernels); torch keeps the autograd graph and the two tiny per-instance projections.
        `REPLAY_IMPL = "aten"` (and any CPU tensor, bf16 autocast, N > 1024) selects the same math as plain torch ops.
  3. `pomo_shared_baseline_loss` = rl4co REINFORCE with the shared (POMO) baseline [rl4co-recalled], rl.py:119-128.

The plain-torch form is checked against the oracle's per-step decoder on the CPU (tests/test_training_handoff.py); the kernels
against fp64 torch op by op and against the plain-torch form on sampled rollouts, and the replay against the log-likelihood of
the sampling kernel itself, on the GPU (tests/test_train_ops.py, tests/test_gpu_parity.py).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from .tdlite import TensorDictLite, batchify


ATTENTION_IMPL = "sdpa"  # "sdpa" | "matmul": how the ATen form of batched_logprobs evaluates the masked 8-head attention
# CUDA tensors: attention, residual FFN and the pointer tail (forward AND backward) run on the hand-written kernels of
# librrnco_b200_train.so (rrnco_b200/train_ops.py; a missing library raises).  "aten" keeps the plain-torch form on the GPU:
# the comparison arm of tests/test_gpu_parity.py and tools/train_step_probe.py, and the bf16-autocast option.
REPLAY_IMPL = "fused"   # "fused" | "aten"


def iter_decode_inputs(decoder, env, td, actions: torch.Tensor, num_starts: int, step_chunk: int = 32):
    """Replays `actions` [R, T] (R = num_starts * n_inst, multistart order) through the env's CUDA step kernels and yields, per
    chunk of `step_chunk` decoder calls, `(t0, t1, inputs)` with what the decoder saw at steps t0+1 .. t1 (step 0 is the forced
    POMO start, decoding.py:186-192): current_node [t1-t0, R], first_node (atsp), ctx_state [t1-t0, R, k], action_mask
    [t1-t0, R, N].  A generator: the replay is launch-bound (one small kernel per step), so `batched_logprobs` consumes the chunks
    as they appear and its kernels run on the GPU while the host issues the next steps."""
    from .models import _ROLLOUT_STATE_KEYS
    name = decoder.env_name
    S = int(num_starts)
    if S < 2:
        raise NotImplementedError("training replay is multistart (POMO) only, as rl.py:119 asserts")
    R, T = actions.shape
    with torch.no_grad():
        roll = TensorDictLite({k: (batchify(td[k], S) if k in _ROLLOUT_STATE_KEYS[name] else td[k])
                               for k in td.keys() if k != "done"}, batch_size=[R])
        roll.set("action", actions[:, 0].contiguous())
        roll = env.step(roll)["next"]
    for t0 in range(0, T - 1, step_chunk):
        t1 = min(T - 1, t0 + step_chunk)
        cur, first, state, mask = [], [], [], []
        with torch.no_grad():   # not held across the yield: the consumer builds its graph in between
            for t in range(t0 + 1, t1 + 1):
                # no copies: every env step hands out freshly allocated state tensors (envs.py `_step`), nothing is updated in place
                cur.append(roll["current_node"].reshape(-1))
                mask.append(roll["action_mask"])
                if name == "atsp":
                    first.append(roll["first_node"].reshape(-1))
                else:
                    state.append(decoder._ctx_state(roll))
                roll.set("action", actions[:, t].contiguous())
                roll = env.step(roll)["next"]
            out = {"current_node": torch.stack(cur), "action_mask": torch.stack(mask)}
            if name == "atsp":
                out["first_node"] = torch.stack(first)
            else:
                out["ctx_state"] = torch.stack(state)
        yield t0, t1, out


def collect_decode_inputs(decoder, env, td, actions: torch.Tensor, num_starts: int) -> dict:
    """All chunks of `iter_decode_inputs` at once: current_node [T-1, R], first_node (atsp), ctx_state [T-1, R, k],
    action_mask [T-1, R, N]."""
    chunks = [c for _, _, c in iter_decode_inputs(decoder, env, td, actions, num_starts)]
    return {k: torch.cat([c[k] for c in chunks]) for k in chunks[0]}


def uses_replay_kernels(col_emb: torch.Tensor, N: int) -> bool:
    """Which form `batched_logprobs` takes: the kernels of train_ops for CUDA fp32 replays of up to 1024 nodes
    (train_ops.MAX_NODES_REPLAY), the plain-torch form for REPLAY_IMPL = "aten", bf16 autocast, CPU or non-fp32 tensors and larger
    instances."""
    if not (col_emb.is_cuda and col_emb.dtype == torch.float32 and REPLAY_IMPL == "fused" and not torch.is_autocast_enabled()):
        return False
    from . import train_ops
    return N <= train_ops.MAX_NODES_REPLAY


def batched_logprobs(decoder, row_emb, col_emb, distance, duration, inputs: dict, actions: torch.Tensor,
                     num_starts: int, temperature: float = 1.0, tanh_clipping: float = 10.0,
                     step_chunk: int = 32, autocast_dtype=None) -> torch.Tensor:
    """log pi(a_t | s_t) for t = 1..T-1, [R, T-1], differentiable w.r.t. the decoder parameters, row_emb and col_emb.
    Rollout r = s * n_inst + b (upstream's batchify order); instance data is never replicated over the starts.
    `autocast_dtype` (e.g. torch.bfloat16): run the contractions under torch.autocast, as upstream's trainer does
    (`configs/trainer/default.yaml:8` precision "16-mixed"); default fp32."""
    if autocast_dtype is not None:
        with torch.autocast(col_emb.device.type, dtype=autocast_dtype):
            return batched_logprobs(decoder, row_emb, col_emb, distance, duration, inputs, actions, num_starts,
                                    temperature, tanh_clipping, step_chunk, None)
    name, E, H = decoder.env_name, decoder.embed_dim, decoder.num_heads
    n_inst, N, _ = col_emb.shape
    S = int(num_starts)
    R = S * n_inst
    Tm = actions.shape[1] - 1

    def chunks():  # `inputs`: the dict of collect_decode_inputs, or the generator iter_decode_inputs (consumed as it is produced)
        if isinstance(inputs, dict):
            for a in range(0, Tm, step_chunk):
                b = min(Tm, a + step_chunk)
                yield a, b, {key: val[a:b] for key, val in inputs.items()}
        else:
            yield from inputs

    fused = uses_replay_kernels(col_emb, N) and E == 128 and H == 8
    k, v, lk = F.linear(col_emb, decoder.project_node_embeddings.weight).chunk(3, dim=-1)  # decoder.py:214-232
    W = decoder.context_embedding.project_context.weight

    def heads(x):  # [n_inst, L, E] -> [n_inst, H, L, E / H]
        return x.unflatten(-1, (H, -1)).transpose(1, 2)

    kh, vh = heads(k), heads(v)
    inst = torch.arange(n_inst, device=col_emb.device)
    w1, b1 = decoder.pointer.ffn.lins[0].weight, decoder.pointer.ffn.lins[0].bias
    w2, b2 = decoder.pointer.ffn.lins[1].weight, decoder.pointer.ffn.lins[1].bias
    if fused:  # node part of project_context as per-instance tables (tiny GEMMs, torch autograd)
        tab_a = F.linear(row_emb, W[:, :E])
        tab_b = F.linear(row_emb, W[:, E:2 * E]) if name == "atsp" else None
    out = []
    for t0, t1, chunk in chunks():
        L = (t1 - t0) * S

        def per_inst(x):  # [Tc, R, ...] with r = s * n_inst + b  ->  [n_inst, Tc * S, ...]
            return x.unflatten(1, (S, n_inst)).movedim(2, 0).flatten(1, 2)

        cur = per_inst(chunk["current_node"])                      # [n_inst, L]
        mask = per_inst(chunk["action_mask"]).bool()               # [n_inst, L, N]
        act = per_inst(actions[:, 1 + t0:1 + t1].t().contiguous())         # [n_inst, L]
        if fused:   # context.py:18-70 with the projection pulled through the gather: q = P[b, cur] (+ P2[b, ..]) + state W_s^T
            from . import train_ops
            cur, mask, act = cur.contiguous(), mask.contiguous(), act.contiguous()    # per_inst returns strided views
            if name == "atsp":
                q = train_ops.context_query(tab_a, per_inst(chunk["first_node"]), tab_b, cur)
            else:
                q = train_ops.context_query(tab_a, cur, None, None, per_inst(chunk["ctx_state"]), W[:, E:].t())
            g = train_ops.fused_attention(q, k, v, mask, add_residual=True)             # decoder.py:281-293 (+ q)
            g = train_ops.fused_ffn(g, w1, b1, w2, b2)                                  # decoder.py:296
            logp = train_ops.pointer_logprob(g, lk, decoder.alpha, decoder.beta if name == "rcvrptw" else None, distance,
                                             duration if name == "rcvrptw" else None, cur, mask, act, tanh_clipping,
                                             temperature)           # decoder.py:183-198, 298-301; decoding.py:311-399
            out.append(logp.unflatten(1, (t1 - t0, S)).permute(2, 0, 1).reshape(R, t1 - t0))
            continue
        emb_cur = row_emb[inst[:, None], cur]                              # [n_inst, L, E]
        if name == "atsp":  # rl4co TSPContext: [first, current] (multistart: never the placeholder)
            first = per_inst(chunk["first_node"])
            ctx = torch.cat([row_emb[inst[:, None], first], emb_cur], -1)
        else:               # context.py:18-31: [current-node embedding, state scalars]
            ctx = torch.cat([emb_cur, per_inst(chunk["ctx_state"]).to(emb_cur.dtype)], -1)
        q = F.linear(ctx, W)                                               # [n_inst, L, E]
        if ATTENTION_IMPL == "sdpa":
            h = F.scaled_dot_product_attention(heads(q), kh, vh, attn_mask=mask.unsqueeze(1))  # decoder.py:281-293
        else:  # explicit: head dim 16 and 101 keys are far from the tile shapes of the fused SDPA kernels
            sc = torch.matmul(heads(q), kh.transpose(-1, -2)) * (1.0 / math.sqrt(E // H))
            sc = sc.masked_fill(~mask.unsqueeze(1), float("-inf"))
            h = torch.matmul(torch.softmax(sc, dim=-1), vh)
        g = h.transpose(1, 2).flatten(-2) + q
        g = F.linear(F.relu(F.linear(g, w1, b1)), w2, b2) + g              # decoder.py:296
        logits = torch.bmm(g, lk.transpose(1, 2)).float() / math.sqrt(E)   # [n_inst, L, N]
        bias = decoder.alpha * distance[inst[:, None], cur]                # decoder.py:183-198
        if name == "rcvrptw":
            bias = bias + decoder.beta * duration[inst[:, None], cur]
        logits = torch.log(torch.exp(logits - bias) + 1e-6)
        if tanh_clipping > 0:                                              # decoding.py:311-361
            logits = torch.tanh(logits) * tanh_clipping
        logits = logits.masked_fill(~mask, float("-inf")) / temperature
        logp = F.log_softmax(logits, dim=-1).gather(-1, act.unsqueeze(-1)).squeeze(-1)   # [n_inst, L]
        out.append(logp.unflatten(1, (t1 - t0, S)).permute(2, 0, 1).reshape(R, t1 - t0))  # back to r = s * n_inst + b
    return torch.cat(out, 1)


def replay_log_likelihood(policy, td, env, actions: torch.Tensor, num_starts: int, phase: str = "train",
                          embeddings=None, temperature=None, tanh_clipping=None, step_chunk: int = 32,
                          autocast_dtype=None):
    """log_likelihood [R] of `actions` with a graph to the decoder parameters and the encoder (policy.py:240-243 for the
    Evaluate strategy, decoding.py:386-399).  `td` is the reset td of the batch the actions were sampled on."""
    row_emb, col_emb = embeddings if embeddings is not None else policy.encoder(td, phase=phase)
    inputs = iter_decode_inputs(policy.decoder, env, td, actions, num_starts, step_chunk)   # consumed chunk by chunk below
    dur = td["duration_matrix"].float() if policy.decoder.env_name == "rcvrptw" else None
    logp = batched_logprobs(policy.decoder, row_emb.float(), col_emb.float(), td["distance_matrix"].float(), dur, inputs,
                            actions, num_starts, policy.temperature if temperature is None else temperature,
                            policy.tanh_clipping if tanh_clipping is None else tanh_clipping, step_chunk, autocast_dtype)
    if not bool((logp > -1000).all()):
        raise AssertionError("Logprobs should not be -inf, check sampling procedure!")
    return logp.sum(1)


def pomo_shared_baseline_loss(reward: torch.Tensor, log_likelihood: torch.Tensor, num_starts: int) -> torch.Tensor:
    """REINFORCE with the shared baseline over the starts of an instance (rl.py:112-128 + rl4co REINFORCE.calculate_loss
    with baseline "shared" [rl4co-recalled]): advantage = reward - mean_s reward; loss = -(advantage * log pi).mean()."""
    S = int(num_starts)
    r = reward.unflatten(0, (S, -1))          # [S, n_inst] (r = s * n_inst + b)
    ll = log_likelihood.unflatten(0, (S, -1))
    advantage = r - r.mean(0, keepdim=True)
    return -(advantage.detach() * ll).mean()
