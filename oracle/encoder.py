"""CPU restatement of the encoder hot spots (SURVEY.md 8(f) rank 4): the neural adaptive bias of an attention-free block
and AFT-full.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

  dist_angle_fusion   rrnco/models/nn/attn_freenet.py:242-289 (DistAngleFusion.forward, both gate variants)
  aft_full            rrnco/models/nn/attn_freenet.py:309-327 (AFTFull.forward)
  attn_free_block_bias rrnco/models/nn/attn_freenet.py:424-430 (the block scales the bias by its `alpha`)

Parameters are plain dicts keyed like the reference modules' state_dict (`dist_emb.0.weight`, ...), so a fixture
recorded from the reference module drives both this restatement and the CUDA kernel.
Pinned by tests/golden/encoder_nab.npz (recorded from the unmodified reference module by tests/golden/make_golden.py).
"""
import torch
import torch.nn.functional as F


def _mlp2(p, prefix, x):
    """nn.Sequential(Linear(1, E), ReLU, Linear(E, E)) on a [..., 1] input (attn_freenet.py:216-232)."""
    h = F.relu(F.linear(x, p[f"{prefix}.0.weight"], p[f"{prefix}.0.bias"]))
    return F.linear(h, p[f"{prefix}.2.weight"], p[f"{prefix}.2.bias"])


def pairwise_angles(coords, rows=None):
    """attn_freenet.py:254-262: angle of x_i - x_j for every ordered pair, [B, N, N] (rows i in range(*rows) only: [B, R, N])."""
    ci = coords if rows is None else coords[:, rows[0]:rows[1]]
    diff = ci.unsqueeze(2) - coords.unsqueeze(1)
    return torch.atan2(diff[..., 1], diff[..., 0])


def dist_angle_fusion(p, coords, cost_mat, duration_mat=None, rows=None):
    """DistAngleFusion.forward (attn_freenet.py:242-289): adapt_bias [B, N, N].
    Materialises [B, N, N, E] embeddings exactly like the reference: small sizes only.  `rows` = (i0, i1) evaluates the
    rows i0 <= i < i1 alone ([B, i1 - i0, N]): every pair is computed by the same ops, so large N can be done in chunks."""
    angles = pairwise_angles(coords, rows)
    if rows is not None:
        cost_mat = cost_mat[:, rows[0]:rows[1]]
        duration_mat = None if duration_mat is None else duration_mat[:, rows[0]:rows[1]]
    dist_emb = _mlp2(p, "dist_emb", cost_mat.unsqueeze(-1))
    angle_emb = _mlp2(p, "angle_emb", angles.unsqueeze(-1))
    if duration_mat is not None:
        dur_emb = _mlp2(p, "dur_emb", duration_mat.unsqueeze(-1))
        gate_in = torch.cat([dist_emb, angle_emb, dur_emb], dim=-1)
        logits = F.linear(F.silu(F.linear(gate_in, p["gate.0.weight"], p["gate.0.bias"])), p["gate.2.weight"], p["gate.2.bias"])
        g = F.softmax(logits / p["gate_temperature"].exp(), dim=-1)
        fused = g[..., [0]] * dist_emb + g[..., [1]] * angle_emb + g[..., [2]] * dur_emb
    else:
        gate_in = torch.cat([dist_emb, angle_emb], dim=-1)
        g = torch.sigmoid(F.linear(gate_in, p["gate.0.weight"], p["gate.0.bias"]))
        fused = g * dist_emb + (1 - g) * angle_emb
    return F.linear(fused, p["out_lin.weight"], p["out_lin.bias"]).squeeze(-1)


def aft_full(p, x, y, adapt_bias):
    """AFTFull.forward (attn_freenet.py:309-327), one head, hidden_dim = dim."""
    q = F.linear(x, p["to_q.weight"], p["to_q.bias"])
    k = F.linear(y, p["to_k.weight"], p["to_k.bias"])
    v = F.linear(y, p["to_v.weight"], p["to_v.bias"])
    a = torch.exp(torch.softmax(adapt_bias, dim=-1))
    k = torch.softmax(k, dim=1)
    temp = a @ (torch.exp(k) * v)
    weighted = temp / (a @ torch.exp(k))
    return F.linear(torch.sigmoid(q) * weighted, p["project.weight"], p["project.bias"])
