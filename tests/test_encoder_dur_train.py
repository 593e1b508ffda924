"""Training through the rcvrptw duration gate of the neural adaptive bias (DistAngleFusion with use_duration_matrix;
attn_freenet.py:242-289): the tcgen05 backward of csrc_train/encoder_dur_train.cu (rrnco_train_nab_dur_backward) and its
autograd wiring.

CPU: an fp64 torch restatement of the kernel's reduction (six E x E contractions over the pairs plus small sums, then the
closed-form gradients) equals torch.autograd through the oracle; the Python-level contracts of `train_duration_gate`.
GPU: the 19 kernel gradients against fp64 autograd (bar: 1e-4 of each tensor's largest magnitude), bitwise
reproducibility, the trainable forward equal to the inference forward, the memory bound, a patched rcvrptw block against the
unpatched one in fp64, and a loud fp16 operand overflow.
"""
import copy
import os

import numpy as np
import pytest
import torch
from torch import nn

from oracle import encoder as oenc

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "encoder_nab.npz")
NAMES = [f"{m}.{i}.{w}" for m in ("dist_emb", "angle_emb", "dur_emb") for i, w in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias"))]
NAMES += ["gate.0.weight", "gate.0.bias", "gate.2.weight", "gate.2.bias", "gate_temperature", "out_lin.weight", "out_lin.bias"]


def _fixture():
    z = np.load(GOLDEN)
    p = {k[len("dur.param."):]: torch.from_numpy(np.array(z[k])) for k in z.files if k.startswith("dur.param.")}
    return torch.from_numpy(z["coords"]), torch.from_numpy(z["cost"]), torch.from_numpy(z["dur"]), p


def _default_params(seed, temperature=None):
    import rrnco_b200 as rb
    torch.manual_seed(seed)
    p = {k: v.detach().clone() for k, v in rb.DistAngleFusion(128, use_duration_matrix=True).state_dict().items()}
    if temperature is not None:
        p["gate_temperature"] = torch.tensor(float(temperature))
    return p


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def autograd_grads(p, coords, cost, dur, G, scale):
    """d(sum G * scale * DistAngleFusion(coords, cost, dur)) / d parameters through the oracle's op sequence, fp64."""
    pd = {k: v.detach().double().cpu().clone().requires_grad_(True) for k, v in p.items()}
    out = oenc.dist_angle_fusion(pd, coords.double().cpu(), cost.double().cpu(), dur.double().cpu()) * scale
    out.backward(G.double().cpu())
    return {k: v.grad for k, v in pd.items()}


def contraction_grads(p, coords, cost, dur, G, scale):
    """What rrnco_train_nab_dur_backward computes, in fp64 torch: per pair only dz, dO and the E-vector r; over the pairs
    A_x = sum r (on_x s_x)^T, B_x = sum r on_x^T and small sums; then the closed forms of the 19 gradients."""
    d = {k: v.double() for k, v in p.items()}
    E = d["out_lin.weight"].shape[1]
    xs = [cost.double().reshape(-1), oenc.pairwise_angles(coords.double()).reshape(-1), dur.double().reshape(-1)]
    mlps = ["dist_emb", "angle_emb", "dur_emb"]
    Wg1, bg1, Wg2, bg2 = d["gate.0.weight"], d["gate.0.bias"], d["gate.2.weight"], d["gate.2.bias"]
    wo, tau = d["out_lin.weight"][0], torch.exp(-d["gate_temperature"])
    gam = scale * G.double().reshape(-1)
    w1 = [d[f"{m}.0.weight"][:, 0] for m in mlps]
    b1 = [d[f"{m}.0.bias"] for m in mlps]
    W2 = [d[f"{m}.2.weight"] for m in mlps]
    b2 = [d[f"{m}.2.bias"] for m in mlps]
    Wg1x = [Wg1[:, x * E:(x + 1) * E] for x in range(3)]
    M = [Wg1x[x] @ W2[x] for x in range(3)]
    pre = [xs[x][:, None] * w1[x] + b1[x] for x in range(3)]
    on = [(q > 0).double() for q in pre]
    h = [torch.relu(q) for q in pre]
    hp = sum(h[x] @ M[x].t() for x in range(3)) + bg1 + sum(Wg1x[x] @ b2[x] for x in range(3))
    sig = hp * torch.sigmoid(hp)
    z = (sig @ Wg2.t() + bg2) * tau
    g = torch.softmax(z, -1)
    O = torch.stack([h[x] @ (W2[x].t() @ wo) + wo @ b2[x] for x in range(3)], -1)
    ob = (g * O).sum(-1, keepdim=True)
    dO = gam[:, None] * g
    dz = gam[:, None] * g * (O - ob)
    sg = torch.sigmoid(hp)
    r = tau * (dz @ Wg2) * (sg * (1 + hp * (1 - sg)))
    rho = r.sum(0)
    out = {}
    dwo = torch.zeros(E, dtype=torch.float64)
    for x, m in enumerate(mlps):
        A = r.t() @ (on[x] * xs[x][:, None])
        B = r.t() @ on[x]
        a1 = (on[x] * (dO[:, x] * xs[x])[:, None]).sum(0)
        a0 = (on[x] * dO[:, x][:, None]).sum(0)
        R = A * w1[x] + B * b1[x]
        eta = w1[x] * a1 + b1[x] * a0
        uo = W2[x].t() @ wo
        sdO = dO[:, x].sum()
        out[f"{m}.0.weight"] = ((M[x] * A).sum(0) + uo * a1)[:, None]
        out[f"{m}.0.bias"] = (M[x] * B).sum(0) + uo * a0
        out[f"{m}.2.weight"] = Wg1x[x].t() @ R + torch.outer(wo, eta)
        out[f"{m}.2.bias"] = Wg1x[x].t() @ rho + wo * sdO
        out[f"_wg1_{x}"] = R @ W2[x].t() + torch.outer(rho, b2[x])
        dwo = dwo + W2[x] @ eta + b2[x] * sdO
    out["gate.0.weight"] = torch.cat([out.pop(f"_wg1_{x}") for x in range(3)], 1)
    out["gate.0.bias"] = rho
    out["gate.2.weight"] = tau * dz.t() @ sig
    out["gate.2.bias"] = tau * dz.sum(0)
    out["gate_temperature"] = -(dz * z).sum()
    out["out_lin.weight"] = dwo[None, :]
    out["out_lin.bias"] = gam.sum()[None]
    return out


def _cases():
    coords, cost, dur, p = _fixture()
    g = torch.Generator().manual_seed(51)
    c2, m2 = torch.rand(2, 11, 2, generator=g), torch.rand(2, 11, 11, generator=g) * 1.4
    d2 = torch.rand(2, 11, 11, generator=g) * 2.0
    return [("fixture", p, coords, cost, dur), ("default init", _default_params(52), c2, m2, d2),
            ("sharp gate T=0", _default_params(53, 0.0), c2, m2, d2), ("sharp gate T=-0.5", _default_params(54, -0.5), c2, m2, d2)]


def test_contraction_backward_equals_autograd_through_the_oracle():
    g = torch.Generator().manual_seed(55)
    for tag, p, coords, cost, dur in _cases():
        G = torch.randn(cost.shape, generator=g, dtype=torch.float64)
        for transposed, scale in ((False, 1.0), (True, 0.7)):
            c, du = (cost.transpose(1, 2), dur.transpose(1, 2)) if transposed else (cost, dur)
            want = autograd_grads(p, coords, c, du, G, scale)
            got = contraction_grads(p, coords, c, du, G, scale)
            for k in NAMES:
                assert got[k].shape == want[k].shape, (tag, k)
                assert _rel(got[k], want[k]) < 1e-10, (tag, transposed, k, _rel(got[k], want[k]))


def test_train_duration_gate_contracts_on_the_host():
    import rrnco_b200 as rb
    coords, cost, dur, p = _fixture()
    m = rb.DistAngleFusion(128, use_duration_matrix=True, trainable=True, train_duration_gate=True)
    m.load_state_dict(p, strict=True)
    assert sorted(n for n, _ in m.named_parameters()) == sorted(NAMES)
    with pytest.raises(NotImplementedError):   # no gradients for the inputs
        m(coords.clone().requires_grad_(True), cost, dur)
    with pytest.raises(NotImplementedError):
        m(coords, cost.clone().requires_grad_(True), dur)
    with pytest.raises(NotImplementedError):
        m(coords, cost, dur.clone().requires_grad_(True))


class _RefDur(nn.Module):  # upstream's rcvrptw module: its parameters, the oracle's op sequence
    def __init__(self):
        super().__init__()
        self.embed_dim = 64
        self.dist_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
        self.angle_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
        self.dur_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
        self.gate = nn.Sequential(nn.Linear(384, 128), nn.SiLU(), nn.Linear(128, 3))
        self.gate_temperature = nn.Parameter(torch.tensor(0.5))
        self.out_lin = nn.Linear(128, 1)

    def forward(self, coords, cost_mat, duration_mat=None):
        return oenc.dist_angle_fusion(dict(self.named_parameters()), coords, cost_mat, duration_mat)


class _AFT(nn.Module):
    def __init__(self):
        super().__init__()
        self.to_q, self.to_k, self.to_v, self.project = (nn.Linear(128, 128) for _ in range(4))

    def forward(self, x, y=None, adapt_bias=None):
        return oenc.aft_full(dict(self.named_parameters()), x, y, adapt_bias)


class _DurBlock(nn.Module):  # upstream's attribute names of an rcvrptw block (attn_freenet.py:360-442)
    def __init__(self):
        super().__init__()
        self.alpha = nn.Parameter(torch.full((1,), 1.3))
        self.attn_free = _AFT()
        self.multi_head_combine = nn.Linear(128, 128)
        self.neural_adaptive_bias = _RefDur()
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(128), nn.LayerNorm(128), nn.LayerNorm(128)
        self.feed_forward = lambda a, b: a + b

    def forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None):
        row_emb, col_emb = self.norm1(row_emb), self.norm2(col_emb)
        bias = self.neural_adaptive_bias(coords, cost_mat, duration_mat) * self.alpha
        out = self.attn_free(row_emb, y=col_emb, adapt_bias=bias)
        return self.feed_forward(self.norm3(self.multi_head_combine(out)), row_emb)


def test_patch_encoder_train_duration_gate_shares_upstream_tensors():
    import rrnco_b200 as rb
    blk = _DurBlock()
    refd = blk.neural_adaptive_bias
    params_before = list(blk.parameters())
    assert rb.patch_encoder(blk, trainable=True, train_duration_gate=True) == 1
    mine = blk.neural_adaptive_bias
    assert isinstance(mine, rb.DistAngleFusion) and mine.trainable and mine.use_duration_matrix
    assert mine.gate_temperature is refd.gate_temperature and mine.dur_emb[2].weight is refd.dur_emb[2].weight
    assert mine.gate[0].weight is refd.gate[0].weight and mine.out_lin.bias is refd.out_lin.bias
    assert sorted(n for n, _ in mine.named_parameters()) == sorted(NAMES)
    assert {id(q) for q in blk.parameters()} == {id(q) for q in params_before}


# ---------------------------------------------------------------------------------------------------------------- GPU

def _module(params, dev="cuda"):
    import rrnco_b200 as rb
    m = rb.DistAngleFusion(128, use_duration_matrix=True, trainable=True, train_duration_gate=True).to(dev)
    m.load_state_dict(params, strict=True)
    return m


def _kernel_grads(m, coords, cost, dur, G, scale):
    for q in m.parameters():
        q.grad = None
    out = m(coords, cost, dur, scale=scale)
    out.backward(G)
    return {k: q.grad.detach().clone() for k, q in m.named_parameters()}, out.detach()


def _check(got, want, tag):
    worst = 0.0
    for k in NAMES:
        assert got[k].shape == want[k].shape and got[k].dtype == torch.float32, (tag, k)
        if want[k].abs().max() < 1e-12:
            err = float(got[k].double().cpu().sub(want[k]).abs().max())
            assert err < 1e-9, (tag, k, err)
            continue
        err = _rel(got[k], want[k])
        worst = max(worst, err)
        assert err <= 1e-4, (tag, k, err)
    return worst


@pytest.mark.gpu
def test_kernel_gradients_match_fp64_autograd():
    dev = "cuda"
    coords, cost, dur, p = _fixture()
    g = torch.Generator().manual_seed(61)
    cases = [("fixture", p, coords, cost, dur, 1.0)]
    for tag, B, N, params in (("default 7 x 51", 7, 51, _default_params(62)), ("default 5 x 101", 5, 101, _default_params(63)),
                              ("sharp gate 5 x 101", 5, 101, _default_params(64, -0.5))):
        cases.append((tag, params, torch.rand(B, N, 2, generator=g), torch.rand(B, N, N, generator=g) * 1.4,
                      torch.rand(B, N, N, generator=g) * 2.0, 1.0))
    cases.append(("grad_out x 1e-6", _default_params(65, 0.0), torch.rand(5, 51, 2, generator=g),
                  torch.rand(5, 51, 51, generator=g) * 1.4, torch.rand(5, 51, 51, generator=g) * 2.0, 1e-6))
    worst = 0.0
    for tag, params, co, cm, du, gscale in cases:
        m = _module(params)
        G = torch.randn(cm.shape, generator=g) * gscale
        for transposed, scale in ((False, 1.0), (True, 0.7)):
            c, dd = (cm.transpose(1, 2), du.transpose(1, 2)) if transposed else (cm, du)
            want = autograd_grads(params, co, c, dd, G, scale)
            got, _ = _kernel_grads(m, co.to(dev), c.to(dev), dd.to(dev), G.to(dev), scale)
            worst = max(worst, _check(got, want, (tag, transposed)))
    print(f"\nworst gradient error / max |gradient| over the 19 tensors: {worst:.2e}")


@pytest.mark.gpu
def test_gradients_are_reproducible_and_forward_is_the_inference_kernel():
    dev = "cuda"
    m = _module(_default_params(66, 1.0))
    g = torch.Generator(device=dev).manual_seed(67)
    B, N = 37, 101
    coords = torch.rand(B, N, 2, device=dev, generator=g)
    cost = torch.rand(B, N, N, device=dev, generator=g) * 1.4
    dur = torch.rand(B, N, N, device=dev, generator=g) * 2.0
    G = torch.randn(B, N, N, device=dev, generator=g)
    for c, d in ((cost, dur), (cost.transpose(1, 2), dur.transpose(1, 2))):
        g1, out = _kernel_grads(m, coords, c, d, G, 1.3)
        g2, _ = _kernel_grads(m, coords, c, d, G, 1.3)
        for k in NAMES:
            assert torch.equal(g1[k], g2[k]), k
        with torch.no_grad():
            inf = m(coords, c, d, scale=1.3)
        assert torch.equal(out, inf)


@pytest.mark.gpu
def test_forward_backward_materialises_no_pair_embeddings():
    from rrnco_b200 import train_ops
    dev = "cuda"
    m = _module(_default_params(68))
    B, N = 512, 101
    g = torch.Generator(device=dev).manual_seed(69)
    coords = torch.rand(B, N, 2, device=dev, generator=g)
    cost = torch.rand(B, N, N, device=dev, generator=g)
    dur = torch.rand(B, N, N, device=dev, generator=g)
    G = torch.randn(B, N, N, device=dev, generator=g)
    ws = train_ops.lib().rrnco_train_nab_dur_workspace_bytes(B, N)
    m(coords, cost, dur).backward(G)   # warm-up: the parameters' .grad tensors exist before the measured window
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    m(coords, cost, dur).backward(G)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    assert 0 < rise < 4 * B * N * N * 4 + ws, (rise, ws)


@pytest.mark.gpu
def test_patched_rcvrptw_block_trains_like_the_unpatched_block():
    import rrnco_b200 as rb
    torch.manual_seed(70)
    blk = _DurBlock()
    ref = copy.deepcopy(blk).double()
    blk = blk.cuda()
    assert rb.patch_encoder(blk, trainable=True, train_duration_gate=True) == 1
    g = torch.Generator().manual_seed(71)
    B, N = 3, 40
    row, col = torch.randn(B, N, 128, generator=g), torch.randn(B, N, 128, generator=g)
    coords, cost, dur = torch.rand(B, N, 2, generator=g), torch.rand(B, N, N, generator=g), torch.rand(B, N, N, generator=g)
    W = torch.randn(B, N, 128, generator=g)
    args = (row.cuda(), col.cuda(), cost.cuda().transpose(1, 2), coords.cuda(), dur.cuda().transpose(1, 2))
    rargs = (row.double(), col.double(), cost.double().transpose(1, 2), coords.double(), dur.double().transpose(1, 2))
    (blk(*args) * W.cuda()).sum().backward()
    (ref(*rargs) * W.double()).sum().backward()
    rp = dict(ref.named_parameters())
    names = [k for k, _ in blk.named_parameters()]
    assert names == list(rp) and any(k.startswith("neural_adaptive_bias.") for k in names)
    for k, q in blk.named_parameters():
        if rp[k].grad.abs().max() < 1e-12:
            assert q.grad.abs().max() < 1e-5, k   # identically zero in exact arithmetic (softmax shift invariances)
        else:
            assert _rel(q.grad, rp[k].grad) <= 1e-4, (k, _rel(q.grad, rp[k].grad))
    torch.optim.SGD(blk.parameters(), lr=0.05).step()
    with torch.no_grad():
        for k, q in blk.named_parameters():
            rp[k].copy_(q.double().cpu())
    out = blk(*args)
    want = ref(*rargs)
    assert _rel(out.detach(), want.detach()) < 2e-5
    with torch.no_grad():   # the fused inference path sees the new parameters too
        assert _rel(blk(*args), want) < 2e-5


@pytest.mark.gpu
def test_operand_overflow_under_grad_raises():
    dev = "cuda"
    p = _default_params(72)
    p["dur_emb.0.weight"] = p["dur_emb.0.weight"] * 1e-3   # hidden activations stay small in the forward ...
    m = _module(p)
    g = torch.Generator().manual_seed(73)
    coords, cost = torch.rand(2, 20, 2, generator=g).to(dev), torch.rand(2, 20, 20, generator=g).to(dev)
    dur = torch.full((2, 20, 20), 5000.0, device=dev)                # ... but 16 x 5000 overflows the fp16 pair operand
    out = m(coords, cost, dur)
    with pytest.raises(AssertionError):
        out.backward(torch.ones_like(out))
