"""Training through the encoder's gating neural adaptive bias (DistAngleFusion, two-way gate; attn_freenet.py:242-289):
the segment-histogram backward of csrc_train/encoder_train.cu (rrnco_train_nab_backward) and its autograd wiring.

CPU: an fp64 torch restatement of the histogram backward equals torch.autograd through the oracle, which pins the
derivation and the rank / sign rule of the active units; the Python-level contracts that need no kernel.
GPU: the 12 kernel gradients against fp64 autograd (bar: 1e-4 of each tensor's largest magnitude), bitwise reproducibility,
the trainable forward equal to the inference forward, the memory bound, and a patched block against the unpatched one in fp64.
"""
import copy
import os

import numpy as np
import pytest
import torch
from torch import nn

from oracle import encoder as oenc

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "encoder_nab.npz")
NAMES = ["dist_emb.0.weight", "dist_emb.0.bias", "dist_emb.2.weight", "dist_emb.2.bias",
         "angle_emb.0.weight", "angle_emb.0.bias", "angle_emb.2.weight", "angle_emb.2.bias",
         "gate.0.weight", "gate.0.bias", "out_lin.weight", "out_lin.bias"]


def _fixture():
    z = np.load(GOLDEN)
    p = {k[len("nodur.param."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("nodur.param.")}
    return torch.from_numpy(z["coords"]), torch.from_numpy(z["cost"]), p


def autograd_grads(p, coords, cost, G, scale):
    """d(sum G * scale * DistAngleFusion(coords, cost)) / d parameters through the oracle's op sequence, fp64."""
    pd = {k: v.detach().double().cpu().clone().requires_grad_(True) for k, v in p.items()}
    out = oenc.dist_angle_fusion(pd, coords.double().cpu(), cost.double().cpu()) * scale
    out.backward(G.double().cpu())
    return {k: v.grad for k, v in pd.items()}


def histogram_grads(p, coords, cost, G, scale):
    """What rrnco_train_nab_backward computes, in fp64 torch: (alpha x, alpha, t x, t) histogrammed over the segments of the
    sorted breakpoints, prefix / suffix sums in rank order per unit, then the rank-2 gradient formulas."""
    d = {k: v.double() for k, v in p.items()}
    E = d["out_lin.weight"].shape[1]
    wg, wo = d["gate.0.weight"][0], d["out_lin.weight"][0]
    s = scale * G.double()
    xs = {"dist_emb": cost.double(), "angle_emb": oenc.pairwise_angles(coords.double())}
    halves = {"dist_emb": wg[:E], "angle_emb": wg[E:]}
    # forward quantities of the collapsed module
    f = {}
    for m, x in xs.items():
        h = torch.relu(x.unsqueeze(-1) * d[f"{m}.0.weight"][:, 0] + d[f"{m}.0.bias"])
        W2 = d[f"{m}.2.weight"]
        f[m] = (h @ (W2.t() @ halves[m]) + halves[m] @ d[f"{m}.2.bias"], h @ (W2.t() @ wo) + wo @ d[f"{m}.2.bias"])
    g = torch.sigmoid(f["dist_emb"][0] + f["angle_emb"][0] + d["gate.0.bias"][0])
    t = s * (f["dist_emb"][1] - f["angle_emb"][1]) * g * (1 - g)
    alphas = {"dist_emb": s * g, "angle_emb": s * (1 - g)}
    out = {}
    dwo = torch.zeros(E, dtype=torch.float64)
    for m, x in xs.items():
        w, b, W2, b2 = d[f"{m}.0.weight"][:, 0], d[f"{m}.0.bias"], d[f"{m}.2.weight"], d[f"{m}.2.bias"]
        bp = torch.where(w != 0, -b / w, torch.full_like(w, float("inf")))
        rank = torch.empty(E, dtype=torch.long)
        rank[torch.sort(bp, stable=True).indices] = torch.arange(E)   # ties broken by unit index
        seg = torch.searchsorted(torch.sort(bp).values, x.reshape(-1).contiguous())  # breakpoints strictly below x
        a = alphas[m].reshape(-1)
        tt = t.reshape(-1)
        xx = x.reshape(-1)
        hist = torch.zeros(E + 1, 4, dtype=torch.float64).index_add_(0, seg, torch.stack([a * xx, a, tt * xx, tt], 1))
        pre = hist.cumsum(0)
        tot = pre[E]
        on = torch.where((w > 0)[:, None], tot - pre[rank], torch.where((w < 0)[:, None], pre[rank],
                                                                        torch.where((b > 0)[:, None], tot, 0.0 * tot)))
        ug, uo = W2.t() @ halves[m], W2.t() @ wo
        out[f"{m}.0.weight"] = (uo * on[:, 0] + ug * on[:, 2])[:, None]
        out[f"{m}.0.bias"] = uo * on[:, 1] + ug * on[:, 3]
        sah, sth = w * on[:, 0] + b * on[:, 1], w * on[:, 2] + b * on[:, 3]
        out[f"{m}.2.weight"] = torch.outer(wo, sah) + torch.outer(halves[m], sth)
        out[f"{m}.2.bias"] = wo * tot[1] + halves[m] * tot[3]
        out[f"gate_half.{m}"] = W2 @ sth + b2 * tot[3]
        dwo += W2 @ sah + b2 * tot[1]
    out["gate.0.weight"] = torch.cat([out.pop("gate_half.dist_emb"), out.pop("gate_half.angle_emb")])[None]
    out["gate.0.bias"] = t.sum().reshape(1)
    out["out_lin.weight"] = dwo[None]
    out["out_lin.bias"] = s.sum().reshape(1)
    return out


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).abs().max() / b.double().cpu().abs().max().clamp_min(1e-300)).item()


def test_histogram_backward_equals_autograd_through_the_oracle():
    coords, cost, p = _fixture()
    g = torch.Generator().manual_seed(31)
    G = torch.randn(cost.shape, generator=g)
    for cm, scale in ((cost, 1.0), (cost.transpose(1, 2), 0.63), (cost * 3.0, -1.7)):
        want = autograd_grads(p, coords, cm, G, scale)
        got = histogram_grads(p, coords, cm, G, scale)
        assert set(got) == set(want) == set(NAMES)
        for k in NAMES:
            assert got[k].shape == want[k].shape, k
            assert _rel(got[k], want[k]) < 1e-10, (k, _rel(got[k], want[k]))


def test_trainable_module_contracts_on_the_host():
    import rrnco_b200 as rb
    with pytest.raises(NotImplementedError):
        rb.DistAngleFusion(128, use_duration_matrix=True, trainable=True)
    coords, cost, p = _fixture()
    m = rb.DistAngleFusion(128, trainable=True)
    m.load_state_dict(p, strict=True)
    assert [n for n, _ in m.named_parameters()] == NAMES
    with pytest.raises(NotImplementedError):   # the backward follows the segment tables
        m(coords, cost, variant=1)
    with pytest.raises(NotImplementedError):   # no gradients for the inputs
        m(coords.clone().requires_grad_(True), cost)
    with pytest.raises(NotImplementedError):
        m(coords, cost.clone().requires_grad_(True))


def test_patch_encoder_trainable_swaps_only_the_two_way_gate():
    import rrnco_b200 as rb

    class RefFusion(nn.Module):
        def __init__(self):
            super().__init__()
            self.embed_dim = 128
            self.dist_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
            self.angle_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
            self.gate = nn.Sequential(nn.Linear(256, 1), nn.Sigmoid())
            self.out_lin = nn.Linear(128, 1)

    class RefDur(nn.Module):  # the rcvrptw module's distinguishing attributes (attn_freenet.py:226-238)
        def __init__(self):
            super().__init__()
            self.dur_emb = nn.Linear(1, 2)
            self.gate_temperature = nn.Parameter(torch.tensor(5.0))

    class GateBlock(nn.Module):
        def __init__(self):
            super().__init__()
            self.angle_distance_fusion = RefFusion()

    class DurBlock(nn.Module):
        def __init__(self):
            super().__init__()
            self.neural_adaptive_bias = RefDur()

    enc = nn.ModuleList([GateBlock(), DurBlock()])
    ref, refd = enc[0].angle_distance_fusion, enc[1].neural_adaptive_bias
    params_before = list(enc.parameters())
    assert rb.patch_encoder(enc, trainable=True) == 1
    mine = enc[0].angle_distance_fusion
    assert isinstance(mine, rb.DistAngleFusion) and mine.trainable
    assert enc[1].neural_adaptive_bias is refd
    # the patched module trains upstream's own tensors: an optimizer built before the patch still sees them
    assert mine.dist_emb[0].weight is ref.dist_emb[0].weight and mine.out_lin.bias is ref.out_lin.bias
    assert {id(q) for q in enc.parameters()} == {id(q) for q in params_before}


# ---------------------------------------------------------------------------------------------------------------- GPU

def _kernel_grads(m, coords, cost, G, scale):
    for q in m.parameters():
        q.grad = None
    out = m(coords, cost, scale=scale)
    out.backward(G)
    return {k: q.grad.detach().clone() for k, q in m.named_parameters()}, out.detach()


@pytest.mark.gpu
def test_kernel_gradients_match_fp64_autograd():
    import rrnco_b200 as rb
    dev = "cuda"
    coords, cost, p = _fixture()
    cases = [("fixture", p, coords, cost)]
    torch.manual_seed(41)
    p2 = {k: v.detach() for k, v in rb.DistAngleFusion(128).state_dict().items()}   # default initialisation
    g = torch.Generator().manual_seed(42)
    cases.append(("default init 5 x 101", p2, torch.rand(5, 101, 2, generator=g), torch.rand(5, 101, 101, generator=g) * 1.4))
    worst = 0.0
    for tag, params, co, cm in cases:
        m = rb.DistAngleFusion(128, trainable=True).to(dev)
        m.load_state_dict(params, strict=True)
        G = torch.randn(cm.shape, generator=g)
        for transposed, scale in ((False, 1.0), (True, 0.8)):
            c = cm.transpose(1, 2) if transposed else cm
            want = autograd_grads(params, co, c, G, scale)
            got, _ = _kernel_grads(m, co.to(dev), c.to(dev), G.to(dev), scale)
            for k in NAMES:
                assert got[k].shape == want[k].shape and got[k].dtype == torch.float32, k
                err = _rel(got[k], want[k])
                worst = max(worst, err)
                assert err <= 1e-4, (tag, transposed, k, err)
    print(f"\nworst gradient error / max |gradient| over the 12 tensors: {worst:.2e}")


@pytest.mark.gpu
def test_gradients_are_reproducible_and_forward_is_the_inference_kernel():
    import rrnco_b200 as rb
    dev = "cuda"
    torch.manual_seed(43)
    m = rb.DistAngleFusion(128, trainable=True).to(dev)
    g = torch.Generator(device=dev).manual_seed(44)
    B, N = 37, 101
    coords = torch.rand(B, N, 2, device=dev, generator=g)
    cost = torch.rand(B, N, N, device=dev, generator=g) * 1.4
    G = torch.randn(B, N, N, device=dev, generator=g)
    for c in (cost, cost.transpose(1, 2)):
        g1, out = _kernel_grads(m, coords, c, G, 1.3)
        g2, _ = _kernel_grads(m, coords, c, G, 1.3)
        for k in NAMES:
            assert torch.equal(g1[k], g2[k]), k
        with torch.no_grad():
            inf = m(coords, c, scale=1.3)
        assert torch.equal(out, inf)


@pytest.mark.gpu
def test_forward_backward_materialises_no_pair_embeddings():
    import rrnco_b200 as rb
    from rrnco_b200 import train_ops
    dev = "cuda"
    torch.manual_seed(45)
    m = rb.DistAngleFusion(128, trainable=True).to(dev)
    B, N = 512, 101
    g = torch.Generator(device=dev).manual_seed(46)
    coords = torch.rand(B, N, 2, device=dev, generator=g)
    cost = torch.rand(B, N, N, device=dev, generator=g)
    G = torch.randn(B, N, N, device=dev, generator=g)
    ws = train_ops.lib().rrnco_train_nab_workspace_bytes(B, N)
    m(coords, cost).backward(G)   # warm-up: the parameters' .grad tensors exist before the measured window
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    m(coords, cost).backward(G)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    assert 0 < rise < 4 * B * N * N * 4 + ws, (rise, ws)


class _AFT(nn.Module):
    def __init__(self):
        super().__init__()
        self.to_q, self.to_k, self.to_v, self.project = (nn.Linear(128, 128) for _ in range(4))

    def forward(self, x, y=None, adapt_bias=None):
        return oenc.aft_full(dict(self.named_parameters()), x, y, adapt_bias)


class _RefFusion(nn.Module):  # upstream's module: its parameters, the oracle's op sequence
    def __init__(self):
        super().__init__()
        self.embed_dim = 128
        self.dist_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
        self.angle_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
        self.gate = nn.Sequential(nn.Linear(256, 1), nn.Sigmoid())
        self.out_lin = nn.Linear(128, 1)

    def forward(self, coords, cost_mat, duration_mat=None):
        return oenc.dist_angle_fusion(dict(self.named_parameters()), coords, cost_mat)


class _Block(nn.Module):  # upstream's attribute names (attn_freenet.py:360-442)
    def __init__(self):
        super().__init__()
        self.alpha = nn.Parameter(torch.full((1,), 1.3))
        self.attn_free = _AFT()
        self.multi_head_combine = nn.Linear(128, 128)
        self.angle_distance_fusion = _RefFusion()
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(128), nn.LayerNorm(128), nn.LayerNorm(128)
        self.feed_forward = lambda a, b: a + b

    def forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None):  # attn_freenet.py:417-442
        row_emb, col_emb = self.norm1(row_emb), self.norm2(col_emb)
        bias = self.angle_distance_fusion(coords, cost_mat, duration_mat) * self.alpha
        out = self.attn_free(row_emb, y=col_emb, adapt_bias=bias)
        return self.feed_forward(self.norm3(self.multi_head_combine(out)), row_emb)


@pytest.mark.gpu
def test_patched_block_trains_like_the_unpatched_block():
    import rrnco_b200 as rb
    torch.manual_seed(47)
    blk = _Block()
    ref = copy.deepcopy(blk).double()
    blk = blk.cuda()
    assert rb.patch_encoder(blk, trainable=True) == 1
    g = torch.Generator().manual_seed(48)
    B, N = 3, 40
    row, col = torch.randn(B, N, 128, generator=g), torch.randn(B, N, 128, generator=g)
    coords, cost = torch.rand(B, N, 2, generator=g), torch.rand(B, N, N, generator=g)
    W = torch.randn(B, N, 128, generator=g)
    args = (row.cuda(), col.cuda(), cost.cuda().transpose(1, 2), coords.cuda())   # the col-encoding block's view
    rargs = (row.double(), col.double(), cost.double().transpose(1, 2), coords.double())
    (blk(*args) * W.cuda()).sum().backward()
    (ref(*rargs) * W.double()).sum().backward()
    rp = dict(ref.named_parameters())
    names = [k for k, _ in blk.named_parameters()]
    assert names == list(rp) and any(k.startswith("angle_distance_fusion.") for k in names)
    for k, q in blk.named_parameters():
        if rp[k].grad.abs().max() < 1e-12:
            # identically zero in exact arithmetic: attn_free.to_k.bias (cancels in the softmax over the keys) and the
            # fusion's out_lin.bias (shifts a whole row of the bias softmax); fp32 leaves rounding residue only
            assert q.grad.abs().max() < 1e-5, k
        else:
            assert _rel(q.grad, rp[k].grad) <= 1e-4, (k, _rel(q.grad, rp[k].grad))
    # one SGD step; the next forward (packed tables rebuilt) is the fp64 block at the new parameters
    torch.optim.SGD(blk.parameters(), lr=0.05).step()
    with torch.no_grad():
        for k, q in blk.named_parameters():
            rp[k].copy_(q.double().cpu())
    out = blk(*args)
    want = ref(*rargs)
    assert _rel(out.detach(), want.detach()) < 2e-5
    with torch.no_grad():   # and the fused inference path sees the new parameters too
        assert _rel(blk(*args), want) < 2e-5
