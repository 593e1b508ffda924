"""Encoder hot spot (SURVEY.md 8(f) rank 4): DistAngleFusion / AFTFull of the attention-free block.

CPU: the oracle restatement reproduces the fixture recorded from the UNMODIFIED reference module
(tests/golden/encoder_nab.npz <- tests/golden/make_golden.py encoder), and the algebraic collapse the CUDA kernel evaluates
(four E-vectors per module) is the same function.  GPU: the kernel against the fixture and against the oracle at n = 100.
"""
import os

import numpy as np
import pytest
import torch

from oracle import encoder as oenc

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "encoder_nab.npz")


def _fixture():
    z = np.load(GOLDEN)
    t = {k: torch.from_numpy(z[k]) for k in z.files}
    params = {tag: {k[len(tag) + 7:]: v for k, v in t.items() if k.startswith(tag + ".param.")} for tag in ("nodur", "dur", "aft")}
    params["aft"] = {k[10:]: v for k, v in t.items() if k.startswith("aft.param.")}
    return t, params


def _assert_same_ops_reordered(got, want):
    """Same torch ops as the recording, so the only difference is the order in which the host's GEMM sums (its SIMD code
    path and thread count: one thread instead of eight on the recording CPU already changes bits).  Measured across MKL's
    AVX-512 / AVX2 / SSE4.2 paths and 1-16 threads: at most 7 fp32 ulps of the output's largest magnitude; bound: 32.
    A 0.1 % change to 32 of the fixture's 39 parameter tensors exceeds it, and a 10 % change to the duration variant's
    `dist_emb.2.bias`.  The other six stay within it even at 10 %, so no tolerance pins them: AFT's `to_k.bias` cancels in the
    key softmax over the nodes, and the duration gate's `gate_temperature` of 15 (divided out as exp(15)) leaves that gate
    near uniform, whatever its other parameters."""
    atol = 32 * torch.finfo(torch.float32).eps * want.abs().max().item()
    torch.testing.assert_close(got, want, rtol=0, atol=atol)


def test_oracle_matches_reference_fixture():
    t, params = _fixture()
    for tag in ("nodur", "dur"):
        dur = t["dur"] if tag == "dur" else None
        out = oenc.dist_angle_fusion(params[tag], t["coords"], t["cost"], dur)
        _assert_same_ops_reordered(out, t[tag + ".bias"])
        outT = oenc.dist_angle_fusion(params[tag], t["coords"], t["cost"].transpose(1, 2), None if dur is None else dur.transpose(1, 2))
        _assert_same_ops_reordered(outT, t[tag + ".bias_T"])
    out = oenc.aft_full(params["aft"], t["aft.x"], t["aft.y"], t["nodur.bias"] * 1.7)
    _assert_same_ops_reordered(out, t["aft.out"])


def collapsed_bias(p, coords, cost):
    """What rrnco_nab_gating computes, in fp64 torch: the module collapsed to four E-vectors (encoder_kernels.cu header)."""
    d = {k: v.double() for k, v in p.items()}
    E = d["out_lin.weight"].shape[1]
    wg, wo = d["gate.0.weight"][0], d["out_lin.weight"][0]
    ug_d, uo_d = d["dist_emb.2.weight"].t() @ wg[:E], d["dist_emb.2.weight"].t() @ wo
    ug_a, uo_a = d["angle_emb.2.weight"].t() @ wg[E:], d["angle_emb.2.weight"].t() @ wo
    cg = d["gate.0.bias"][0] + wg[:E] @ d["dist_emb.2.bias"] + wg[E:] @ d["angle_emb.2.bias"]
    hd = torch.relu(cost.double().unsqueeze(-1) * d["dist_emb.0.weight"][:, 0] + d["dist_emb.0.bias"])
    ha = torch.relu(oenc.pairwise_angles(coords).double().unsqueeze(-1) * d["angle_emb.0.weight"][:, 0] + d["angle_emb.0.bias"])
    g = torch.sigmoid(hd @ ug_d + ha @ ug_a + cg)
    return g * (hd @ uo_d + wo @ d["dist_emb.2.bias"]) + (1 - g) * (ha @ uo_a + wo @ d["angle_emb.2.bias"]) + d["out_lin.bias"][0]


def test_collapsed_form_is_the_same_function():
    t, params = _fixture()
    got = collapsed_bias(params["nodur"], t["coords"], t["cost"])
    assert (got - t["nodur.bias"].double()).abs().max() < 2e-5  # fp32 reference vs fp64 collapse (values up to 11)


def test_mirror_module_has_the_reference_parameter_names():
    import rrnco_b200 as rb
    _, params = _fixture()
    m = rb.DistAngleFusion(128)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == {k: tuple(v.shape) for k, v in params["nodur"].items()}
    m.load_state_dict(params["nodur"], strict=True)
    md = rb.DistAngleFusion(128, use_duration_matrix=True)  # rcvrptw variant (attn_freenet.py:226-238)
    assert {k: tuple(v.shape) for k, v in md.state_dict().items()} == {k: tuple(v.shape) for k, v in params["dur"].items()}
    md.load_state_dict(params["dur"], strict=True)


@pytest.mark.gpu
def test_nab_kernel_matches_reference_fixture_and_oracle():
    import rrnco_b200 as rb
    dev = "cuda"
    t, params = _fixture()
    m = rb.DistAngleFusion(128).to(dev)
    m.load_state_dict(params["nodur"], strict=True)
    coords, cost = t["coords"].to(dev), t["cost"].to(dev)
    with torch.no_grad():
        for variant in (0, 1):  # 0 = piecewise-linear segment tables (default), 1 = sum over the hidden units
            out = m(coords, cost, variant=variant)
            outT = m(coords, cost.transpose(1, 2), variant=variant)  # the col-encoding block's transposed view: read through its base
            out2 = m(coords, cost, scale=0.37, variant=variant)
            assert (out.cpu() - t["nodur.bias"]).abs().max() < 2e-5, variant
            assert (outT.cpu() - t["nodur.bias_T"]).abs().max() < 2e-5, variant
            assert torch.allclose(out2, out * 0.37, rtol=1e-6, atol=1e-7)
    with pytest.raises(NotImplementedError):  # forward-only
        m(coords, cost)
    # n = 100 customers + depot, default initialisation (what a freshly built encoder holds), ragged tail of the pair chunks
    torch.manual_seed(3)
    m2 = rb.DistAngleFusion(128).to(dev)
    p2 = {k: v.detach().cpu() for k, v in m2.state_dict().items()}
    g = torch.Generator().manual_seed(4)
    coords = torch.rand(5, 101, 2, generator=g)
    cost = torch.rand(5, 101, 101, generator=g) * 1.4
    want = oenc.dist_angle_fusion(p2, coords, cost)
    with torch.no_grad():
        got = m2(coords.to(dev), cost.to(dev))
        got1 = m2(coords.to(dev), cost.to(dev), variant=1)
        # arguments exactly ON breakpoints and far outside their range (every segment incl. the two unbounded ones)
        w, bb = m2.dist_emb[0].weight[:, 0], m2.dist_emb[0].bias
        edge = torch.cat([-bb / w, torch.tensor([-1e6, -50.0, 0.0, 50.0, 1e6], device=dev)])
        ce = edge[torch.randint(0, edge.numel(), (2, 101, 101), device=dev, generator=torch.Generator(device=dev).manual_seed(5))]
        e0, e1 = m2(coords[:2].to(dev), ce, variant=0), m2(coords[:2].to(dev), ce, variant=1)
    assert (got.cpu() - want).abs().max() < 2e-6 * max(1.0, want.abs().max().item())
    assert (got1.cpu() - want).abs().max() < 2e-6 * max(1.0, want.abs().max().item())
    assert torch.isfinite(e0).all() and ((e0 - e1).abs() <= 1e-5 * e1.abs() + 1e-5).all()
    # a parameter update invalidates the packed cache
    with torch.no_grad():
        m2.out_lin.bias.add_(1.0)
        got2 = m2(coords.to(dev), cost.to(dev))
    assert (got2 - got - 1.0).abs().max() < 1e-5


@pytest.mark.gpu
def test_patch_encoder_swaps_the_gating_modules():
    import rrnco_b200 as rb
    from torch import nn

    class RefFusion(nn.Module):  # structure of the reference module (attn_freenet.py:201-240), torch forward = the oracle's
        def __init__(self):
            super().__init__()
            self.embed_dim = 128
            self.dist_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
            self.angle_emb = nn.Sequential(nn.Linear(1, 128), nn.ReLU(), nn.Linear(128, 128))
            self.gate = nn.Sequential(nn.Linear(256, 1), nn.Sigmoid())
            self.out_lin = nn.Linear(128, 1)

        def forward(self, coords, cost_mat, duration_mat=None):
            return oenc.dist_angle_fusion({k: v for k, v in self.state_dict().items()}, coords, cost_mat)

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.angle_distance_fusion = RefFusion()

    enc = nn.ModuleList([Block(), Block()]).to("cuda")
    g = torch.Generator().manual_seed(8)
    coords, cost = torch.rand(2, 30, 2, generator=g).cuda(), torch.rand(2, 30, 30, generator=g).cuda()
    with torch.no_grad():
        want = [b.angle_distance_fusion(coords, cost.transpose(1, 2)) for b in enc]
        assert rb.patch_encoder(enc) == 2 and rb.patch_encoder(enc) == 0
        got = [b.angle_distance_fusion(coords, cost.transpose(1, 2)) for b in enc]
    for a, b in zip(got, want):
        assert (a - b).abs().max() < 5e-6


def aft_core(q, k, v, bias):
    """AFTFull.forward (attn_freenet.py:309-327) between its Linear layers, fp64."""
    a = torch.exp(torch.softmax(bias.double(), dim=-1))
    e1 = torch.exp(torch.softmax(k.double(), dim=1))
    return torch.sigmoid(q.double()) * (a @ (e1 * v.double())) / (a @ e1)


@pytest.mark.gpu
def test_fused_aft_nab_kernel_matches_reference_fixture_and_oracle():
    import rrnco_b200 as rb
    import torch.nn.functional as F
    dev = "cuda"
    t, params = _fixture()
    m = rb.DistAngleFusion(128).to(dev)
    m.load_state_dict(params["nodur"], strict=True)
    pa = {k: v.to(dev) for k, v in params["aft"].items()}
    x, y = t["aft.x"].to(dev), t["aft.y"].to(dev)
    coords, cost = t["coords"].to(dev), t["cost"].to(dev)
    with torch.no_grad():
        q = F.linear(x, pa["to_q.weight"], pa["to_q.bias"])
        k = F.linear(y, pa["to_k.weight"], pa["to_k.bias"])
        v = F.linear(y, pa["to_v.weight"], pa["to_v.bias"])
        core = rb.aft_nab(q, k, v, coords, cost, m, scale=1.7)  # the fixture's AFT call used adapt_bias * 1.7
        out = F.linear(core, pa["project.weight"], pa["project.bias"])
    assert (out.cpu() - t["aft.out"]).abs().max() < 2e-5
    # n = 100 + depot, default-initialised modules, transposed cost view (col-encoding block), ragged row groups
    torch.manual_seed(9)
    m2 = rb.DistAngleFusion(128).to(dev)
    p2 = {kk: vv.detach().cpu() for kk, vv in m2.state_dict().items()}
    g = torch.Generator().manual_seed(10)
    B, N = 6, 101
    coords = torch.rand(B, N, 2, generator=g)
    cost = torch.rand(B, N, N, generator=g) * 1.4
    q, k, v = (torch.randn(B, N, 128, generator=g) for _ in range(3))
    for transposed in (False, True):
        cm = cost.transpose(1, 2) if transposed else cost
        want = aft_core(q, k, v, oenc.dist_angle_fusion(p2, coords, cm) * 0.8)
        with torch.no_grad():
            got = rb.aft_nab(q.to(dev), k.to(dev), v.to(dev), coords.to(dev), cm.to(dev), m2, scale=0.8)
        assert (got.cpu().double() - want).abs().max() < 2e-6 * max(1.0, want.abs().max().item()), transposed
    # given-bias form (any gate variant upstream of it): same result as torch on an arbitrary bias
    bias = torch.randn(B, N, N, generator=g)
    with torch.no_grad():
        got = rb.aft_nab(q.to(dev), k.to(dev), v.to(dev), None, bias.to(dev), None, scale=1.3)
        gotT = rb.aft_nab(q.to(dev), k.to(dev), v.to(dev), None, bias.to(dev).transpose(1, 2), None, scale=1.3)
    assert (got.cpu().double() - aft_core(q, k, v, bias * 1.3)).abs().max() < 2e-6 * 4
    assert (gotT.cpu().double() - aft_core(q, k, v, bias.transpose(1, 2) * 1.3)).abs().max() < 2e-6 * 4
    with pytest.raises(NotImplementedError):
        rb.aft_nab(torch.zeros(1, 130, 128, device=dev), torch.zeros(1, 130, 128, device=dev), torch.zeros(1, 130, 128, device=dev),
                   torch.zeros(1, 130, 2, device=dev), torch.zeros(1, 130, 130, device=dev), m2)


@pytest.mark.gpu
def test_patch_encoder_fuses_the_block():
    """patch_encoder on a block with upstream's attribute names (attn_freenet.py:360-442): the fused forward equals the
    unfused one (bias module -> AFTFull with torch ops)."""
    import rrnco_b200 as rb
    from torch import nn
    import torch.nn.functional as F

    class AFT(nn.Module):
        def __init__(self):
            super().__init__()
            self.to_q, self.to_k, self.to_v, self.project = (nn.Linear(128, 128) for _ in range(4))

        def forward(self, x, y=None, adapt_bias=None):
            p = {k: v for k, v in self.state_dict().items()}
            return oenc.aft_full(p, x, y, adapt_bias)

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.alpha = nn.Parameter(torch.full((1,), 1.3))
            self.attn_free = AFT()
            self.multi_head_combine = nn.Linear(128, 128)
            self.angle_distance_fusion = rb.DistAngleFusion(128)  # (stands for upstream's module: same parameters)
            self.norm1, self.norm2, self.norm3 = nn.LayerNorm(128), nn.LayerNorm(128), nn.LayerNorm(128)
            self.feed_forward = lambda a, b: a + b

        def forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None):  # attn_freenet.py:417-442
            row_emb, col_emb = self.norm1(row_emb), self.norm2(col_emb)
            bias = self.angle_distance_fusion(coords, cost_mat, duration_mat) * self.alpha
            out = self.attn_free(row_emb, y=col_emb, adapt_bias=bias)
            return self.feed_forward(self.norm3(self.multi_head_combine(out)), row_emb)

    torch.manual_seed(12)
    blk = Block().to("cuda")
    ref_fusion = blk.angle_distance_fusion

    class Ref(nn.Module):  # what upstream's module looks like to patch_encoder: not a DistAngleFusion instance
        def __init__(self, m):
            super().__init__()
            self.embed_dim, self.dist_emb, self.angle_emb, self.gate, self.out_lin = 128, m.dist_emb, m.angle_emb, m.gate, m.out_lin

        def forward(self, coords, cost_mat, duration_mat=None):
            return ref_fusion(coords, cost_mat)
    blk.angle_distance_fusion = Ref(ref_fusion)
    g = torch.Generator().manual_seed(13)
    row, col = torch.randn(3, 40, 128, generator=g).cuda(), torch.randn(3, 40, 128, generator=g).cuda()
    coords, cost = torch.rand(3, 40, 2, generator=g).cuda(), torch.rand(3, 40, 40, generator=g).cuda()
    with torch.no_grad():
        want = blk(row, col, cost.transpose(1, 2), coords)
        assert rb.patch_encoder(blk) == 1
        got = blk(row, col, cost.transpose(1, 2), coords)
    assert (got - want).abs().max() < 2e-5


@pytest.mark.gpu
def test_duration_gate_kernel_matches_reference_fixture_and_oracle():
    """rcvrptw variant on tcgen05 (encoder_dur_kernel.cu): the fixture recorded from the reference module (parameters x3),
    both matrix orientations; then default initialisation at n = 50 (2601 pairs per instance: ragged last tile) vs the
    CPU restatement; the col-encoding block's transposed views; the status word on an operand overflow."""
    import rrnco_b200 as rb
    dev = "cuda"
    t, params = _fixture()
    m = rb.DistAngleFusion(128, use_duration_matrix=True).to(dev)
    m.load_state_dict(params["dur"], strict=True)
    coords, cost, dur = t["coords"].to(dev), t["cost"].to(dev), t["dur"].to(dev)
    with torch.no_grad():
        out = m(coords, cost, dur)
        outT = m(coords, cost.transpose(1, 2), dur.transpose(1, 2))
        out2 = m(coords, cost, dur, scale=1.9)
    assert (out.cpu() - t["dur.bias"]).abs().max() < 3e-5, (out.cpu() - t["dur.bias"]).abs().max()
    assert (outT.cpu() - t["dur.bias_T"]).abs().max() < 3e-5
    assert torch.allclose(out2, out * 1.9, rtol=1e-6, atol=1e-6)
    torch.manual_seed(21)
    m2 = rb.DistAngleFusion(128, use_duration_matrix=True).to(dev)
    p2 = {k: v.detach().cpu() for k, v in m2.state_dict().items()}
    g = torch.Generator().manual_seed(22)
    B, N = 7, 51
    coords = torch.rand(B, N, 2, generator=g)
    cost, dur = torch.rand(B, N, N, generator=g) * 1.4, torch.rand(B, N, N, generator=g)
    want = oenc.dist_angle_fusion(p2, coords, cost, dur)
    with torch.no_grad():
        got = m2(coords.to(dev), cost.to(dev), dur.to(dev))
        again = m2(coords.to(dev), cost.to(dev), dur.to(dev))
    assert (got.cpu() - want).abs().max() < 3e-6 * max(1.0, want.abs().max().item()), (got.cpu() - want).abs().max()
    assert torch.equal(got, again)  # one issuing thread, fixed order: bitwise reproducible
    with torch.no_grad(), pytest.raises(ValueError):
        m2(coords.to(dev), cost.to(dev))
    with torch.no_grad(), pytest.raises(AssertionError, match="fp16 operand range"):
        m2(coords.to(dev), cost.to(dev) * 1e6, dur.to(dev))
