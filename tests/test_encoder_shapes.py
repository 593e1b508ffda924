"""The encoder's inference kernels against fp64 at the shapes the encoder runs: the two-way gate (`rrnco_nab_gating`, table and
brute-force variants), the fused bias + AFT-full block (`rrnco_aft_nab`, N <= 128) and the rcvrptw duration gate on tcgen05
(`rrnco_nab_dur_gating`), including the tile regimes of its persistent grid and non-finite inputs.

Every GPU check calls the C ABI directly, into an output pre-filled with NaN and followed by a canary tail of CANARY_FLOATS
floats, and then looks at every element: no NaN is left where the reference is finite, the tail is bitwise unchanged, and
    |got - want| <= c * 2^-24 * cond
per element.  `want` is the oracle's op sequence (`oracle.encoder.dist_angle_fusion`, and `aft_core` as
tests/test_encoder_ops.py writes it) in fp64, evaluated in chunks of instances, and of rows at large N, so that its peak
memory stays under REF_BYTES.  `cond` is the sum of the absolute values of the terms the kernel adds, computed in fp64 from
the parameters collapsed the way the kernels collapse them (these vectors are used for the bars only, never as the
reference).  Each test's docstring states its c and the worst ratio err / (2^-24 cond) measured on a B200.
"""
import copy

import pytest
import torch

from oracle import encoder as oenc

EPS = 2.0 ** -24
CANARY_FLOATS = 3 * 128          # three rows of Y after the fused block's output; > 256 floats after every output
CANARY_BITS = 0x5EED1234
REF_BYTES = 12 << 30             # peak memory of one reference evaluation on the GPU
PAIRS_PER_CHUNK = 1 << 19        # ~14 KB of fp64 intermediates per pair in the duration gate's reference
TILE_PAIRS = 128                 # pairs per tile of nab_dur_kernel; its grid is min(tiles, 2 x SMs)


# ---------------------------------------------------------------------------------------------------------------------
# shapes
# ---------------------------------------------------------------------------------------------------------------------
def dur_tiles(B, N):
    return -(-B * N * N // TILE_PAIRS)


def dur_regimes(sms):
    """(B, N) per tile regime of the duration gate's persistent grid of min(tiles, 2 sms) CTAs, for a device with `sms`
    SMs: `under` has fewer tiles than CTAs (one tile per CTA at most, instances straddling tiles), `exact` exactly 3 tiles
    per CTA, `tail<r>` more than two rounds of the grid plus a partial round, with n_pairs mod 128 = r."""
    G = 2 * sms
    out = {"under": (max(1, G - 1), 11), "exact": (3 * sms, 16)}
    for name, N, r in (("tail1", 63, 1), ("tail64", 40, 64), ("tail127", 63, 127)):
        B = 1
        while not (B * N * N % TILE_PAIRS == r and dur_tiles(B, N) > 2 * G and dur_tiles(B, N) % G):
            B += 1
        out[name] = (B, N)
    return out


def _chunks(B, N, pairs=PAIRS_PER_CHUNK):
    """(b0, b1, r0, r1): instance chunks of whole matrices, or one instance in row chunks when a matrix alone is larger."""
    if N * N <= pairs:
        step = max(1, pairs // (N * N))
        for b0 in range(0, B, step):
            yield b0, min(B, b0 + step), 0, N
    else:
        step = max(1, pairs // N)
        for b in range(B):
            for r0 in range(0, N, step):
                yield b, b + 1, r0, min(N, r0 + step)


# ---------------------------------------------------------------------------------------------------------------------
# fp64 reference and condition numbers
# ---------------------------------------------------------------------------------------------------------------------
def _active(w, b, s):
    """|w s| + |b| of the units a kernel may count as active at s ([..., E]): relu's argument is positive or within
    rounding of zero (a scalar on a breakpoint)."""
    ws = s.unsqueeze(-1) * w
    mag = ws.abs() + b.abs()
    return torch.where(ws + b >= -2.0 ** -20 * mag, mag, torch.zeros_like(mag)), torch.relu(ws + b)


def _cond_two_way(p, s_cost, s_angle):
    """Sum of |terms| of the collapsed two-way gate (encoder_kernels.cu header): per MLP the four functions
    sum_k u_k relu(w_k x + b_k), then z, the sigmoid and the blend; the gate's sensitivity g(1-g)|OD - OA| times z's terms."""
    E = p["out_lin.weight"].shape[1]
    wg, wo = p["gate.0.weight"][0], p["out_lin.weight"][0]
    parts = []
    for pre, s, wgx in (("dist_emb", s_cost, wg[:E]), ("angle_emb", s_angle, wg[E:])):
        W2 = p[f"{pre}.2.weight"]
        mag, h = _active(p[f"{pre}.0.weight"][:, 0], p[f"{pre}.0.bias"], s)
        ug, uo = W2.t() @ wgx, W2.t() @ wo
        parts.append((h @ ug, h @ uo + wo @ p[f"{pre}.2.bias"], mag @ ug.abs(), mag @ uo.abs() + (wo @ p[f"{pre}.2.bias"]).abs()))
    cg = p["gate.0.bias"][0] + wg[:E] @ p["dist_emb.2.bias"] + wg[E:] @ p["angle_emb.2.bias"]
    (zd, od, szd, sod), (za, oa, sza, soa) = parts
    g = torch.sigmoid(zd + za + cg)
    y = g * od + (1 - g) * oa + p["out_lin.bias"][0]
    return (g * sod + (1 - g) * soa + p["out_lin.bias"][0].abs() + g * (1 - g) * (od - oa).abs() * (szd + sza + cg.abs() + 1)
            + y.abs())


def _cond_duration(p, s):
    """Sum of |terms| of the duration gate as nab_dur_kernel evaluates it: O_x = uo_x . h_x + co_x, the gate's first layer
    collapsed to M_x h_x + c0 (M_x = Wg1[:, x] W2_x, the MMA), SiLU, the E -> 3 layer, the tempered softmax and the blend;
    the softmax's sensitivity g_c |O_c - sum g O| times the terms of its logit."""
    E = p["out_lin.weight"].shape[1]
    wo, Wg1 = p["out_lin.weight"][0], p["gate.0.weight"]
    hp, hp_mag, O, SO = p["gate.0.bias"].clone(), p["gate.0.bias"].abs(), [], []
    for x, pre in enumerate(("dist_emb", "angle_emb", "dur_emb")):
        W2, b2 = p[f"{pre}.2.weight"], p[f"{pre}.2.bias"]
        mag, h = _active(p[f"{pre}.0.weight"][:, 0], p[f"{pre}.0.bias"], s[x])
        M = Wg1[:, x * E:(x + 1) * E] @ W2
        hp = hp + h @ M.t() + Wg1[:, x * E:(x + 1) * E] @ b2
        hp_mag = hp_mag + mag @ M.t().abs() + (Wg1[:, x * E:(x + 1) * E] @ b2).abs()
        uo = W2.t() @ wo
        O.append(h @ uo + wo @ b2)
        SO.append(mag @ uo.abs() + (wo @ b2).abs())
    sg = torch.sigmoid(hp)
    si, dsi = hp * sg, (sg * (1 + hp * (1 - sg))).abs()
    W3, b3 = p["gate.2.weight"], p["gate.2.bias"]
    inv_t = torch.exp(-p["gate_temperature"])
    g = torch.softmax((si @ W3.t() + b3) * inv_t, dim=-1)
    Ob = sum(g[..., x] * O[x] for x in range(3))
    cz = inv_t * ((si.abs() + dsi * hp_mag + 1) @ W3.t().abs() + b3.abs())
    y = Ob + p["out_lin.bias"][0]
    return (sum(g[..., x] * SO[x] + g[..., x] * (O[x] - Ob).abs() * cz[..., x] for x in range(3))
            + p["out_lin.bias"][0].abs() + y.abs())


def fusion_reference(p, coords, cost, dur=None, scale=1.0, pairs=PAIRS_PER_CHUNK):
    """(want, cond) [B, N, N] fp64 of DistAngleFusion.forward * scale: the oracle's op sequence in chunks (`cost` / `dur`
    may be transposed views; they are read as the module reads them).  Runs where the inputs are."""
    p = {k: v.to(coords.device, torch.float64) for k, v in p.items()}
    B, N = cost.shape[0], cost.shape[-1]
    want = torch.empty(B, N, N, dtype=torch.float64, device=coords.device)
    cond = torch.empty_like(want)
    for b0, b1, r0, r1 in _chunks(B, N, pairs):
        c64 = coords[b0:b1].double()
        cm = cost[b0:b1].double()
        dm = None if dur is None else dur[b0:b1].double()
        want[b0:b1, r0:r1] = oenc.dist_angle_fusion(p, c64, cm, dm, rows=(r0, r1)) * scale
        s = (cm[:, r0:r1], oenc.pairwise_angles(c64, (r0, r1)), None if dm is None else dm[:, r0:r1])
        cond[b0:b1, r0:r1] = (_cond_two_way(p, s[0], s[1]) if dm is None else _cond_duration(p, s)) * abs(scale)
    return want, cond


def aft_core(q, k, v, bias):
    """AFTFull.forward (attn_freenet.py:309-327) between its Linear layers, fp64 (as tests/test_encoder_ops.py writes it)."""
    a = torch.exp(torch.softmax(bias.double(), dim=-1))
    e1 = torch.exp(torch.softmax(k.double(), dim=1))
    return torch.sigmoid(q.double()) * (a @ (e1 * v.double())) / (a @ e1)


def aft_reference(q, k, v, bias, bias_cond, inst=64):
    """(want, cond) [B, N, E] of the fused block given the fp64 bias and its cond: the products' |terms|, plus the change of
    a_ij = exp(softmax(bias)_ij) under the bias's own rounding (a_ij p_ij (cond_ij + max_j cond_ij) against |E2| and |y E1|)."""
    B = q.shape[0]
    want = torch.empty(q.shape, dtype=torch.float64, device=q.device)
    cond = torch.empty_like(want)
    for b0 in range(0, B, inst):
        b1 = min(B, b0 + inst)
        bb, cb = bias[b0:b1], bias_cond[b0:b1]
        pr = torch.softmax(bb, dim=-1)
        a = torch.exp(pr)
        e1 = torch.exp(torch.softmax(k[b0:b1].double(), dim=1))
        e2 = e1 * v[b0:b1].double()
        den = a @ e1
        y0 = (a @ e2) / den
        sig = torch.sigmoid(q[b0:b1].double())
        want[b0:b1] = aft_core(q[b0:b1], k[b0:b1], v[b0:b1], bb)
        prop = a * pr * (cb + cb.amax(dim=-1, keepdim=True))
        cond[b0:b1] = sig * ((a @ e2.abs() + y0.abs() * den + prop @ e2.abs() + y0.abs() * (prop @ e1)) / den + y0.abs()) \
            + want[b0:b1].abs()
    return want, cond


def reference_peak(fn):
    """Runs fn() and asserts that the memory it allocated at its peak stays under REF_BYTES; returns (result, peak bytes)."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < REF_BYTES, peak
    return out, peak


# ---------------------------------------------------------------------------------------------------------------------
# kernel calls through the C ABI, and the per-element check
# ---------------------------------------------------------------------------------------------------------------------
def _out_buffer(n, dev="cuda"):
    buf = torch.full((n + CANARY_FLOATS,), float("nan"), device=dev)
    buf[n:].view(torch.int32).fill_(CANARY_BITS)
    return buf


def _canary_intact(buf, n):
    return bool((buf[n:].view(torch.int32) == CANARY_BITS).all())


def run_gating(packed, coords, cost, transpose, scale, variant):
    from rrnco_b200._lib import call, ptr, stream_ptr
    B, N = cost.shape[0], cost.shape[-1]
    buf = _out_buffer(B * N * N)
    call("rrnco_nab_gating", B, N, ptr(coords), ptr(cost), transpose, ptr(packed), float(scale), variant, ptr(buf), stream_ptr())
    torch.cuda.synchronize()
    assert _canary_intact(buf, B * N * N), "rrnco_nab_gating wrote past the end of out"
    return buf[:B * N * N].view(B, N, N)


def run_aft(q, k, v, coords, cost, transpose, packed, scale):
    from rrnco_b200._lib import call, ptr, stream_ptr
    B, N, E = q.shape
    buf = _out_buffer(B * N * E)
    call("rrnco_aft_nab", B, N, ptr(q), ptr(k), ptr(v), ptr(coords), ptr(cost), transpose, ptr(packed), float(scale), ptr(buf),
         stream_ptr())
    torch.cuda.synchronize()
    assert _canary_intact(buf, B * N * E), "rrnco_aft_nab wrote past the end of Y"
    return buf[:B * N * E].view(B, N, E)


def run_duration(packed, coords, cost, dur, transpose, scale):
    """(out, status word)"""
    from rrnco_b200._lib import call, ptr, stream_ptr
    B, N = cost.shape[0], cost.shape[-1]
    buf = _out_buffer(B * N * N)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    call("rrnco_nab_dur_gating", B, N, ptr(coords), ptr(cost), ptr(dur), transpose, ptr(packed), float(scale), ptr(buf),
         ptr(status), stream_ptr())
    torch.cuda.synchronize()
    assert _canary_intact(buf, B * N * N), "rrnco_nab_dur_gating wrote past the end of out"
    return buf[:B * N * N].view(B, N, N), int(status.item())


def check_bar(got, want, cond, c, what):
    """Every element: no NaN where want is finite, |got - want| <= c 2^-24 cond.  Returns the worst err / (2^-24 cond)."""
    fin = torch.isfinite(want)
    assert fin.all(), f"{what}: non-finite reference"
    assert not torch.isnan(got).any(), f"{what}: {int(torch.isnan(got).sum())} elements unwritten or NaN"
    ratio = ((got.double() - want).abs() / (EPS * cond)).max().item()
    print(f"RATIO {what}: {ratio:.3f} (c = {c})")
    assert ratio <= c, f"{what}: worst err / (2^-24 cond) = {ratio:.2f} > {c}"
    return ratio


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _module(dur, params, seed):
    """(module on cuda, fp64 state dict): default init, x3 (every parameter, like tests/golden/encoder_nab.npz) or sharp
    (duration gate with gate_temperature = -2: logits times e^2)."""
    import rrnco_b200 as rb
    torch.manual_seed(seed)
    m = rb.DistAngleFusion(128, use_duration_matrix=dur).to("cuda")
    with torch.no_grad():
        if params == "x3":
            for t in m.parameters():
                t.mul_(3.0)
        elif params == "sharp":
            m.gate_temperature.fill_(-2.0)
    return m, {k: v.detach().double() for k, v in m.state_dict().items()}


def _lattice_coords(B, N, g):
    """Coordinates on a 5 x 5 lattice: duplicates (atan2(0, 0)), collinear pairs with dy = +0 and dx < 0 (angle pi) and, on
    the row y = 0, signed zeros (-0 - +0 = -0: angle -pi)."""
    xy = torch.randint(0, 5, (B, N, 2), generator=g).float() / 4
    y = xy[..., 1]
    y[(y == 0) & (torch.rand(B, N, generator=g) < 0.5)] = -0.0
    return xy


def _cost_with_breakpoints(m, B, N, g):
    """cost entries in [0, 1.4), a tenth of them exactly on breakpoints of the distance MLP (the tables' segment edges)."""
    cost = torch.rand(B, N, N, generator=g) * 1.4
    w, b = m.dist_emb[0].weight[:, 0].detach().cpu(), m.dist_emb[0].bias.detach().cpu()
    t = -b / w
    t = t[(t > 0) & (t < 1.4)]
    if t.numel():
        sel = torch.rand(B, N, N, generator=g) < 0.1
        cost[sel] = t[torch.randint(0, t.numel(), (int(sel.sum()),), generator=g)]
    return cost


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests of the machinery
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dur", [False, True])
def test_chunked_reference_equals_unchunked(dur):
    """The chunked fp64 reference (instance chunks and row chunks) is the oracle's op sequence on every pair."""
    import rrnco_b200 as rb
    torch.manual_seed(5)
    m = rb.DistAngleFusion(128, use_duration_matrix=dur)
    p = {k: v.detach().double() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(6)
    for B, N, pairs in ((5, 9, 200), (2, 23, 100)):  # 2 instances per chunk; rows of 4 (ragged last row chunk)
        coords = torch.rand(B, N, 2, generator=g, dtype=torch.float64)
        cost = torch.rand(B, N, N, generator=g, dtype=torch.float64).transpose(1, 2)
        dm = torch.rand(B, N, N, generator=g, dtype=torch.float64).transpose(1, 2) if dur else None
        assert len(list(_chunks(B, N, pairs))) > 1
        want = oenc.dist_angle_fusion(p, coords, cost, dm) * 0.7
        got, cond = fusion_reference(p, coords, cost, dm, scale=0.7, pairs=pairs)
        assert (got - want).abs().max() < 1e-12
        _, cond1 = fusion_reference(p, coords, cost, dm, scale=0.7, pairs=10 ** 9)
        assert (cond - cond1).abs().max() < 1e-12 and (cond >= want.abs()).all()


@pytest.mark.parametrize("sms", [1, 2, 3, 7, 80, 132, 148, 160])
def test_duration_gate_tile_regimes_hold_for_any_sm_count(sms):
    G = 2 * sms
    r = dur_regimes(sms)
    B, N = r["under"]
    assert dur_tiles(B, N) < G or (sms == 1 and dur_tiles(B, N) == 1)
    B, N = r["exact"]
    assert B * N * N % TILE_PAIRS == 0 and dur_tiles(B, N) == 3 * G
    for name, rem in (("tail1", 1), ("tail64", 64), ("tail127", 127)):
        B, N = r[name]
        assert B * N * N % TILE_PAIRS == rem and dur_tiles(B, N) > 2 * G and dur_tiles(B, N) % G != 0, name
    assert dur_tiles(1024, 101) == 81608 and dur_tiles(1, 1000) == 7813 and 1000 ** 2 % TILE_PAIRS == 64


def test_oracle_nonfinite_pattern():
    """What the non-finite tests hold the kernels to: upstream's op sequence turns a NaN cost entry into NaN at that pair
    only (both gate variants), and a NaN coordinate into NaN on the node's row and column; a NaN bias entry spreads along
    its row through AFT-full's row softmax."""
    import rrnco_b200 as rb
    g = torch.Generator().manual_seed(7)
    B, N = 2, 6
    coords = torch.rand(B, N, 2, generator=g, dtype=torch.float64)
    cost = torch.rand(B, N, N, generator=g, dtype=torch.float64)
    dur = torch.rand(B, N, N, generator=g, dtype=torch.float64)
    for use_dur in (False, True):
        torch.manual_seed(8)
        p = {k: v.detach().double() for k, v in rb.DistAngleFusion(128, use_duration_matrix=use_dur).state_dict().items()}
        c = cost.clone()
        c[1, 2, 3] = float("nan")
        out = oenc.dist_angle_fusion(p, coords, c, dur if use_dur else None)
        want = torch.zeros(B, N, N, dtype=torch.bool)
        want[1, 2, 3] = True
        assert torch.equal(torch.isnan(out), want)
        xy = coords.clone()
        xy[1, 4, 0] = float("nan")
        out = oenc.dist_angle_fusion(p, xy, cost, dur if use_dur else None)
        want = torch.zeros(B, N, N, dtype=torch.bool)
        want[1, 4, :] = want[1, :, 4] = True
        assert torch.equal(torch.isnan(out), want)
    bias = torch.rand(B, N, N, dtype=torch.float64)
    bias[1, 2, 3] = float("nan")
    q, k, v = (torch.randn(B, N, 128, dtype=torch.float64) for _ in range(3))
    rows = torch.isnan(aft_core(q, k, v, bias)).all(dim=-1)
    want = torch.zeros(B, N, dtype=torch.bool)
    want[1, 2] = True
    assert torch.equal(rows, want) and torch.isnan(aft_core(q, k, v, bias)).any(dim=-1).equal(want)


# ---------------------------------------------------------------------------------------------------------------------
# A. two-way gate
# ---------------------------------------------------------------------------------------------------------------------
GATING_C = 2


@pytest.mark.gpu
@pytest.mark.parametrize("params", ["default", "x3"])
@pytest.mark.parametrize("N,B", [(1, 37), (2, 33), (13, 9), (101, 7), (128, 3), (129, 3), (200, 2), (1000, 1), (101, 1024)])
def test_two_way_gate_against_fp64(N, B, params):
    """rrnco_nab_gating, table (0) and brute-force (1) variants, both cost orientations, scale 0.8, every element.  B is
    chosen so that the 1024-pair chunks of an instance end raggedly (N = 128: exactly 16 chunks).  Lattice coordinates
    (duplicates, angles pi and -pi), a tenth of the cost entries on breakpoints.  c = 2; worst measured ratio 1.43
    (brute-force variant), 1.03 (table variant).  Scaling the out intercept of the most used segment by 1 + 1e-5 gives 9.5."""
    m, p = _module(False, params, seed=100 + N)
    g = torch.Generator().manual_seed(N * 7 + B)
    coords = _lattice_coords(B, N, g).cuda()
    cost = _cost_with_breakpoints(m, B, N, g).cuda()
    packed = m.packed_parameters()
    for transpose in (0, 1):
        cm = cost.transpose(1, 2) if transpose else cost
        (want, cond), peak = reference_peak(lambda: fusion_reference(p, coords, cm, scale=0.8))
        print(f"reference peak {peak / 2**30:.2f} GiB")
        for variant in (0, 1):
            got = run_gating(packed, coords, cost, transpose, 0.8, variant)
            check_bar(got, want, cond, GATING_C, f"gating v{variant} N={N} B={B} {params} T={transpose}")
    # batch-position independence: first, middle and last instance alone
    for b in sorted({0, B // 2, B - 1}):
        alone = run_gating(packed, coords[b:b + 1].contiguous(), cost[b:b + 1].contiguous(), 0, 0.8, 0)
        assert _same_bits(alone[0], run_gating(packed, coords, cost, 0, 0.8, 0)[b]), b


# ---------------------------------------------------------------------------------------------------------------------
# B. fused bias + AFT-full
# ---------------------------------------------------------------------------------------------------------------------
AFT_C = 1          # fusion form
AFT_GIVEN_C = 8    # given-bias form: rows of a random bias, some x40


def _qkv(B, N, g):
    """q, k, v with K columns spanning e^-3 .. e^3 in scale (peaked and flat column softmaxes) and V of mixed signs."""
    q = torch.randn(B, N, 128, generator=g)
    k = torch.randn(B, N, 128, generator=g) * torch.exp(torch.linspace(-3, 3, 128))
    v = torch.randn(B, N, 128, generator=g) + 0.3
    return q.cuda(), k.cuda(), v.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 2, 31, 32, 33, 64, 65, 97, 101, 127, 128])
def test_aft_nab_against_fp64(N):
    """rrnco_aft_nab at every key-slot and row-group boundary: the fusion form (x3 parameters, scale 40: peaked bias rows)
    and the given-bias form (a random bias with some rows x40, scale 1.3), both orientations, every element, canary rows
    after Y.  B = 1024 at N = 128 (138 KB of shared memory per CTA).  c = 1 for the fusion form, worst measured ratio
    0.32; c = 8 for the given-bias form, worst 4.2 (its bar counts only the rounding of the bias entries, and entries
    near zero round to little).  Scaling the out intercept of the most used segment by 1 + 1e-5 gives 1.55."""
    B = 1024 if N == 128 else 5
    m, p = _module(False, "x3", seed=200 + N)
    g = torch.Generator().manual_seed(300 + N)
    coords = torch.rand(B, N, 2, generator=g).cuda()
    cost = (torch.rand(B, N, N, generator=g) * 1.4).cuda()
    q, k, v = _qkv(B, N, g)
    bias = torch.randn(B, N, N, generator=g)
    bias[:, ::3] *= 40
    bias = bias.cuda()
    packed = m.packed_parameters()
    for transpose in (0, 1):
        cm = cost.transpose(1, 2) if transpose else cost
        bw, bc = fusion_reference(p, coords, cm, scale=40.0)
        want, cond = aft_reference(q, k, v, bw, bc)
        got = run_aft(q, k, v, coords, cost, transpose, packed, 40.0)
        check_bar(got, want, cond, AFT_C, f"aft fusion N={N} T={transpose}")
        bm = bias.transpose(1, 2) if transpose else bias
        want, cond = aft_reference(q, k, v, bm.double() * 1.3, (bm.double() * 1.3).abs())
        got = run_aft(q, k, v, None, bias, transpose, None, 1.3)
        check_bar(got, want, cond, AFT_GIVEN_C, f"aft given N={N} T={transpose}")
    for b in sorted({0, B // 2, B - 1}):
        sl = slice(b, b + 1)
        alone = run_aft(q[sl].contiguous(), k[sl].contiguous(), v[sl].contiguous(), coords[sl].contiguous(),
                        cost[sl].contiguous(), 0, packed, 40.0)
        assert _same_bits(alone[0], run_aft(q, k, v, coords, cost, 0, packed, 40.0)[b]), b


@pytest.mark.gpu
def test_aft_nab_rejects_more_than_128_nodes():
    from rrnco_b200._lib import RRNCOError
    m, _ = _module(False, "default", seed=1)
    z = torch.zeros(1, 129, 128, device="cuda")
    with pytest.raises(RRNCOError):
        run_aft(z, z, z, torch.zeros(1, 129, 2, device="cuda"), torch.zeros(1, 129, 129, device="cuda"), 0,
                m.packed_parameters(), 1.0)


class _RefFusion(torch.nn.Module):
    """What upstream's DistAngleFusion looks like to patch_encoder (attn_freenet.py:201-240), forward = the oracle."""

    def __init__(self, dur):
        super().__init__()
        E = self.embed_dim = 128
        mk = lambda: torch.nn.Sequential(torch.nn.Linear(1, E), torch.nn.ReLU(), torch.nn.Linear(E, E))  # noqa: E731
        self.dist_emb, self.angle_emb = mk(), mk()
        if dur:
            self.dur_emb = mk()
            self.gate = torch.nn.Sequential(torch.nn.Linear(3 * E, E), torch.nn.SiLU(), torch.nn.Linear(E, 3))
            self.gate_temperature = torch.nn.Parameter(torch.tensor(5.0))
        else:
            self.gate = torch.nn.Sequential(torch.nn.Linear(2 * E, 1), torch.nn.Sigmoid())
        self.out_lin = torch.nn.Linear(E, 1)

    def forward(self, coords, cost_mat, duration_mat=None):
        return oenc.dist_angle_fusion(dict(self.state_dict()), coords, cost_mat, duration_mat)


class _AFT(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.to_q, self.to_k, self.to_v, self.project = (torch.nn.Linear(128, 128) for _ in range(4))

    def forward(self, x, y=None, adapt_bias=None):
        return oenc.aft_full(dict(self.state_dict()), x, y, adapt_bias)


class _Block(torch.nn.Module):
    """An attention-free block with upstream's attribute names (attn_freenet.py:360-442): the bias module is
    `angle_distance_fusion` (two-way gate) or `neural_adaptive_bias` (rcvrptw)."""

    def __init__(self, dur):
        super().__init__()
        self.alpha = torch.nn.Parameter(torch.full((1,), 1.3))
        self.attn_free = _AFT()
        self.multi_head_combine = torch.nn.Linear(128, 128)
        if dur:
            self.neural_adaptive_bias = _RefFusion(True)
        else:
            self.angle_distance_fusion = _RefFusion(False)
        self.norm1, self.norm2, self.norm3 = (torch.nn.LayerNorm(128) for _ in range(3))
        self.feed_forward = lambda a, b: a + b

    def forward(self, row_emb, col_emb, cost_mat, coords, duration_mat=None):
        row_emb, col_emb = self.norm1(row_emb), self.norm2(col_emb)
        fusion = self.neural_adaptive_bias if duration_mat is not None else self.angle_distance_fusion
        bias = fusion(coords, cost_mat, duration_mat) * self.alpha
        out = self.attn_free(row_emb, y=col_emb, adapt_bias=bias)
        return self.feed_forward(self.norm3(self.multi_head_combine(out)), row_emb)


@pytest.mark.gpu
@pytest.mark.parametrize("dur", [False, True], ids=["two_way", "rcvrptw"])
@pytest.mark.parametrize("N", [128, 129])
def test_patched_block_matches_unpatched_block_in_fp64(N, dur, monkeypatch):
    """patch_encoder on a block: N = 128 goes through the fused aft_nab kernel, N = 129 through the unfused block around
    the bias kernel; both match the unpatched block evaluated in fp64 (col-encoding orientation: transposed views)."""
    import rrnco_b200 as rb
    from rrnco_b200 import encoder_ops
    torch.manual_seed(400 + N)
    blk = _Block(dur).cuda()
    ref = copy.deepcopy(blk).double()
    g = torch.Generator().manual_seed(500 + N)
    B = 3
    row, col = (torch.randn(B, N, 128, generator=g).cuda() for _ in range(2))
    coords, cost, dm = (torch.rand(B, N, 2, generator=g).cuda(), torch.rand(B, N, N, generator=g).cuda(),
                        torch.rand(B, N, N, generator=g).cuda() if dur else None)
    args = (cost.transpose(1, 2), coords, None if dm is None else dm.transpose(1, 2))
    with torch.no_grad():
        want = ref(row.double(), col.double(), *(None if a is None else a.double() for a in args))
        assert rb.patch_encoder(blk) == 1
        calls = []
        monkeypatch.setattr(encoder_ops, "aft_nab", lambda *a, **kw: calls.append(1) or rb.aft_nab(*a, **kw))
        got = blk(row, col, *args)
    assert len(calls) == (1 if N <= 128 else 0)
    err = (got.double() - want).abs().max().item()
    assert err < 2e-5 * max(1.0, want.abs().max().item()), err


# ---------------------------------------------------------------------------------------------------------------------
# C. duration gate
# ---------------------------------------------------------------------------------------------------------------------
DUR_C = 2


def _dur_inputs(B, N, seed):
    g = torch.Generator().manual_seed(seed)
    coords = torch.rand(B, N, 2, generator=g).cuda()
    cost = (torch.rand(B, N, N, generator=g) * 1.4).cuda()
    dur = torch.rand(B, N, N, generator=g).cuda()
    return coords, cost, dur


def _check_duration(m, p, coords, cost, dur, scale, what, orientations=(0, 1)):
    packed = m._packed_duration()
    outs = {}
    for transpose in orientations:
        cm, dm = (cost.transpose(1, 2), dur.transpose(1, 2)) if transpose else (cost, dur)
        (want, cond), peak = reference_peak(lambda: fusion_reference(p, coords, cm, dm, scale=scale))
        print(f"reference peak {peak / 2**30:.2f} GiB")
        got, status = run_duration(packed, coords, cost, dur, transpose, scale)
        assert status == 0, what
        check_bar(got, want, cond, DUR_C, f"{what} T={transpose}")
        outs[transpose] = got
    return packed, outs


def _position_independent(packed, coords, cost, dur, out, scale, instances):
    for b in sorted(set(instances)):
        sl = slice(b, b + 1)
        alone, status = run_duration(packed, coords[sl].contiguous(), cost[sl].contiguous(), dur[sl].contiguous(), 0, scale)
        assert status == 0 and _same_bits(alone[0], out[b]), b


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["under", "exact", "tail1", "tail64", "tail127"])
def test_duration_gate_tile_regimes(regime):
    """rrnco_nab_dur_gating in every regime of its persistent grid (dur_regimes for this device's SM count): fewer tiles
    than CTAs, exactly 3 tiles per CTA, more than two rounds plus a partial one with n_pairs mod 128 in {1, 64, 127}.
    Both orientations, scale 0.7, every element; status 0; bitwise run to run; the first instance, the last, and the one
    holding the first pair of the grid's second round equal the same instance computed alone, bitwise (MMA rows are
    independent: a pair's result does not depend on its row in the tile).  c = 2; worst measured ratio 0.76.  Skipping
    `scale` from a CTA's second tile on gives 3.8e5; scaling the largest entry of the packed uo_dist by 1 + 1e-5 gives 3.1."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B, N = dur_regimes(sms)[regime]
    m, p = _module(True, "default", seed=600)
    coords, cost, dur = _dur_inputs(B, N, 601)
    packed, outs = _check_duration(m, p, coords, cost, dur, 0.7, f"dur {regime} B={B} N={N}")
    again, _ = run_duration(packed, coords, cost, dur, 0, 0.7)
    assert _same_bits(again, outs[0])
    second_round = min(B - 1, 2 * sms * TILE_PAIRS // (N * N))
    _position_independent(packed, coords, cost, dur, outs[0], 0.7, (0, second_round, B - 1))


@pytest.mark.gpu
@pytest.mark.parametrize("N,B,params", [(1, 300, "x3"), (2, 100, "sharp"), (101, 37, "default"), (101, 37, "x3"),
                                        (101, 37, "sharp"), (128, 5, "default"), (200, 3, "sharp"), (1000, 1, "x3")])
def test_duration_gate_sizes(N, B, params):
    """rrnco_nab_dur_gating at N from 1 to 1000 (1 x 1000^2 = 7813 tiles, a tail of 64 pairs) with the three parameter sets
    (default init, x3 like the fixture, gate_temperature = -2), both orientations, scale 0.7, every element; status 0;
    bitwise run to run.  c = 2; worst measured ratio 0.84."""
    m, p = _module(True, params, seed=700 + N)
    coords, cost, dur = _dur_inputs(B, N, 701 + N)
    packed, outs = _check_duration(m, p, coords, cost, dur, 0.7, f"dur N={N} B={B} {params}")
    again, _ = run_duration(packed, coords, cost, dur, 0, 0.7)
    assert _same_bits(again, outs[0])


@pytest.mark.gpu
def test_duration_gate_at_c3_batch():
    """Config C3's shape, 1024 x 101^2 = 81 608 tiles (about 276 per CTA on 148 SMs), every element, scale 1; position
    independence of the first, the last and a middle instance.  c = 2; worst measured ratio 1.14."""
    m, p = _module(True, "default", seed=800)
    B, N = 1024, 101
    coords, cost, dur = _dur_inputs(B, N, 801)
    packed, outs = _check_duration(m, p, coords, cost, dur, 1.0, "dur C3", orientations=(0,))
    _position_independent(packed, coords, cost, dur, outs[0], 1.0, (0, 517, B - 1))


@pytest.mark.gpu
def test_duration_gate_overflow_on_a_late_tile_raises():
    """One pair of the last instance out of the fp16 operand range: the CTA that reaches it on its last round sets the
    status word, and the module raises."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B, N = dur_regimes(sms)["tail127"]
    m, _ = _module(True, "default", seed=900)
    coords, cost, dur = _dur_inputs(B, N, 901)
    cost[-1, N - 1, N - 2] = 1e6
    _, status = run_duration(m._packed_duration(), coords, cost, dur, 0, 1.0)
    assert status != 0
    with torch.no_grad(), pytest.raises(AssertionError, match="fp16 operand range"):
        m(coords, cost, dur)


# ---------------------------------------------------------------------------------------------------------------------
# D. non-finite inputs
# ---------------------------------------------------------------------------------------------------------------------
def _poison(x, where, value):
    x = x.clone()
    x[where] = value
    return x


def _nonfinite_cases(B, N, dur):
    """(name, which input, index in the last instance, value, mask of the pairs that read it)"""
    i, j, n = N - 3, 2, N - 4
    pair = torch.zeros(B, N, N, dtype=torch.bool, device="cuda")
    pair[-1, i, j] = True
    node = torch.zeros(B, N, N, dtype=torch.bool, device="cuda")
    node[-1, n, :] = node[-1, :, n] = True
    for value in (float("nan"), float("inf")):
        yield f"cost={value}", "cost", (-1, i, j), value, pair
        if dur:
            yield f"dur={value}", "dur", (-1, i, j), value, pair
        yield f"coord={value}", "coords", (-1, n, 1), value, node


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [0, 1], ids=["table", "brute_force"])
def test_two_way_gate_nonfinite_inputs(variant):
    """A NaN or +inf cost entry or coordinate in the last instance: the output is non-finite exactly where the fp64
    oracle's is, every pair that does not read the changed input is bitwise the clean run's, and the finite pairs that do
    are within the bar."""
    m, p = _module(False, "x3", seed=1000)
    B, N = 3, 37
    coords, cost, _ = _dur_inputs(B, N, 1001)
    packed = m.packed_parameters()
    clean = run_gating(packed, coords, cost, 0, 1.0, variant)
    for name, which, idx, value, touched in _nonfinite_cases(B, N, False):
        xy = _poison(coords, idx, value) if which == "coords" else coords
        cm = _poison(cost, idx, value) if which == "cost" else cost
        want, cond = fusion_reference(p, xy, cm)
        got = run_gating(packed, xy, cm, 0, 1.0, variant)
        bad = ~torch.isfinite(want)
        assert bad.any() and torch.equal(~torch.isfinite(got), bad), name
        assert _same_bits(got[~touched], clean[~touched]), name
        ok = touched & ~bad
        if ok.any():
            check_bar(got[ok], want[ok], cond[ok], GATING_C, f"gating v{variant} {name} touched pairs")


@pytest.mark.gpu
def test_aft_nab_nonfinite_inputs():
    """The fused block with a NaN or +inf cost entry or coordinate: its output is non-finite exactly where AFT-full's is in
    fp64 on the oracle's bias (a non-finite bias entry spreads along its row through the row softmax); with a poisoned cost
    entry every other row is bitwise the clean run's.  Where upstream's bias is NaN, the table form's may be an infinity
    of either sign, which the row softmax treats differently (+inf: NaN row, -inf: weight 0), so at those entries the
    reference takes the bias the two-way gate kernel computes (non-finite there: test_two_way_gate_nonfinite_inputs)."""
    m, p = _module(False, "x3", seed=1100)
    B, N = 3, 37
    g = torch.Generator().manual_seed(1101)
    coords, cost, _ = _dur_inputs(B, N, 1102)
    q, k, v = _qkv(B, N, g)
    packed = m.packed_parameters()
    clean = run_aft(q, k, v, coords, cost, 0, packed, 1.0)
    for name, which, idx, value, _ in _nonfinite_cases(B, N, False):
        xy = _poison(coords, idx, value) if which == "coords" else coords
        cm = _poison(cost, idx, value) if which == "cost" else cost
        bias, _ = fusion_reference(p, xy, cm)
        bias = torch.where(torch.isfinite(bias), bias, run_gating(packed, xy, cm, 0, 1.0, 0).double())
        want = aft_core(q, k, v, bias)
        got = run_aft(q, k, v, xy, cm, 0, packed, 1.0)
        bad = ~torch.isfinite(want)
        assert bad.any() and torch.equal(~torch.isfinite(got), bad), name
        if which == "cost":
            rows = torch.ones(B, N, dtype=torch.bool, device="cuda")
            rows[idx[:2]] = False
            assert _same_bits(got[rows], clean[rows]), name


@pytest.mark.gpu
def test_duration_gate_nonfinite_inputs():
    """The duration gate with a NaN or +inf cost entry, duration entry or coordinate in the last instance of a multi-tile
    batch: the module raises; with check_overflow = False the pairs the fp64 oracle makes non-finite are non-finite, and
    every pair that does not read the changed input is bitwise the clean run's."""
    m, p = _module(True, "default", seed=1200)
    B, N = 9, 61
    coords, cost, dur = _dur_inputs(B, N, 1201)
    packed = m._packed_duration()
    clean, status = run_duration(packed, coords, cost, dur, 0, 1.0)
    assert status == 0
    for name, which, idx, value, touched in _nonfinite_cases(B, N, True):
        xy = _poison(coords, idx, value) if which == "coords" else coords
        cm = _poison(cost, idx, value) if which == "cost" else cost
        dm = _poison(dur, idx, value) if which == "dur" else dur
        m.check_overflow = True
        with torch.no_grad(), pytest.raises(AssertionError):
            m(xy, cm, dm)
        m.check_overflow = False
        with torch.no_grad():
            got = m(xy, cm, dm)
        want, _ = fusion_reference(p, xy, cm, dm)
        bad = ~torch.isfinite(want)
        assert bad.any() and torch.equal(~torch.isfinite(got), bad), name
        assert _same_bits(got[~touched], clean[~touched]), name


@pytest.mark.gpu
def test_duration_gate_backward_nonfinite_scalar_raises():
    """nab_dur_gating_backward promises to raise on a value that is not finite: a NaN cost entry must not pass its bound."""
    from rrnco_b200 import encoder_ops
    m, _ = _module(True, "default", seed=1300)
    B, N = 2, 40
    coords, cost, dur = _dur_inputs(B, N, 1301)
    flat = torch.cat([t.detach().float().reshape(-1) for t in encoder_ops._dur_params(m)])
    grad_out = torch.randn(B, N, N, device="cuda")
    packed = m._packed_duration()
    encoder_ops.nab_dur_gating_backward(coords, cost, dur, 0, packed, flat, 1.0, grad_out)  # clean: no error
    for which in ("cost", "dur", "coords"):
        args = [coords, cost, dur]
        k = ("coords", "cost", "dur").index(which)
        args[k] = _poison(args[k], (-1, 3, 1), float("nan"))
        with pytest.raises(AssertionError, match="not finite"):
            encoder_ops.nab_dur_gating_backward(*args, 0, packed, flat, 1.0, grad_out)
